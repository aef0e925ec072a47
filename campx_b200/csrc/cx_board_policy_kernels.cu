// cx_policy_sample with the policy input given as the uint8 BOARD (examples/actor_critic.py:64-98 on
// `layered_board.view(-1).float()`, actor_critic.py:147,173): the layered board is a function of the board in occluded
// games (campx/rendering.py:204-215: channel k = (board == chars[k])), so the float32 planes -- n_chars * cells floats
// per env, 13 KB for Hello World against its 468-byte board -- are never written or read.
//
// k_policy_sample_board<WMODE, LIST> keeps the CTA of k_policy_sample: eight warps own 32 envs, lane = env, warp w
// accumulates hidden units 4w..4w+3.  The CTA's 32 boards are staged in shared memory (row pitch an odd number of words:
// the lanes' reads are conflict-free).  The hidden layer then takes one of two walks:
//   LIST   only the set inputs, at most one per cell (policy_hidden_shares_list): every env's list of input indices
//          k * cells + cell in ascending order is built by a counting sort over channels -- warp w counts, per env and
//          channel, the cells of its eighth of the board, warp 0 turns the counts into offsets (channel-major, then warp,
//          so that each channel's cells stay ascending), and every warp scatters its cells -- into a [cells][32] u32 tile;
//          each warp then gathers the W1^T rows of its lane's list.  Used whenever the tile fits shared memory (boards
//          up to ~1,000-1,200 cells, by n_chars).
//   dense  all n_chars * cells inputs, four cells per board word (policy_hidden_shares_board): every lane of a warp reads
//          the same W1^T row, x in {0, 1}.  Larger boards.
// Where W1^T is read from:
//   W_STAGED      the whole of it staged once per CTA, hidden units padded to 32 with zeros (as k_policy_sample does),
//                 when it fits the budget below (boat_race: 175 x 128 B = 22 KB);
//   W_GLOBAL_VEC  otherwise, straight from global memory with one 16-byte load per input and warp (n_hidden == 32 and a
//                 16-byte aligned W1^T): the eight warps read the same rows, which stay in L1 / L2
//                 (Hello World: 3,276 x 128 B = 419 KB);
//   W_GLOBAL      the same with four predicated scalar loads (rows of n_hidden floats are not 16-byte aligned).
// Logits, the Philox stream and the sampling are those of k_policy_sample (policy_logits, sample_categorical), so equal
// inputs give equal bits.
#include "cx_internal.cuh"
#include "cx_policy.cuh"

namespace {

enum { W_STAGED = 0, W_GLOBAL_VEC = 1, W_GLOBAL = 2 };

// dynamic shared memory above this stages W1^T no longer (two CTAs per SM must still fit)
constexpr size_t BOARD_POLICY_STAGE_BUDGET = 100 * 1024;
constexpr size_t BOARD_POLICY_SMEM_MAX = 200 * 1024;   // the dynamic shared memory the launcher allows
constexpr size_t BOARD_POLICY_SHARES_BYTES = (size_t)(POLICY_THREADS / 32) * CX_MAX_ACTIONS * POLICY_PITCH * sizeof(float);

// bytes per staged board: whole words, an odd number of them (lane * pitch spreads the lanes over all 32 banks)
__host__ __device__ inline int board_pitch(int cells) {
  const int words = (cells + 3) >> 2;
  return 4 * (words | 1);
}

// shared memory of the LIST walk beyond boards and W1^T: byte -> channel table, per-warp counts, counts, list tile
__host__ __device__ inline size_t board_list_bytes(int cells, int n_chars) {
  return 256 + (size_t)(POLICY_THREADS / 32) * n_chars * 32 * sizeof(uint32_t) + 32 * sizeof(uint32_t) +
         (size_t)cells * 32 * sizeof(uint32_t);
}

template <int WMODE, bool LIST>
__global__ void __launch_bounds__(POLICY_THREADS)
    k_policy_sample_board(const uint8_t* __restrict__ board, int64_t n, int cells, const uint8_t* __restrict__ chars,
                          int n_chars, const float* __restrict__ w1t, const float* __restrict__ b1, int n_hidden,
                          const float* __restrict__ w2, const float* __restrict__ b2, int A, uint64_t seed,
                          uint64_t env_offset, const uint64_t* __restrict__ d_step, uint64_t step_offset,
                          uint8_t* __restrict__ actions, float* __restrict__ logp, float* __restrict__ logits_out) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int n_in = n_chars * cells, pitch = board_pitch(cells);
  float* s_h = reinterpret_cast<float*>(smem_raw);                          // [8 warps][CX_MAX_ACTIONS][33]
  float* s_w = s_h + (POLICY_THREADS / 32) * CX_MAX_ACTIONS * POLICY_PITCH;  // W_STAGED: [n_in][32] W1^T
  uint8_t* s_b = reinterpret_cast<uint8_t*>(s_w + (WMODE == W_STAGED ? (size_t)n_in * 32 : 0));   // [32][pitch]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t e0 = (int64_t)blockIdx.x * 32;
  const int n_here = (int)min((int64_t)32, n - e0);
  const PolicyRegs R = policy_load_small(b1, w2, b2, n_hidden, A, warp, lane);
  const uint64_t step = (d_step ? *d_step : 0ull) + step_offset;
  if (WMODE == W_STAGED) {
    if (n_hidden == 32 && (reinterpret_cast<uintptr_t>(w1t) & 15) == 0) {
      // every thread requests 8 float4 before it stores any (a load -> store loop pays the latency per iteration)
      constexpr int DEPTH = 8;
      for (int base = tid; base < n_in * 8; base += DEPTH * POLICY_THREADS) {
        float4 v[DEPTH];
#pragma unroll
        for (int u = 0; u < DEPTH; ++u)
          if (base + u * POLICY_THREADS < n_in * 8) v[u] = __ldg(reinterpret_cast<const float4*>(w1t) + base + u * POLICY_THREADS);
#pragma unroll
        for (int u = 0; u < DEPTH; ++u)
          if (base + u * POLICY_THREADS < n_in * 8) reinterpret_cast<float4*>(s_w)[base + u * POLICY_THREADS] = v[u];
      }
    } else {
#pragma unroll 4
      for (int k = tid; k < n_in * 32; k += POLICY_THREADS) {
        const int d = k >> 5, j = k & 31;
        s_w[k] = j < n_hidden ? __ldg(w1t + (size_t)d * n_hidden + j) : 0.0f;
      }
    }
  }
  // ---- the CTA's boards: one contiguous [n_here][cells] block -> rows of `pitch` bytes ----
  const uint8_t* blk = board + e0 * cells;
  if ((cells & 3) == 0 && (reinterpret_cast<uintptr_t>(blk) & 3) == 0) {
    const uint32_t wpr = (uint32_t)cells >> 2;
    const int total = n_here * (int)wpr;
#pragma unroll 4
    for (int q = tid; q < total; q += POLICY_THREADS) {
      const uint32_t e = (uint32_t)q / wpr, c = (uint32_t)q - e * wpr;
      reinterpret_cast<uint32_t*>(s_b + e * pitch)[c] = __ldg(reinterpret_cast<const uint32_t*>(blk) + q);
    }
  } else {
    const int total = n_here * cells;
#pragma unroll 4
    for (int k = tid; k < total; k += POLICY_THREADS) {
      const uint32_t e = (uint32_t)k / (uint32_t)cells, c = (uint32_t)k - e * (uint32_t)cells;
      s_b[e * pitch + c] = __ldg(blk + k);
    }
  }
  if (n_here < 32)                                      // lanes without an env compute on boards of zero bytes
    for (int k = tid; k < (32 - n_here) * (pitch >> 2); k += POLICY_THREADS)
      reinterpret_cast<uint32_t*>(s_b + n_here * pitch)[k] = 0u;
  // LIST: byte -> channel table (0xFF: no character of the game), then the tiles behind the boards
  uint8_t* s_lut = s_b + 32 * pitch;
  uint32_t* s_cnt = reinterpret_cast<uint32_t*>(s_lut + 256);             // [8 warps][n_chars][32 envs]
  uint32_t* s_count = s_cnt + (POLICY_THREADS / 32) * n_chars * 32;       // [32 envs]
  uint32_t* s_list = s_count + 32;                                        // [cells][32 envs]
  if (LIST) {
    s_lut[tid] = 0xFF;                                                    // (POLICY_THREADS == 256)
    __syncthreads();
    if (tid < n_chars) s_lut[__ldg(chars + tid)] = (uint8_t)tid;
  }
  __syncthreads();
  const int j0 = warp * 4;
  const uint8_t* mine = s_b + lane * pitch;
  auto walk = [&](const auto& row) {
    if (LIST) {
      // counting sort of this lane's cells by channel; warp w owns cells [c_lo, c_hi)
      const int per_warp = (cells + 7) >> 3, c_lo = min(cells, warp * per_warp), c_hi = min(cells, c_lo + per_warp);
      uint32_t* cnt = s_cnt + warp * n_chars * 32 + lane;                 // cnt[k * 32]: this thread's column only
      for (int k = 0; k < n_chars; ++k) cnt[k * 32] = 0;
      for (int c = c_lo; c < c_hi; ++c) {
        const uint32_t k = s_lut[mine[c]];
        if (k != 0xFF) cnt[k * 32] += 1;
      }
      __syncthreads();
      if (warp == 0) {                                                    // offsets: channel-major, then warp order
        uint32_t run = 0;
        for (int k = 0; k < n_chars; ++k)
          for (int w = 0; w < POLICY_THREADS / 32; ++w) {
            uint32_t* p = s_cnt + (w * n_chars + k) * 32 + lane;
            const uint32_t t = *p;
            *p = run;
            run += t;
          }
        s_count[lane] = run;
      }
      __syncthreads();
      for (int c = c_lo; c < c_hi; ++c) {
        const uint32_t k = s_lut[mine[c]];
        if (k != 0xFF) {
          const uint32_t pos = cnt[k * 32];
          cnt[k * 32] = pos + 1;
          s_list[pos * 32 + lane] = k * (uint32_t)cells + (uint32_t)c;
        }
      }
      __syncthreads();
      const int count = (int)s_count[lane];
      const int max_count = (int)__reduce_max_sync(0xffffffffu, (unsigned)count);
      policy_hidden_shares_list(s_list + lane, count, max_count, row, s_h, A, R, warp, lane);
    } else {
      policy_hidden_shares_board(mine, chars, n_chars, cells, row, s_h, A, R, warp, lane);
    }
  };
  if (WMODE == W_STAGED) {
    const float4* wp = reinterpret_cast<const float4*>(s_w + j0);
    walk([&](uint32_t d) { return wp[d * 8]; });
  } else if (WMODE == W_GLOBAL_VEC) {
    const float4* wp = reinterpret_cast<const float4*>(w1t + j0);
    walk([&](uint32_t d) { return __ldg(wp + (size_t)d * 8); });
  } else {
    walk([&](uint32_t d) {
      const float* r = w1t + (size_t)d * n_hidden + j0;
      return make_float4(j0 + 0 < n_hidden ? __ldg(r + 0) : 0.0f, j0 + 1 < n_hidden ? __ldg(r + 1) : 0.0f,
                         j0 + 2 < n_hidden ? __ldg(r + 2) : 0.0f, j0 + 3 < n_hidden ? __ldg(r + 3) : 0.0f);
    });
  }
  __syncthreads();
  // ---- the eight shares in warp order, plus b2; sample: warp 0, lane = env (as k_policy_sample) ----
  if (warp == 0) {
    float w[CX_MAX_ACTIONS];
    policy_logits(s_h, R, A, lane, w);
    if (lane < n_here) {
      const int64_t i = e0 + lane;
      if (logits_out) {
#pragma unroll
        for (int a = 0; a < CX_MAX_ACTIONS; ++a)
          if (a < A) logits_out[i * A + a] = w[a];
      }
      float lp;
      const int pick = sample_categorical(w, A, 1, seed, env_offset + (uint64_t)i, step, &lp);
      actions[i] = (uint8_t)pick;
      if (logp) logp[i] = lp;
    }
  }
}

template <int WMODE, bool LIST>
int launch_board_policy(size_t smem, unsigned grid, const uint8_t* d_board, int64_t n, int cells, const uint8_t* d_chars,
                        int n_chars, const float* d_w1t, const float* d_b1, int n_hidden, const float* d_w2,
                        const float* d_b2, int A, uint64_t seed, uint64_t env_offset, const uint64_t* d_step,
                        uint64_t step_offset, uint8_t* d_actions, float* d_logp, float* d_logits, cudaStream_t s) {
  static CxPerDevice configured;
  if (configured.need()) {
    CX_CUDA_OK(cudaFuncSetAttribute(k_policy_sample_board<WMODE, LIST>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)BOARD_POLICY_SMEM_MAX));
    configured.mark();
  }
  k_policy_sample_board<WMODE, LIST><<<grid, POLICY_THREADS, smem, s>>>(d_board, n, cells, d_chars, n_chars, d_w1t,
                                                                         d_b1, n_hidden, d_w2, d_b2, A, seed, env_offset,
                                                                         d_step, step_offset, d_actions, d_logp, d_logits);
  CX_CUDA_OK(cudaGetLastError());
  return CX_OK;
}

}  // namespace

extern "C" int cx_policy_sample_board(const cx_game* g, const uint8_t* d_board, int64_t n, const float* d_w1t,
                                      const float* d_b1, int32_t n_hidden, const float* d_w2, const float* d_b2,
                                      uint64_t seed, uint64_t env_offset, const uint64_t* d_step, uint64_t step_offset,
                                      uint8_t* d_actions, float* d_logp, float* d_logits, void* stream) {
  if (!g || !d_board || !d_w1t || !d_b1 || !d_w2 || !d_b2 || !d_actions || n < 1 || n_hidden < 1 || n_hidden > 32) {
    cx_set_error("cx_policy_sample_board: bad argument (null pointer, n_envs < 1 or n_hidden outside 1..32)");
    return CX_ERR_INVALID_ARG;
  }
  if (g->desc.unoccluded_layers) {
    cx_set_error("cx_policy_sample_board: unoccluded layers (occlusion_in_layers=False) are not a function of the board");
    return CX_ERR_UNSUPPORTED;
  }
  const int cells = g->info.cells, n_chars = g->info.n_chars, A = g->info.n_actions;
  const int64_t grid = (n + 31) / 32;
  if (grid > 0x7fffffff) {
    cx_set_error("cx_policy_sample_board: too many environments for one launch");
    return CX_ERR_INVALID_ARG;
  }
  const size_t boards = (size_t)32 * board_pitch(cells), w_bytes = (size_t)n_chars * cells * 32 * sizeof(float);
  const size_t list = board_list_bytes(cells, n_chars);
  const bool use_list = BOARD_POLICY_SHARES_BYTES + boards + list <= BOARD_POLICY_SMEM_MAX;
  const size_t smem = BOARD_POLICY_SHARES_BYTES + boards + (use_list ? list : 0);   // dense: <= 8,448 + 32 * 4,100 B
  const bool staged = smem + w_bytes <= BOARD_POLICY_STAGE_BUDGET;
  const bool vec = n_hidden == 32 && (reinterpret_cast<uintptr_t>(d_w1t) & 15) == 0;
#define CX_BOARD_POLICY_LAUNCH(MODE, LST, BYTES)                                                                     \
  return launch_board_policy<MODE, LST>(BYTES, (unsigned)grid, d_board, n, cells, g->d_chars, n_chars, d_w1t, d_b1,   \
                                        n_hidden, d_w2, d_b2, A, seed, env_offset, d_step, step_offset, d_actions,    \
                                        d_logp, d_logits, (cudaStream_t)stream)
  if (use_list) {
    if (staged) CX_BOARD_POLICY_LAUNCH(W_STAGED, true, smem + w_bytes);
    if (vec) CX_BOARD_POLICY_LAUNCH(W_GLOBAL_VEC, true, smem);
    CX_BOARD_POLICY_LAUNCH(W_GLOBAL, true, smem);
  }
  if (staged) CX_BOARD_POLICY_LAUNCH(W_STAGED, false, smem + w_bytes);
  if (vec) CX_BOARD_POLICY_LAUNCH(W_GLOBAL_VEC, false, smem);
  CX_BOARD_POLICY_LAUNCH(W_GLOBAL, false, smem);
#undef CX_BOARD_POLICY_LAUNCH
}
