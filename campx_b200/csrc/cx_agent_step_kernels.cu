// Single-agent fast path, ONE Engine.play() per launch (cx_step / cx_step_observations): the kernel an on-device
// policy loop calls once per env-batch step (examples/actor_critic.py:146-173: state = layered_board.float(),
// action = policy(state), game.play(action)).
//
// The fused rollout kernels (cx_agent_kernels.cu, cx_agent_obs_kernels.cu) keep a pre-tiled byte image of their
// envs' boards in shared memory and patch it step by step; staging that image costs more than the single step it
// would serve (15 us for one step of 2^20 envs against 5.5 us of HBM traffic).  For T = 1 nothing needs to persist,
// so this kernel is a stateless COMPOSER over the flat output streams:
//   phase 1  thread = env: the step itself -- one lookup in the (action, cell) transition table built by
//            cx_game_create (action dispatch, toroidal move, wall gate against the last render, first-entry
//            rewards, plot directives: the same table k_agent_rollout uses, so the kernels cannot disagree),
//            time limit / auto reset / episode statistics, state write-back; the cell where the agent is drawn
//            afterwards goes to shared memory (one byte per env);
//   phase 2  the CTA's slice of every output stream is written in 16-byte pieces of the FLAT arrays, a warp store
//            being one aligned 512-byte run: a piece of the board is the static scene at that phase (a 16-byte row
//            of the tiling pattern, L1-resident); a piece of the layered board (campx/rendering.py:204-215,
//            layers[ch] = board == ord(ch), canonical channel order) is the static layered image at that phase,
//            emitted as uint8, float32 or bfloat16 -- the float planes ARE the policy input (actor_critic.py:147,173
//            `layered_board.view(-1).float()`), so no second pass over HBM converts them;
//   phase 3  thread = env again: the agent.  One byte of the board and at most two elements of the layered board
//            (agent plane on, the plane of the character it covers off) are stored over the static streams.
// No table staging (tables are a few hundred bytes, read through L1), two block barriers, no tensor cores (nothing
// here is a contraction).  Envs per CTA are chosen by the launcher so that the grid is a few waves deep at any
// batch size: 32 envs per CTA for a 4,096-env policy loop (128 CTAs), 256 (one thread per env) for 2^20 envs.
#include "cx_agent_common.cuh"

namespace {

struct StepParams {
  CxAgentHeader h;
  const uint8_t* blob;
  uint8_t* cell;
  uint16_t* tstep;
  float* ret;
  double* stats;
  const uint8_t* actions;  // [n]
  float* reward;           // [n]
  float* discount;         // [n] or null
  uint8_t* flags;          // [n]
  uint8_t* board;          // [n, cells]
  void* layered;           // [n, chars, cells] of the LAY element type, or null
  int64_t n;
  int32_t envs_per_cta;    // multiple of 32
  uint64_t inv_cells, inv_lc;  // ceil(2^40 / cells), ceil(2^40 / (n_chars * cells))
  float* perf;             // [n] (PERF)
};

constexpr int ST_THREADS = 256;   // upper bound; small batches launch 128-thread CTAs

// four consecutive bytes of a table starting at any byte offset: two aligned words and a funnel shift
__device__ __forceinline__ uint32_t ldg_u32_unaligned(const uint8_t* base, uint32_t off) {
  const uint32_t* w = reinterpret_cast<const uint32_t*>(base) + (off >> 2);
  const uint32_t lo = __ldg(w), hi = __ldg(w + 1);
  return __funnelshift_r(lo, hi, (off & 3u) * 8u);
}

// set byte `pos` (0..15) of a 16-byte piece held in four words
__device__ __forceinline__ void put_byte(uint32_t (&w)[4], uint32_t pos, uint32_t v) {
  const uint32_t sh = (pos & 3u) * 8u, word = pos >> 2;
#pragma unroll
  for (int j = 0; j < 4; ++j)
    if (word == (uint32_t)j) w[j] = (w[j] & ~(0xFFu << sh)) | (v << sh);
}

// LAY: 0 no layered board, 1 uint8, 2 float32, 4 bfloat16 (the value is the element size except for "none"); PERF
// (TRACK builds of games that track performance): the running performance beside the return
template <bool TRACK, bool PERF, int LAY>
__global__ void __launch_bounds__(ST_THREADS) k_agent_step_flat(const __grid_constant__ StepParams P) {
  extern __shared__ __align__(16) uint8_t s_show[];  // [envs_per_cta] cell where the agent is drawn after the step
  uint8_t* s_stood = s_show + P.envs_per_cta;        // [envs_per_cta] its real cell in that frame (unoccluded layers)
  const CxAgentHeader& H = P.h;
  const int tid = threadIdx.x, nthreads = blockDim.x;
  const uint32_t cells = H.cells, none = cells;
  const int E = P.envs_per_cta;
  const int64_t env0 = (int64_t)blockIdx.x * E;
  const int nenv = (int)min((int64_t)E, P.n - env0);

  asm volatile("griddepcontrol.launch_dependents;");
  const uint32_t* __restrict__ g_tt = reinterpret_cast<const uint32_t*>(P.blob + H.off_tt);
  const float* __restrict__ g_tr = reinterpret_cast<const float*>(P.blob + H.off_tr);
  const float* __restrict__ g_td = reinterpret_cast<const float*>(P.blob + H.off_td);
  const uint8_t* __restrict__ g_basech = P.blob + H.off_basech;
  const uint8_t* __restrict__ g_basek = P.blob + H.off_basek;
  const uint4* __restrict__ g_pat = reinterpret_cast<const uint4*>(P.blob + H.off_pat);
  const uint8_t* __restrict__ g_lay = P.blob + H.off_baselay_wrap;
  const uint32_t stride = H.stride, n_actions = H.n_actions, agent_char = H.agent_char;
  const uint32_t max_steps = H.max_steps > 0 ? (uint32_t)H.max_steps : 0xFFFFFFFFu;
  const bool auto_reset = H.auto_reset != 0, want_discount = P.discount != nullptr;
  // x / cells and x / (chars * cells) by multiplication: q = (x * ceil(2^40 / d)) >> 40, exact while x * d < 2^40
  // (x < 2^22 elements per CTA, d < 2^13)
  const uint64_t inv_cells = P.inv_cells, inv_lc = P.inv_lc;
  auto div_cells = [&](uint32_t x) { return (uint32_t)(((uint64_t)x * inv_cells) >> 40); };
  auto div_lc = [&](uint32_t x) { return (uint32_t)(((uint64_t)x * inv_lc) >> 40); };
  asm volatile("griddepcontrol.wait;" ::: "memory");  // the previous step's state and outputs are complete

  // ---- phase 1: the step of every env of this CTA ----
  LaneStatsT<PERF> st;
  if (TRACK) st.clear();
  for (int el = tid; el < nenv; el += nthreads) {
    const int64_t env = env0 + el;
    const uint32_t cell = min((uint32_t)P.cell[env], none);
    if (P.actions == nullptr) {  // render only (cx_render_observations): the frame of the current state
      s_show[el] = __ldg(P.blob + H.off_shown + cell);
      s_stood[el] = (uint8_t)cell;
      continue;
    }
    const uint32_t a = min((uint32_t)P.actions[env], n_actions);
    const uint32_t idx = a * stride + cell;
    uint32_t e = __ldg(g_tt + idx);
    float r = __ldg(g_tr + idx);
    float dc = want_discount ? __ldg(g_td + (H.td_per_cell ? idx : a)) : 1.0f;
    uint32_t ts = 0;
    float rt = 0.0f, pf = 0.0f;
    if (TRACK) {
      ts = P.tstep[env];
      rt = P.ret[env];
      if (PERF) pf = P.perf[env];
      if (ts & CX_OVER_BIT) {  // auto_reset == 0 and the episode ended: frozen env, board stays as it was drawn
        e = cell | ((uint32_t)__ldg(P.blob + H.off_shown + cell) << 8) | (CX_FROZEN_FLAGS << 16);
        r = 0.0f;
        dc = 0.0f;
      }
    }
    uint32_t p = e & 0xFF;
    const uint32_t show = (e >> 8) & 0xFF;
    s_stood[el] = (uint8_t)p;    // before any auto reset: the frame shows the terminal state
    uint32_t f = cx_tt_flags<PERF>(e);
    // (the address of pf only in PERF builds: taking it in the others changed their register allocation)
    if (TRACK && cx_episode_step<PERF>(f, r, ts, rt, st, max_steps, auto_reset, PERF ? &pf : nullptr, cx_tt_perf(e)))
      p = H.init_cell;
    P.cell[env] = (uint8_t)p;
    if (TRACK) {
      P.tstep[env] = (uint16_t)ts;
      P.ret[env] = rt;
      if (PERF) P.perf[env] = pf;
    }
    P.reward[env] = r;
    if (want_discount) P.discount[env] = dc;
    P.flags[env] = (uint8_t)f;
    s_show[el] = (uint8_t)show;
  }
  __syncthreads();  // the only block barrier

  // ---- phase 2: the output streams.  Every stream is the STATIC image of the game repeated env after env (the
  // scene without the agent; its layered image), so it is written first, 16 bytes of the flat arrays per thread and
  // iteration straight from the L1-resident tables -- no per-piece search for the agent -- and the one to three
  // elements per env that the agent changes are stored over it afterwards, thread = env, behind a block barrier (the
  // lines are still in L2: the small stores merge there).
  {
    const uint32_t nbytes = (uint32_t)nenv * cells, nfull = nbytes >> 4;
    uint8_t* out = P.board + env0 * cells;
    uint32_t ph = ((uint32_t)tid << 4) - div_cells((uint32_t)tid << 4) * cells;   // phase of this thread's first piece
    const uint32_t step = ((uint32_t)nthreads << 4) - div_cells((uint32_t)nthreads << 4) * cells;
#pragma unroll 4
    for (uint32_t k = tid; k < nfull; k += nthreads) {
      *reinterpret_cast<uint4*>(out + (k << 4)) = __ldg(g_pat + ph);  // the static scene from phase `ph` on (wraps)
      ph += step;
      ph = min(ph, ph - cells);
    }
    for (uint32_t b = (nfull << 4) + tid; b < nbytes; b += nthreads)  // ragged tail of the last CTA
      out[b] = __ldg(g_basech + (b - div_cells(b) * cells));
  }
  constexpr uint32_t ES = LAY == 1 ? 1u : (LAY == 2 ? 4u : 2u);  // element size of the layered board
  const uint32_t LC = (uint32_t)H.n_chars * cells;
  uint8_t* lay_out = LAY != 0 ? static_cast<uint8_t*>(P.layered) + env0 * (int64_t)LC * ES : nullptr;
  if (LAY != 0) {
    constexpr uint32_t EPC = 16u / ES;                              // elements per 16-byte piece
    const uint32_t nelem = (uint32_t)nenv * LC, nfull = nelem / EPC;
    uint32_t rem = (uint32_t)tid * EPC - div_lc((uint32_t)tid * EPC) * LC;        // element phase inside the env
    const uint32_t step = (uint32_t)nthreads * EPC - div_lc((uint32_t)nthreads * EPC) * LC;
#pragma unroll 2
    for (uint32_t k = tid; k < nfull; k += nthreads) {
      uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
      for (uint32_t j = 0; j < EPC / 4; ++j) w[j] = ldg_u32_unaligned(g_lay, rem + 4u * j);
      uint4 v;
      if (LAY == 1) {
        v = make_uint4(w[0], w[1], w[2], w[3]);
      } else if (LAY == 2) {  // 4 bytes -> 4 floats (0.0f / 1.0f)
        v = make_uint4((w[0] & 1u) * 0x3F800000u, ((w[0] >> 8) & 1u) * 0x3F800000u,
                       ((w[0] >> 16) & 1u) * 0x3F800000u, (w[0] >> 24) * 0x3F800000u);
      } else {                // 8 bytes -> 8 bfloat16 (0x0000 / 0x3F80)
        v = make_uint4(((w[0] & 1u) | ((w[0] << 8) & 0x10000u)) * 0x3F80u,
                       (((w[0] >> 16) & 1u) | ((w[0] >> 8) & 0x10000u)) * 0x3F80u,
                       ((w[1] & 1u) | ((w[1] << 8) & 0x10000u)) * 0x3F80u,
                       (((w[1] >> 16) & 1u) | ((w[1] >> 8) & 0x10000u)) * 0x3F80u);
      }
      *reinterpret_cast<uint4*>(lay_out + (size_t)k * 16u) = v;
      rem += step;
      rem = min(rem, rem - LC);
    }
    for (uint32_t i = nfull * EPC + tid; i < nelem; i += nthreads) {  // ragged tail of the last CTA
      const uint32_t b = __ldg(g_lay + (i - div_lc(i) * LC)) & 1u;
      if (LAY == 1)
        lay_out[i] = (uint8_t)b;
      else if (LAY == 2)
        reinterpret_cast<uint32_t*>(lay_out)[i] = b * 0x3F800000u;
      else
        reinterpret_cast<uint16_t*>(lay_out)[i] = (uint16_t)(b * 0x3F80u);
    }
  }
  __syncthreads();  // the static streams of this CTA's envs are written: now the agent
  {
    const bool unocc = H.unoccluded != 0;
    const uint32_t agent_off = (uint32_t)H.agent_k * cells;
    auto put = [&](uint32_t i, uint32_t bit) {  // one element of the layered board
      if (LAY == 1)
        lay_out[i] = (uint8_t)bit;
      else if (LAY == 2)
        reinterpret_cast<uint32_t*>(lay_out)[i] = bit * 0x3F800000u;
      else if (LAY == 4)
        reinterpret_cast<uint16_t*>(lay_out)[i] = (uint16_t)(bit * 0x3F80u);
    };
    for (int el = tid; el < nenv; el += nthreads) {
      const uint32_t show = s_show[el];
      if (show != none) (P.board + env0 * cells)[(uint32_t)el * cells + show] = (uint8_t)agent_char;
      if (LAY != 0) {
        // occluded layers follow the board (agent plane on where it is DRAWN, the covered character's plane off);
        // unoccluded layers follow the curtains (agent plane on where the agent STANDS, nothing else changes)
        const uint32_t sh = unocc ? s_stood[el] : show;
        if (sh != none) {
          const uint32_t kb = unocc ? 0xFFu : __ldg(g_basek + sh);   // plane of the covered character (0xFF: none)
          if (kb != 0xFFu) put((uint32_t)el * LC + kb * cells + sh, 0u);
          put((uint32_t)el * LC + agent_off + sh, 1u);
        }
      }
    }
  }

  if (TRACK && P.actions != nullptr) {
    // the env-steps of the whole grid are added once, by its first thread, not by every warp
    if (blockIdx.x == 0 && tid == 0) atomicAdd(cx_stat_stripe(P.stats, 0) + CX_STAT_ENV_STEPS, (double)P.n);
    cx_flush_stats<PERF>(st, P.stats, (uint32_t)(blockIdx.x * (blockDim.x >> 5) + (tid >> 5)), 0u, 0);
  }
}

template <bool TRACK, bool PERF, int LAY>
int launch_step(const StepParams& P, unsigned grid, unsigned block, size_t smem, cudaStream_t s) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  CX_CUDA_OK(cudaLaunchKernelEx(&cfg, k_agent_step_flat<TRACK, PERF, LAY>, P));
  return CX_OK;
}

template <bool TRACK, bool PERF>
int launch_step_lay(int lay, const StepParams& P, unsigned grid, unsigned block, size_t smem, cudaStream_t s) {
  switch (lay) {
    case 0: return launch_step<TRACK, PERF, 0>(P, grid, block, smem, s);
    case 1: return launch_step<TRACK, PERF, 1>(P, grid, block, smem, s);
    case 2: return launch_step<TRACK, PERF, 2>(P, grid, block, smem, s);
    default: return launch_step<TRACK, PERF, 4>(P, grid, block, smem, s);
  }
}

}  // namespace

// The composer writes whole 16-byte pieces: every output array must start 16-byte aligned (CTA slices then do too,
// because a CTA owns a multiple of 32 envs).  Callers fall back to the tile kernels otherwise.
bool cx_agent_step_applies(const cx_game* g, const void* d_board, const void* d_layered) {
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  return g->path == CX_PATH_AGENT && !g->info.n_pickups && al16(d_board) && al16(d_layered);
}

int cx_launch_agent_step(const cx_game* g, void* d_state, int64_t n, const uint8_t* d_actions, float* d_reward,
                         float* d_discount, uint8_t* d_flags, uint8_t* d_board, void* d_layered, int lay_dtype,
                         cudaStream_t s) {
  const CxStateLayout L = cx_layout(g, n);
  uint8_t* base = static_cast<uint8_t*>(d_state);
  StepParams P;
  P.h = g->ah;
  P.blob = g->d_blob;
  P.cell = base + L.off_dyn;
  P.tstep = reinterpret_cast<uint16_t*>(base + L.off_tstep);
  P.ret = reinterpret_cast<float*>(base + L.off_ret);
  P.stats = reinterpret_cast<double*>(base + L.off_stats);
  P.actions = d_actions;
  P.reward = d_reward;
  P.discount = d_discount;
  P.flags = d_flags;
  P.board = d_board;
  P.layered = d_layered;
  P.n = n;
  P.perf = reinterpret_cast<float*>(base + L.off_perf);
  // envs per CTA: a multiple of 32 that makes the grid about four CTAs per SM deep -- 32 for a 4,096-env policy loop
  // (128 CTAs of 128 threads) -- up to 256 with one thread per env (2^20 envs: 4,096 CTAs of 256 threads; fatter
  // CTAs with several envs per thread serialise the state loads and measured 2x slower there)
  int64_t per = (n + (int64_t)g->sm_count * 4 - 1) / ((int64_t)g->sm_count * 4);
  per = (per + 31) / 32 * 32;
  if (per < 32) per = 32;
  if (per > ST_THREADS) per = ST_THREADS;
  P.envs_per_cta = (int32_t)per;
  const unsigned block = per > 128 ? 256u : 128u;
  const uint64_t lc = (uint64_t)g->ah.n_chars * g->ah.cells;
  P.inv_cells = ((1ull << 40) + g->ah.cells - 1) / g->ah.cells;
  P.inv_lc = ((1ull << 40) + lc - 1) / lc;
  const int64_t grid = (n + per - 1) / per;
  if (grid > 0x7fffffff) {
    cx_set_error("cx_step: too many environments for one launch");
    return CX_ERR_INVALID_ARG;
  }
  const int lay = d_layered ? (lay_dtype == CX_DTYPE_U8 ? 1 : (lay_dtype == CX_DTYPE_F32 ? 2 : 4)) : 0;
  const size_t smem = 2 * (size_t)per;
  if (g->info.tracks_performance) return launch_step_lay<true, true>(lay, P, (unsigned)grid, block, smem, s);
  return g->ah.track ? launch_step_lay<true, false>(lay, P, (unsigned)grid, block, smem, s)
                     : launch_step_lay<false, false>(lay, P, (unsigned)grid, block, smem, s);
}
