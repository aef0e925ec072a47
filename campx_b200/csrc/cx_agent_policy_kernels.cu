// The reference's actor-critic ROLLOUT in one launch (examples/actor_critic.py:146-173, BASELINE config 5): for T steps
//     state  = layered_board.view(-1).float()                       actor_critic.py:147,173
//     action ~ Categorical(softmax(action_head(relu(affine1(state)))))   actor_critic.py:64-98
//     board, reward, done = game.play(action)                       campx/engine.py:114-166
// for every env of a single-agent game, with the time limit, auto reset and episode statistics of the other kernels.
//
// Why one kernel.  At the 4,096 envs of config 5 an env-batch step moves 3 MB and is launch-bound: two launches per
// step (cx_policy_sample + cx_step_observations) take 10.5 us under a CUDA graph, most of it launch gaps and the
// re-staging of operands that do not change.  Here a CTA of eight warps OWNS 32 envs for the whole rollout:
//   * W1^T is staged once; the policy input of the CTA's envs lives in shared memory for all T steps (xo[env][d], what
//     the learner gets) and a step changes four floats of it per env (the layered board of a single-agent game is a
//     static image plus the agent, as in k_agent_rollout_obs): nothing is re-read from HBM;
//   * the hidden layer visits only the inputs that are nonzero -- a layered board is one 0/1 plane per character, so
//     one input per cell is set: the static scene's cells (minus the one the agent covers) plus one term of the agent's
//     plane, `cells` + 1 of L x cells inputs -- in ascending input order, which gives the bits of the dense loop of
//     k_policy_sample (cx_policy.cuh); the sampled actions are therefore bit-identical to the two-kernel rollout;
//   * the uniform numbers of the next 64 steps come from all warps at once (Philox does not depend on the state);
//   * nine warps: warps 1-8 run the hidden layer (four hidden units each, lane = env); warp 0, lane = env, is the actor:
//     it sums the logits, samples, looks the step up in the (action, cell) table of k_agent_rollout and publishes where
//     the agent is drawn -- that is all the next hidden layer waits for.  Everything else of the step (time limit,
//     auto reset, statistics, the action / reward / flags / log-prob stores, the four pokes into xo and its bulk store:
//     32 x n_in floats, contiguous in HBM, one cp.async.bulk per step) happens on warp 0 WHILE warps 1-8 already run
//     the next hidden layer.
#include <stdlib.h>

#include "cx_agent_common.cuh"
#include "cx_policy.cuh"

namespace {

constexpr int POLICY_RNG_STEPS = 64;   // steps of uniform numbers generated ahead
constexpr int ROLLOUT_THREADS = POLICY_THREADS + 32;   // warp 0: the actor; warps 1-8: the hidden layer

struct PolicyRolloutParams {
  CxAgentHeader h;
  const uint8_t* blob;
  uint8_t* cell;
  uint16_t* tstep;
  float* ret;
  double* stats;
  const float *w1t, *b1, *w2, *b2;
  int32_t n_hidden;
  float* states;      // [T + 1, n, n_in]: states[t] is the policy input before action t (states[0]: the current frame)
  uint8_t* actions;   // [T, n]
  float* reward;      // [T, n]
  uint8_t* flags;     // [T, n]
  float* logp;        // [T, n] or null
  int64_t n;          // a multiple of 32
  int32_t T;
  uint64_t seed, env_offset, step0;
  const uint64_t* d_step;
  float* perf;        // [n] (PERF)
};

// PERF: the game tracks performance; the running performance lives beside the return
template <bool PERF>
__global__ void __launch_bounds__(ROLLOUT_THREADS) k_agent_policy_rollout(const __grid_constant__ PolicyRolloutParams P) {
  extern __shared__ __align__(16) uint8_t smem[];
  const CxAgentHeader& H = P.h;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int cells = H.cells, L = H.n_chars, n_in = L * cells, A = H.n_actions;
  // shared memory: [tables blob][W1^T [n_in][32]][xo [32][n_in]][logit shares [8][8][33]][random bits [64][32]]
  // [input list [2 * cells]][drawn cell [32]][lane stats]; blob, W1^T and xo are multiples of 16 bytes (xo is the
  // source of the bulk stores), the statistics start 16-aligned
  float* s_w = reinterpret_cast<float*>(smem + H.blob_bytes_ext);
  float* s_o = s_w + (size_t)n_in * 32;
  float* s_h = s_o + (size_t)32 * n_in;
  uint32_t* s_bits = reinterpret_cast<uint32_t*>(s_h + (POLICY_THREADS / 32) * CX_MAX_ACTIONS * POLICY_PITCH);
  uint32_t* s_list = s_bits + POLICY_RNG_STEPS * 32;
  uint32_t* s_drawn = s_list + 2 * cells;
  __shared__ int s_n_list[2];   // static entries in front of the agent's plane, all static entries
  const size_t stats_off = (reinterpret_cast<uint8_t*>(s_drawn + 32) - smem + 15) / 16 * 16;
  LaneStatsT<PERF>& stats = reinterpret_cast<LaneStatsT<PERF>*>(smem + stats_off)[lane];

  const int mw = warp > 0 ? warp - 1 : 0;   // hidden-layer warp index (warp 0 only needs b2 from the small operands)
  const PolicyRegs R = policy_load_small(P.b1, P.w2, P.b2, P.n_hidden, A, mw, lane);
  const uint64_t step_base = (P.d_step ? *P.d_step : 0ull) + P.step0;
  const int64_t n = P.n, e0 = (int64_t)blockIdx.x * 32, env = e0 + lane;
  // ---- stage the tables and W1^T (every 16-byte load requested before the first store) ----
  {
    const uint4* src = reinterpret_cast<const uint4*>(P.blob);
    uint4* dst = reinterpret_cast<uint4*>(smem);
    for (int i = tid; i < H.blob_bytes_ext / 16; i += ROLLOUT_THREADS) dst[i] = src[i];
    const bool w_vec = P.n_hidden == 32 && (reinterpret_cast<uintptr_t>(P.w1t) & 15) == 0;
    if (w_vec) {
      constexpr int DEPTH = 8;
      for (int base = tid; base < n_in * 8; base += DEPTH * ROLLOUT_THREADS) {
        float4 v[DEPTH];
#pragma unroll
        for (int u = 0; u < DEPTH; ++u)
          if (base + u * ROLLOUT_THREADS < n_in * 8) v[u] = __ldg(reinterpret_cast<const float4*>(P.w1t) + base + u * ROLLOUT_THREADS);
#pragma unroll
        for (int u = 0; u < DEPTH; ++u)
          if (base + u * ROLLOUT_THREADS < n_in * 8) reinterpret_cast<float4*>(s_w)[base + u * ROLLOUT_THREADS] = v[u];
      }
    } else {
      for (int k = tid; k < n_in * 32; k += ROLLOUT_THREADS) {
        const int d = k >> 5, j = k & 31;
        s_w[k] = j < P.n_hidden ? __ldg(P.w1t + (size_t)d * P.n_hidden + j) : 0.0f;
      }
    }
  }
  __syncthreads();
  const uint32_t* __restrict__ s_tt = reinterpret_cast<const uint32_t*>(smem + H.off_tt);
  const float* __restrict__ s_tr = reinterpret_cast<const float*>(smem + H.off_tr);
  const uint8_t* __restrict__ s_shown = smem + H.off_shown;
  const uint8_t* __restrict__ s_basek = smem + H.off_basek;
  const uint8_t* __restrict__ s_baselay = smem + H.off_baselay;
  const uint32_t none = cells, agent_k = H.agent_k;
  // ---- the policy input of the static scene; its nonzero inputs, ascending (none of them in the agent's plane) ----
  for (int k = tid; k < n_in * 32; k += ROLLOUT_THREADS) {
    const int d = k >> 5, e = k & 31;
    s_o[e * n_in + d] = (float)s_baselay[d];
  }
  if (tid == 0) {
    int m = 0, before = 0;
    for (int d = 0; d < n_in; ++d) {
      const uint32_t k = (uint32_t)d / (uint32_t)cells, c = (uint32_t)d - k * (uint32_t)cells;
      if (k != agent_k && s_baselay[d]) {
        s_list[m++] = ((uint32_t)d * 8u) | (c << 16);          // row of W1^T as a float4 index | cell
        if (k < agent_k) before = m;
      }
    }
    s_n_list[0] = before;
    s_n_list[1] = m;
  }
  __syncthreads();
  const int n_before = s_n_list[0], n_static = s_n_list[1];
  // ---- warp 0, lane = env: state, the agent in both copies, states[0] ----
  uint32_t cell = none, ts = 0, drawn = none;
  float rt = 0.0f, pf = 0.0f;
  const uint64_t l2pol = l2_evict_first_policy();
  // planes of a frame with the agent drawn at c: its own plane set, the plane of the character it covers cleared
  auto draw = [&](uint32_t c) {
    const uint32_t k = s_basek[c];
    if (k != 0xFF) s_o[lane * n_in + k * cells + c] = 0.0f;
    s_o[lane * n_in + agent_k * cells + c] = 1.0f;
  };
  auto erase = [&](uint32_t c) {
    s_o[lane * n_in + agent_k * cells + c] = 0.0f;
    const uint32_t k = s_basek[c];
    if (k != 0xFF) s_o[lane * n_in + k * cells + c] = 1.0f;
  };
  if (warp == 0) {
    cell = min((uint32_t)P.cell[env], none);
    if (H.track) {
      ts = P.tstep[env];
      rt = P.ret[env];
      if (PERF) pf = P.perf[env];
    }
    stats.clear();
    drawn = s_shown[cell];
    s_drawn[lane] = drawn;
    if (drawn != none) draw(drawn);
    fence_async_smem();
    __syncwarp();
    if (lane == 0) {
      bulk_store_s2g(P.states + e0 * n_in, s_o, (uint32_t)(32 * n_in * sizeof(float)), l2pol);
      bulk_commit();
    }
  }
  __syncthreads();

  const uint32_t stride = H.stride, n_actions = H.n_actions;
  const uint32_t max_steps = H.max_steps > 0 ? (uint32_t)H.max_steps : 0xFFFFFFFFu;
  const uint64_t quad0 = (P.env_offset + (uint64_t)e0) >> 2;   // env_offset is a multiple of 4: the CTA's envs are 8 quads
  // what warp 0 still owes the previous step while the hidden layer of this one runs
  bool owed = false;
  uint32_t o_a = 0, o_f = 0, o_show = none;
  float o_rw = 0.0f, o_lp = 0.0f;
  int o_t = 0;
  auto settle = [&]() {   // warp 0: stores of step o_t, the agent's move in xo, xo -> states[o_t + 1]
    const int64_t row = (int64_t)o_t * n + env;
    P.actions[row] = (uint8_t)o_a;
    __stcs(P.reward + row, o_rw);
    P.flags[row] = (uint8_t)o_f;
    if (P.logp) __stcs(P.logp + row, o_lp);
    if (lane == 0) bulk_wait_read();   // the store of the previous frame has read xo (a whole step ago)
    __syncwarp();
    if (drawn != o_show) {
      if (drawn != none) erase(drawn);
      if (o_show != none) draw(o_show);
      drawn = o_show;
    }
    fence_async_smem();
    __syncwarp();
    if (lane == 0) {
      bulk_store_s2g(P.states + ((int64_t)(o_t + 1) * n + e0) * n_in, s_o, (uint32_t)(32 * n_in * sizeof(float)), l2pol);
      bulk_commit();
    }
  };
  for (int t = 0; t < P.T; ++t) {
    if ((t % POLICY_RNG_STEPS) == 0) {   // the random bits of the next POLICY_RNG_STEPS steps, four envs per Philox call
      for (int k = tid; k < POLICY_RNG_STEPS * 8; k += ROLLOUT_THREADS) {
        const int tt = k >> 3, q = k & 7;
        const CxPhilox4 p = cx_philox4(P.seed ^ 0x5A4D504C45ull, quad0 + (uint64_t)q, step_base + (uint64_t)(t + tt));
        reinterpret_cast<uint4*>(s_bits)[tt * 8 + q] = make_uint4(p.w[0], p.w[1], p.w[2], p.w[3]);
      }
    }
    if (warp > 0) {
      policy_hidden_shares_layered(s_w, s_list, n_before, n_static, agent_k * (uint32_t)cells, (uint32_t)cells,
                                   s_drawn[lane], s_h, A, R, mw, lane);
    } else if (owed) {
      settle();
    }
    __syncthreads();   // the logit shares of step t are complete
    if (warp == 0) {
      float w[CX_MAX_ACTIONS];
      policy_logits(s_h, R, A, lane, w);
      float lp;
      const uint32_t a = (uint32_t)sample_categorical_bits(w, A, 1, s_bits[(t % POLICY_RNG_STEPS) * 32 + lane], &lp);
      // ---- Engine.play(a) of this env: the (action, cell) table of k_agent_rollout ----
      const uint32_t idx = min(a, n_actions) * stride + cell;
      uint32_t e = s_tt[idx];
      float rw = s_tr[idx];
      const bool frozen = H.track && (ts & CX_OVER_BIT);   // auto_reset == 0 and the episode ended
      const uint32_t show = frozen ? s_drawn[lane] : (e >> 8) & 0xFF;
      s_drawn[lane] = show;                                 // all the next hidden layer waits for
      if (frozen) {
        e = cell | (show << 8) | (CX_FROZEN_FLAGS << 16);
        rw = 0.0f;
      }
      uint32_t p = e & 0xFF;
      uint32_t f = cx_tt_flags<PERF>(e);
      if (H.track && cx_episode_step<PERF>(f, rw, ts, rt, stats, max_steps, H.auto_reset, &pf, cx_tt_perf(e)))
        p = H.init_cell;
      cell = p;
      owed = true;
      o_t = t;
      o_a = a;
      o_f = f;
      o_show = show;
      o_rw = rw;
      o_lp = lp;
    }
    __syncthreads();   // the drawn cells of step t are published; the logit shares may be overwritten
  }
  if (warp == 0) {
    if (owed) settle();
    if (lane == 0) bulk_wait_read();   // shared memory must outlive the last bulk read
    __syncwarp();
    P.cell[env] = (uint8_t)cell;
    if (H.track) {
      P.tstep[env] = (uint16_t)ts;
      P.ret[env] = rt;
      if (PERF) P.perf[env] = pf;
      cx_flush_stats<PERF>(stats, P.stats, blockIdx.x, 32u, P.T);
    }
  }
}

size_t policy_rollout_smem(const cx_game* g) {
  const size_t n_in = (size_t)g->ah.n_chars * g->ah.cells;
  return (size_t)g->ah.blob_bytes_ext +
         (n_in * 32 + 32 * n_in + (POLICY_THREADS / 32) * CX_MAX_ACTIONS * POLICY_PITCH) * sizeof(float) +
         (POLICY_RNG_STEPS * 32 + 2 * (size_t)g->ah.cells + 32) * sizeof(uint32_t) + 16 +
         32 * (g->info.tracks_performance ? sizeof(LaneStatsPerf) : sizeof(LaneStats));
}

template <bool PERF>
int launch_policy_rollout(const PolicyRolloutParams& P, unsigned grid, size_t smem, cudaStream_t s) {
  static CxPerDevice configured;
  if (configured.need()) {
    CX_CUDA_OK(cudaFuncSetAttribute(k_agent_policy_rollout<PERF>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    200 * 1024));
    configured.mark();
  }
  k_agent_policy_rollout<PERF><<<grid, ROLLOUT_THREADS, smem, s>>>(P);
  CX_CUDA_OK(cudaGetLastError());
  return CX_OK;
}

}  // namespace

int cx_launch_agent_policy_rollout(const cx_game* g, void* d_state, int64_t n, int32_t T, const float* d_w1t,
                                   const float* d_b1, int32_t n_hidden, const float* d_w2, const float* d_b2, uint64_t seed,
                                   uint64_t env_offset, const uint64_t* d_step, uint64_t step_offset, float* d_states,
                                   uint8_t* d_actions, float* d_reward, uint8_t* d_flags, float* d_logp, cudaStream_t s) {
  if (g->path != CX_PATH_AGENT || g->ah.unoccluded) {
    cx_set_error("cx_rollout_policy: single-agent games with occluded layers only");
    return CX_ERR_UNSUPPORTED;
  }
  const size_t smem = policy_rollout_smem(g);
  if (n % 32 != 0 || (env_offset & 3) != 0 || (reinterpret_cast<uintptr_t>(d_states) & 15) != 0 || smem > 200 * 1024) {
    cx_set_error("cx_rollout_policy: n_envs must be a multiple of 32, env_offset of 4, states 16-byte aligned, the "
                 "policy input small enough for shared memory (%zu bytes needed)", smem);
    return CX_ERR_UNSUPPORTED;
  }
  const CxStateLayout L = cx_layout(g, n);
  uint8_t* base = static_cast<uint8_t*>(d_state);
  PolicyRolloutParams P;
  P.h = g->ah;
  P.blob = g->d_blob;
  P.cell = base + L.off_dyn;
  P.tstep = reinterpret_cast<uint16_t*>(base + L.off_tstep);
  P.ret = reinterpret_cast<float*>(base + L.off_ret);
  P.stats = reinterpret_cast<double*>(base + L.off_stats);
  P.w1t = d_w1t;
  P.b1 = d_b1;
  P.w2 = d_w2;
  P.b2 = d_b2;
  P.n_hidden = n_hidden;
  P.states = d_states;
  P.actions = d_actions;
  P.reward = d_reward;
  P.flags = d_flags;
  P.logp = d_logp;
  P.n = n;
  P.T = T;
  P.seed = seed;
  P.env_offset = env_offset;
  P.step0 = step_offset;
  P.d_step = d_step;
  P.perf = reinterpret_cast<float*>(base + L.off_perf);
  const int64_t grid = n / 32;
  if (grid > 0x7fffffff) {
    cx_set_error("cx_rollout_policy: too many environments for one launch");
    return CX_ERR_INVALID_ARG;
  }
  return g->info.tracks_performance ? launch_policy_rollout<true>(P, (unsigned)grid, smem, s)
                                    : launch_policy_rollout<false>(P, (unsigned)grid, smem, s);
}
