// Episode bookkeeping shared by every rollout kernel: what happens to an env's step counter, running return and
// episode statistics on each env-step, and the end-of-launch flush of the statistics into their stripe
// (cx_internal.cuh: CX_STAT_STRIPES).  The game rules live in each kernel's step; only this bookkeeping is common.
//
// Games that track the hidden safety performance (cx_game_desc::perf_regions) run PERF builds of the single-agent
// kernels: the PERF variants below keep each env's running performance `pf` beside its running return and follow the
// same episode rules with it.
#pragma once
#include <type_traits>

#include "cx_internal.cuh"

namespace {

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// atomic max on a double that is only ever raised (stats slots start at -inf)
__device__ __forceinline__ void atomic_max_double(double* addr, double v) {
  unsigned long long* a = reinterpret_cast<unsigned long long*>(addr);
  unsigned long long old = *a;
  while (__longlong_as_double((long long)old) < v) {
    const unsigned long long assumed = old;
    old = atomicCAS(a, assumed, (unsigned long long)__double_as_longlong(v));
    if (old == assumed) break;
  }
}

// The episodes one lane finished during a launch.  The multi-step agent kernels keep it in shared memory (touched only
// when an episode ends, about once per hundred steps, so it costs no registers in the step loop); k_agent_step_flat and
// k_generic_rollout keep it in registers.
struct LaneStats {
  double sum, sumsq;
  uint32_t cnt, len;
  float mx, negmn;
  __device__ __forceinline__ void clear() {
    sum = sumsq = 0.0;
    cnt = len = 0;
    mx = negmn = -INFINITY;
  }
  __device__ __forceinline__ void episode(float ret, uint32_t steps) {
    cnt += 1;
    len += steps;
    sum += (double)ret;
    sumsq += (double)ret * (double)ret;
    mx = fmaxf(mx, ret);
    negmn = fmaxf(negmn, -ret);
  }
};

// ... and, in PERF builds, the sum of their performance (a separate type: LaneStats keeps its size and layout)
struct LaneStatsPerf : LaneStats {
  double perf;
  __device__ __forceinline__ void clear() {
    LaneStats::clear();
    perf = 0.0;
  }
  __device__ __forceinline__ void episode(float ret, uint32_t steps, float pf) {
    LaneStats::episode(ret, steps);
    perf += (double)pf;
  }
};
template <bool PERF>
using LaneStatsT = typename std::conditional<PERF, LaneStatsPerf, LaneStats>::type;

// A transition word of the agent tables (CxAgentHeader::off_tt): the step's flags, and its performance (PERF builds;
// the top byte is 0 in the tables of every other game, so their builds take the flags as e >> 16)
template <bool PERF>
__device__ __forceinline__ uint32_t cx_tt_flags(uint32_t e) {
  return PERF ? (e >> 16) & 0xFFu : e >> 16;
}
__device__ __forceinline__ float cx_tt_perf(uint32_t e) { return (float)((int32_t)e >> 24); }

// The step of a frozen env (auto_reset == 0 and its episode has ended: CX_OVER_BIT in the step counter) goes nowhere:
// the env keeps its state and its frame, earns reward 0 and discount 0, and reports these flags.
constexpr uint32_t CX_FROZEN_FLAGS = CX_FLAG_ALREADY_OVER | CX_FLAG_REWARD_NONE;

// The bookkeeping of one env-step, after the game's step produced the flags `f` and reward `r`.  A step that counts
// (no BAD_ACTION, not ALREADY_OVER) advances the step counter `ts` (15 bits, saturating at CX_STEP_MAX) and the
// running return `rt`, and is TRUNCATED when it reaches `max_steps` (0xFFFFFFFF: no time limit) without terminating.
// An episode that ends is added to `stats`; then the env either restarts (auto_reset: counter and return cleared,
// true returned, the caller resets the game state) or freezes (CX_OVER_BIT set).
// PERF: the step's performance `dp` is added to the running performance `*pf` like the reward to `rt` (the terminal
// step counts), the episode's total goes to `stats`, and an auto reset clears it; a frozen env keeps it.
template <bool PERF = false>
__device__ __forceinline__ bool cx_episode_step(uint32_t& f, float r, uint32_t& ts, float& rt, LaneStatsT<PERF>& stats,
                                                uint32_t max_steps, bool auto_reset, float* pf = nullptr,
                                                float dp = 0.0f) {
  if (f & (CX_FLAG_BAD_ACTION | CX_FLAG_ALREADY_OVER)) return false;
  const uint32_t steps = min(ts + 1u, (uint32_t)CX_STEP_MAX);
  rt += r;
  if constexpr (PERF) *pf += dp;
  if (!(f & CX_FLAG_TERMINATED) && steps >= max_steps) f |= CX_FLAG_TRUNCATED;   // time limit (SURVEY H4)
  ts = steps;
  if (!(f & (CX_FLAG_TERMINATED | CX_FLAG_TRUNCATED))) return false;
  if constexpr (PERF)
    stats.episode(rt, steps, *pf);
  else
    stats.episode(rt, steps);
  if (auto_reset) {   // the next play() starts from the its_showtime state
    ts = 0;
    rt = 0.0f;
    if constexpr (PERF) *pf = 0.0f;
    return true;
  }
  ts |= CX_OVER_BIT;
  return false;
}

// All 32 lanes of a warp, once per launch: add the warp's episodes and its `envs` x `steps` env-steps to statistics
// stripe `key`.  The env-steps are passed as two integers and multiplied in lane 0 only: a double computed by the
// caller stays live across the reductions and cost the 64-env tile build two registers.  PERF: also the performance
// sum of the warp's episodes (CX_STAT_PERFORMANCE_SUM).
template <bool PERF = false>
__device__ __forceinline__ void cx_flush_stats(const LaneStatsT<PERF>& s, double* stats, uint32_t key, uint32_t envs,
                                               int32_t steps) {
  const double cnt = warp_sum((double)s.cnt), len = warp_sum((double)s.len);
  const double sum = warp_sum(s.sum), sumsq = warp_sum(s.sumsq);
  const float mx = warp_max(s.mx), ngmn = warp_max(s.negmn);
  double perf = 0.0;
  if constexpr (PERF) perf = warp_sum(s.perf);
  if ((threadIdx.x & 31) == 0) {
    double* sp = cx_stat_stripe(stats, key);
    if (cnt > 0.0) {
      if constexpr (PERF) atomicAdd(sp + CX_STAT_PERFORMANCE_SUM, perf);
      atomicAdd(sp + CX_STAT_EPISODES, cnt);
      atomicAdd(sp + CX_STAT_RETURN_SUM, sum);
      atomicAdd(sp + CX_STAT_RETURN_SUMSQ, sumsq);
      atomicAdd(sp + CX_STAT_LENGTH_SUM, len);
      atomic_max_double(sp + CX_STAT_RETURN_MAX, (double)mx);
      atomic_max_double(sp + CX_STAT_NEG_RETURN_MIN, (double)ngmn);
    }
    if (envs != 0) atomicAdd(sp + CX_STAT_ENV_STEPS, (double)envs * (double)steps);
  }
}

}  // namespace
