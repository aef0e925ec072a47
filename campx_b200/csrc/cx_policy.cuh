// The acting half of the reference's policy (examples/actor_critic.py:64-98: affine1 -> relu -> action_head -> softmax ->
// Categorical.sample()) as device functions shared by k_policy_sample (cx_aux_kernels.cu: one launch per env-batch step)
// and k_agent_policy_rollout (cx_agent_policy_kernels.cu: the whole T-step rollout in one launch), so that the two give
// the same bits for the same inputs.
#pragma once
#include <math.h>

#include "cx_internal.cuh"
#include "cx_philox.cuh"

namespace {

constexpr int POLICY_THREADS = 256;   // 8 warps: warp w accumulates hidden units 4w .. 4w+3 of its CTA's 32 envs
constexpr int POLICY_PITCH = 33;      // row pitch of the [.][env] tiles in shared memory (conflict-free both ways)

// Categorical(w).sample() for env i (w: probabilities, or logits when is_logits): shared by cx_sample_actions and
// cx_policy_sample, so that the two agree on equal scores.  Returns the action; *logp_out = log p(action).
// the 32 random bits of env g at `step` (Philox4x32-10, one call per four consecutive envs)
__device__ __forceinline__ uint32_t sample_bits(uint64_t seed, uint64_t g, uint64_t step) {
  const CxPhilox4 p = cx_philox4(seed ^ 0x5A4D504C45ull, g >> 2, step);   // a stream apart from cx_fill_actions
  const uint32_t gi = (uint32_t)(g & 3);
  return gi == 0 ? p.w[0] : (gi == 1 ? p.w[1] : (gi == 2 ? p.w[2] : p.w[3]));
}

__device__ __forceinline__ int sample_categorical_bits(float (&w)[CX_MAX_ACTIONS], int A, int is_logits, uint32_t bits,
                                                       float* logp_out) {
  // every loop runs over CX_MAX_ACTIONS with `a < A` predicates and static indices, so that w[] stays in registers
  // (runtime-bounded loops put it in local memory: ~25 dependent LDL/STL per sample, which is most of a step's
  // latency where one warp samples for its CTA, cx_agent_policy_kernels.cu)
  float mx = -INFINITY;
#pragma unroll
  for (int a = 0; a < CX_MAX_ACTIONS; ++a)
    if (a < A) mx = fmaxf(mx, w[a]);
  float total = 0.0f;
#pragma unroll
  for (int a = 0; a < CX_MAX_ACTIONS; ++a) {
    if (a < A) {
      if (is_logits) w[a] = __expf(w[a] - mx);
      w[a] = w[a] > 0.0f ? w[a] : 0.0f;   // negative / NaN weights count as zero
      total += w[a];
    } else {
      w[a] = 0.0f;
    }
  }
  const float u = (float)(bits >> 8) * (1.0f / 16777216.0f) * total;   // [0, total)
  int pick = A - 1;
  float cum = 0.0f;
  bool found = false;
#pragma unroll
  for (int a = 0; a < CX_MAX_ACTIONS; ++a) {
    if (a < A && !found) {
      cum += w[a];
      if (u < cum) {
        pick = a;
        found = true;
      }
    }
  }
#pragma unroll
  for (int a = CX_MAX_ACTIONS - 1; a > 0; --a)   // rounding at the top end must not select a zero-weight action
    if (pick == a && !(w[a] > 0.0f)) pick = a - 1;
  float wp = w[0];
#pragma unroll
  for (int a = 1; a < CX_MAX_ACTIONS; ++a) wp = pick == a ? w[a] : wp;
  *logp_out = __logf(wp / total);
  return pick;
}

__device__ __forceinline__ int sample_categorical(float (&w)[CX_MAX_ACTIONS], int A, int is_logits, uint64_t seed,
                                                  uint64_t g, uint64_t step, float* logp_out) {
  return sample_categorical_bits(w, A, is_logits, sample_bits(seed, g, step), logp_out);
}

// per-lane registers with the small operands: this warp's four b1 entries (lanes 0-3), and in lane a < A row a of this
// warp's 4-column slice of W2 and b2[a]
struct PolicyRegs {
  float b1r, b2r;
  float4 w2r;
};
__device__ __forceinline__ PolicyRegs policy_load_small(const float* __restrict__ b1, const float* __restrict__ w2,
                                                        const float* __restrict__ b2, int n_hidden, int A, int warp, int lane) {
  PolicyRegs R;
  const int j0 = warp * 4;
  R.b1r = 0.0f;
  R.b2r = 0.0f;
  R.w2r = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  if (lane < 4 && j0 + lane < n_hidden) R.b1r = __ldg(b1 + j0 + lane);
  if (lane < A) {
    R.b2r = __ldg(b2 + lane);
    const float* r = w2 + lane * n_hidden + j0;
    R.w2r.x = j0 + 0 < n_hidden ? __ldg(r + 0) : 0.0f;
    R.w2r.y = j0 + 1 < n_hidden ? __ldg(r + 1) : 0.0f;
    R.w2r.z = j0 + 2 < n_hidden ? __ldg(r + 2) : 0.0f;
    R.w2r.w = j0 + 3 < n_hidden ? __ldg(r + 3) : 0.0f;
  }
  return R;
}

// hidden layer: warp w, hidden units 4w .. 4w+3, lane = env (s_w [n_in][32] = W1^T, s_x [n_in][33] = inputs transposed);
// then this warp's share of every action logit -> s_h [8 warps][CX_MAX_ACTIONS][33]
__device__ __forceinline__ void policy_hidden_shares(const float* s_w, const float* s_x, float* s_h, int n_in, int A,
                                                     const PolicyRegs& R, int warp, int lane) {
  const int j0 = warp * 4;
  float acc[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) acc[u] = __shfl_sync(0xffffffffu, R.b1r, u);
  const float* xp = s_x + lane;
  const float4* wp = reinterpret_cast<const float4*>(s_w + j0);
#pragma unroll 8
  for (int d = 0; d < n_in; ++d) {
    const float xv = xp[d * POLICY_PITCH];
    const float4 wa = wp[d * 8];
    acc[0] = fmaf(wa.x, xv, acc[0]);
    acc[1] = fmaf(wa.y, xv, acc[1]);
    acc[2] = fmaf(wa.z, xv, acc[2]);
    acc[3] = fmaf(wa.w, xv, acc[3]);
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) acc[u] = fmaxf(acc[u], 0.0f);                               // relu(affine1(x))
#pragma unroll
  for (int a = 0; a < CX_MAX_ACTIONS; ++a) {
    if (a < A) {                                                                          // warp-uniform
      const float c0 = __shfl_sync(0xffffffffu, R.w2r.x, a), c1 = __shfl_sync(0xffffffffu, R.w2r.y, a);
      const float c2 = __shfl_sync(0xffffffffu, R.w2r.z, a), c3 = __shfl_sync(0xffffffffu, R.w2r.w, a);
      s_h[(warp * CX_MAX_ACTIONS + a) * POLICY_PITCH + lane] = fmaf(c3, acc[3], fmaf(c2, acc[2], fmaf(c1, acc[1], c0 * acc[0])));
    }
  }
}

// The same hidden layer for inputs that are a layered board (campx/rendering.py:204-215: one 0/1 plane per character, so
// exactly one input per cell is 1): only the inputs that are nonzero are visited, in ascending input order -- the static
// scene's set cells (list[i] = row of W1^T as a float4 index d * 8 | cell << 16; the first n_before of them lie in
// front of the agent's plane), minus the one the agent covers, plus ONE term of the agent's plane, W1^T[agent_k * cells +
// drawn], gathered per lane.  Lane = env: `drawn` is the cell where this env's agent is drawn (>= cells: nowhere).
// Skipped inputs are 0 and fmaf(w, 0, acc) == acc, so the result has the bits of policy_hidden_shares on the full row.
__device__ __forceinline__ void policy_hidden_shares_layered(const float* s_w, const uint32_t* s_list, int n_before, int n_static,
                                                             uint32_t agent_row, uint32_t cells, uint32_t drawn, float* s_h,
                                                             int A, const PolicyRegs& R, int mw, int lane) {
  const int j0 = mw * 4;
  float acc[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) acc[u] = __shfl_sync(0xffffffffu, R.b1r, u);
  const float4* wp = reinterpret_cast<const float4*>(s_w + j0);
  auto statics = [&](int lo, int hi) {
#pragma unroll 4
    for (int i = lo; i < hi; ++i) {
      const uint32_t it = s_list[i];
      const float xv = (it >> 16) != drawn ? 1.0f : 0.0f;     // set unless the agent covers the cell
      const float4 wa = wp[it & 0xFFFFu];
      acc[0] = fmaf(wa.x, xv, acc[0]);
      acc[1] = fmaf(wa.y, xv, acc[1]);
      acc[2] = fmaf(wa.z, xv, acc[2]);
      acc[3] = fmaf(wa.w, xv, acc[3]);
    }
  };
  statics(0, n_before);
  {
    const bool on = drawn < cells;
    const float4 wa = wp[(agent_row + (on ? drawn : 0u)) * 8u];
    const float xv = on ? 1.0f : 0.0f;
    acc[0] = fmaf(wa.x, xv, acc[0]);
    acc[1] = fmaf(wa.y, xv, acc[1]);
    acc[2] = fmaf(wa.z, xv, acc[2]);
    acc[3] = fmaf(wa.w, xv, acc[3]);
  }
  statics(n_before, n_static);
#pragma unroll
  for (int u = 0; u < 4; ++u) acc[u] = fmaxf(acc[u], 0.0f);                               // relu(affine1(x))
#pragma unroll
  for (int a = 0; a < CX_MAX_ACTIONS; ++a) {
    if (a < A) {                                                                          // warp-uniform
      const float c0 = __shfl_sync(0xffffffffu, R.w2r.x, a), c1 = __shfl_sync(0xffffffffu, R.w2r.y, a);
      const float c2 = __shfl_sync(0xffffffffu, R.w2r.z, a), c3 = __shfl_sync(0xffffffffu, R.w2r.w, a);
      s_h[(mw * CX_MAX_ACTIONS + a) * POLICY_PITCH + lane] = fmaf(c3, acc[3], fmaf(c2, acc[2], fmaf(c1, acc[1], c0 * acc[0])));
    }
  }
}

// The same hidden layer with the input given as the uint8 BOARD of env `lane` (s_b: its cells, 4-byte aligned, padded to
// whole words): input k * cells + c is (board[c] == chars[k]) (campx/rendering.py:204-215), so the planes are never
// materialised.  Inputs are visited in ascending order, channel-major, each with fmaf(w, x, acc) and x in {0, 1} -- the
// instruction sequence of policy_hidden_shares on the expanded planes, hence its bits.  The four cells of a board word
// are compared at once (__vcmpeq4); row(d) returns this warp's float4 slice of row d of W1^T (shared or global memory).
template <class RowLoad>
__device__ __forceinline__ void policy_hidden_shares_board(const uint8_t* s_b, const uint8_t* __restrict__ chars, int n_chars,
                                                           int cells, const RowLoad& row, float* s_h, int A,
                                                           const PolicyRegs& R, int warp, int lane) {
  float acc[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) acc[u] = __shfl_sync(0xffffffffu, R.b1r, u);
  const uint32_t* bw = reinterpret_cast<const uint32_t*>(s_b);
  const int words = cells >> 2;
  auto term = [&](int d, bool on) {
    const float4 wa = row(d);
    const float xv = on ? 1.0f : 0.0f;
    acc[0] = fmaf(wa.x, xv, acc[0]);
    acc[1] = fmaf(wa.y, xv, acc[1]);
    acc[2] = fmaf(wa.z, xv, acc[2]);
    acc[3] = fmaf(wa.w, xv, acc[3]);
  };
  for (int k = 0; k < n_chars; ++k) {
    const uint32_t ch = __ldg(chars + k), pat = ch * 0x01010101u;
    const int base = k * cells;
#pragma unroll 2
    for (int q = 0; q < words; ++q) {
      const uint32_t m = __vcmpeq4(bw[q], pat);                // 0xFF in every byte that shows chars[k]
#pragma unroll
      for (int u = 0; u < 4; ++u) term(base + 4 * q + u, (m >> (8 * u)) & 1u);
    }
    for (int c = words * 4; c < cells; ++c) term(base + c, s_b[c] == ch);
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) acc[u] = fmaxf(acc[u], 0.0f);                               // relu(affine1(x))
#pragma unroll
  for (int a = 0; a < CX_MAX_ACTIONS; ++a) {
    if (a < A) {                                                                          // warp-uniform
      const float c0 = __shfl_sync(0xffffffffu, R.w2r.x, a), c1 = __shfl_sync(0xffffffffu, R.w2r.y, a);
      const float c2 = __shfl_sync(0xffffffffu, R.w2r.z, a), c3 = __shfl_sync(0xffffffffu, R.w2r.w, a);
      s_h[(warp * CX_MAX_ACTIONS + a) * POLICY_PITCH + lane] = fmaf(c3, acc[3], fmaf(c2, acc[2], fmaf(c1, acc[1], c0 * acc[0])));
    }
  }
}

// The same hidden layer visiting only the SET inputs of env `lane`: s_list[i * 32] (i < count) are their input indices in
// ascending order -- at most one per cell, fewer where a byte is no character of the game -- and row(d) returns this
// warp's float4 slice of row d of W1^T.  The loop runs to the warp's largest count; a lane past its own adds
// fmaf(w, 0, acc).  Skipped inputs are 0 and fmaf(w, 0, acc) == acc, so the result has the bits of policy_hidden_shares
// on the expanded planes (as in policy_hidden_shares_layered).
template <class RowLoad>
__device__ __forceinline__ void policy_hidden_shares_list(const uint32_t* s_list, int count, int max_count, const RowLoad& row,
                                                          float* s_h, int A, const PolicyRegs& R, int warp, int lane) {
  float acc[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) acc[u] = __shfl_sync(0xffffffffu, R.b1r, u);
#pragma unroll 4
  for (int i = 0; i < max_count; ++i) {
    const bool on = i < count;
    const float4 wa = row(on ? s_list[i * 32] : 0u);
    const float xv = on ? 1.0f : 0.0f;
    acc[0] = fmaf(wa.x, xv, acc[0]);
    acc[1] = fmaf(wa.y, xv, acc[1]);
    acc[2] = fmaf(wa.z, xv, acc[2]);
    acc[3] = fmaf(wa.w, xv, acc[3]);
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) acc[u] = fmaxf(acc[u], 0.0f);                               // relu(affine1(x))
#pragma unroll
  for (int a = 0; a < CX_MAX_ACTIONS; ++a) {
    if (a < A) {                                                                          // warp-uniform
      const float c0 = __shfl_sync(0xffffffffu, R.w2r.x, a), c1 = __shfl_sync(0xffffffffu, R.w2r.y, a);
      const float c2 = __shfl_sync(0xffffffffu, R.w2r.z, a), c3 = __shfl_sync(0xffffffffu, R.w2r.w, a);
      s_h[(warp * CX_MAX_ACTIONS + a) * POLICY_PITCH + lane] = fmaf(c3, acc[3], fmaf(c2, acc[2], fmaf(c1, acc[1], c0 * acc[0])));
    }
  }
}

// the eight shares summed in warp order, plus b2: the action logits of env `lane` (call with all 32 lanes of a warp)
__device__ __forceinline__ void policy_logits(const float* s_h, const PolicyRegs& R, int A, int lane, float (&w)[CX_MAX_ACTIONS]) {
#pragma unroll
  for (int a = 0; a < CX_MAX_ACTIONS; ++a) {
    w[a] = 0.0f;
    if (a < A) {
      float sum = __shfl_sync(0xffffffffu, R.b2r, a);
#pragma unroll
      for (int q = 0; q < POLICY_THREADS / 32; ++q) sum += s_h[(q * CX_MAX_ACTIONS + a) * POLICY_PITCH + lane];
      w[a] = sum;
    }
  }
}

}  // namespace
