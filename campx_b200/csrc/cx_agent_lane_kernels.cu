// Single-agent fast path for SMALL batches: fused T-step Engine.play(), lane = env.
//
// Same step as k_agent_rollout (cx_agent_kernels.cu: one (action, cell) table look-up = action dispatch, toroidal move,
// wall gate, entry rewards, directives -- examples/boat_race.py:35-91, campx/plot.py:161-211, engine.py:285-290 --
// then the painter's algorithm collapsed to two byte pokes into a pre-tiled image of the static scene,
// engine.py:306-321), written for the regime where that kernel is NOT bandwidth-bound.
//
// Why a third build.  BASELINE config 1 (Demo 1, 65,536 envs) gives an SM 443 envs: one step of the whole batch is
// 2 MB, 0.31 us at the HBM peak = 620 SM clocks.  The tile kernels spend more than that on the step's dependent
// instruction chain: the 64-envs-per-warp build issues 214 warp instructions per warp-step with 7 warps per SM
// (ncu: issue slots 30 % busy, 4.4 stall cycles per issue, `wait` = fixed-latency dependencies on top), and every TMA
// bulk store costs its issuing warp ~240 clocks whatever its size (scripts/chain_probe.cu: STS + fence.proxy.async +
// UBLKCP + wait_group.read with two tiles = 239 clocks per iteration for 800, 1,600 or 6,400 bytes; the fence alone is
// 13-27 clocks and does not wait for global stores).  So for small batches this kernel
//   * gives every env its own lane (32 envs per warp: twice the warps of the 64-env build, no per-quad unpacking),
//   * keeps the step's common case to a handful of instructions: the rare events (episode end, time limit, bad action,
//     frozen env) are ONE test and one out-of-line branch,
//   * ships the warp's board tile (32 * cells bytes, a 32-byte-aligned run of whole sectors) with LDS.128 -> STG.128
//     straight from the generic proxy: no proxy fence, no TMA issue latency, no read-wait; two tiles alternate so that
//     one __syncwarp per step orders the pokes of step t+2 behind the reads of step t.
// Large batches stay on k_agent_rollout (TMA bulk stores: fewer LSU instructions once the SM is full of warps).
#include "cx_agent_common.cuh"
#include "cx_philox.cuh"

namespace {

struct LaneParams {
  CxAgentHeader h;
  const uint8_t* blob;
  uint8_t* cell;
  uint16_t* tstep;
  float* ret;
  double* stats;
  const uint8_t* actions;  // [T, n]
  float* reward;           // [T, n]
  float* discount;         // [T, n] or null
  uint8_t* flags;          // [T, n]
  uint8_t* board;          // [T, n, cells]
  int64_t n;               // envs of the batch = row stride of the [T, n] arrays (n * cells a multiple of 16)
  int64_t env_base;        // this launch covers envs [env_base, n): the whole batch, or the rest behind the whole tiles
                           // of k_agent_rollout; env_base is a multiple of 32 and the last warp may hold 16 envs only
  int32_t T;
  uint64_t seed, env_offset, t0;
  uint8_t* actions_out;    // SYNTH: [T, n] or null
  float* perf;             // [n] (PERF)
};

constexpr int LANE_MAX_WARPS = 4;
constexpr int LANE_UNR = 4;   // steps per unrolled group (tile parity and action registers are indexed statically)

// shared-memory accesses by 32-bit shared-window address: the table reads carry no ordering (read-only data, free to
// schedule), the tile accesses are ordered against __syncwarp by their memory clobber
__device__ __forceinline__ uint32_t lds_tab_u32(uint32_t a) {
  uint32_t v;
  asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ float lds_tab_f32(uint32_t a) {
  float v;
  asm("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ uint32_t lds_tab_u8(uint32_t a) {
  uint32_t v;
  asm("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts_tile_u8(uint32_t a, uint32_t v) {
  asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ uint4 lds_tile_v4(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
  return v;
}

// DISC: the game can change the discount (a [T, n] discount stream is written); SMALL: boards of up to 32 cells (at
// most two 16-byte chunks of the warp's tile per lane); PERF (TRACK builds of games that track performance): the
// running performance beside the return
template <bool TRACK, bool PERF, bool SYNTH, bool DISC, bool SMALL>
__global__ void __launch_bounds__(LANE_MAX_WARPS * 32) k_agent_rollout_lane(const __grid_constant__ LaneParams P) {
  extern __shared__ __align__(16) uint8_t smem[];
  const CxAgentHeader& H = P.h;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, WARPS = blockDim.x >> 5;
  const int cells = H.cells;

  asm volatile("griddepcontrol.launch_dependents;");
  {
    const uint4* src = reinterpret_cast<const uint4*>(P.blob);
    uint4* dst = reinterpret_cast<uint4*>(smem);
    for (int i = tid; i < H.blob_bytes / 16; i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();  // the only block barrier

  const int64_t n = P.n;
  const int64_t env0 = P.env_base + ((int64_t)blockIdx.x * WARPS + warp) * 32;
  if (env0 >= n) return;
  const int64_t env = env0 + lane;
  const int nenv = (int)min((int64_t)32, n - env0);   // 32, or 16 in the last warp of a batch with n % 32 == 16
  const bool mine = lane < nenv;

  const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(smem);
  const uint32_t a_tt = sbase + H.off_tt, a_tr = sbase + H.off_tr, a_td = sbase + H.off_td;
  const uint32_t a_basech = sbase + H.off_basech;
  const uint32_t stride = H.stride, n_actions = H.n_actions;
  const uint32_t agent_char = (uint32_t)H.agent_char & 0xFF;
  const uint32_t none = cells;
  // the step counter's common case ends one short of the time limit / of saturation
  const uint32_t max_steps = H.max_steps > 0 ? (uint32_t)H.max_steps : 0xFFFFFFFFu;
  const uint32_t limit = min(max_steps, (uint32_t)CX_STEP_MAX);

  // two tiles per warp, back to back: 2 * 32 boards of the static scene, written as 16-byte pattern chunks
  const int tile_bytes = 32 * cells, nch = tile_bytes / 16;   // 32 * cells is a multiple of 32
  const int nch_here = nenv * cells / 16;                     // chunks of this warp's boards (nenv is a multiple of 16)
  const int tile0 = H.blob_bytes + warp * 2 * tile_bytes;     // byte offset of this warp's tile 0 in smem[]
  {
    const uint4* pat = reinterpret_cast<const uint4*>(smem + H.off_pat);
    uint4* t16 = reinterpret_cast<uint4*>(smem + tile0);
    for (int k = lane; k < 2 * nch; k += 32) t16[k] = pat[(16 * k) % cells];
  }
  __syncwarp();

  asm volatile("griddepcontrol.wait;" ::: "memory");
  uint32_t cell = mine ? min((uint32_t)P.cell[env], none) : none;
  uint32_t ts = 0;
  float rt = 0.0f, pf = 0.0f;
  if (TRACK && mine) {
    ts = P.tstep[env];
    rt = P.ret[env];
    if (PERF) pf = P.perf[env];
  }
  const uint32_t a_mine = sbase + tile0 + lane * cells;   // this env's board in tile 0; tile 1 is tile_bytes further
  const uint32_t a_copy = sbase + tile0 + lane * 16;      // this lane's first chunk of tile 0
  uint32_t drawn[2];
  drawn[0] = drawn[1] = smem[H.off_shown + cell];
  if (drawn[0] != none) {
    sts_tile_u8(a_mine + drawn[0], agent_char);
    sts_tile_u8(a_mine + tile_bytes + drawn[0], agent_char);
  }
  LaneStatsT<PERF>& stats = reinterpret_cast<LaneStatsT<PERF>*>(smem + H.blob_bytes + (size_t)WARPS * 2 * tile_bytes)[tid];
  if (TRACK) stats.clear();

  // actions: one group of LANE_UNR steps is in flight while the previous one is consumed; running row pointer
  const uint8_t* p_act = SYNTH ? nullptr : P.actions + env;
  int t_fetch = 0;
  auto fetch_action = [&]() -> uint32_t {
    uint32_t a = 0u;
    if (t_fetch < P.T && mine) {
      if (SYNTH) {
        a = cx_synth_action(P.seed, P.env_offset + (uint64_t)env, P.t0 + (uint64_t)t_fetch, n_actions);
        if (P.actions_out) P.actions_out[(int64_t)t_fetch * n + env] = (uint8_t)a;
      } else {
        a = __ldcs(p_act);
        p_act += n;
      }
    }
    ++t_fetch;
    return a;
  };
  uint32_t act[LANE_UNR], act_next[LANE_UNR];
#pragma unroll
  for (int u = 0; u < LANE_UNR; ++u) act[u] = fetch_action();

  // running pointers: one 64-bit add per stream and step
  float* p_rw = P.reward + env;
  float* p_dc = DISC ? P.discount + env : nullptr;
  uint8_t* p_fl = P.flags + env;
  uint4* p_bd = reinterpret_cast<uint4*>(P.board + env0 * cells) + lane;
  const int64_t bd_step = n * cells / 16;   // uint4 per [n, cells] row: n % 32 == 0
  const bool one = lane < nch_here, two = lane + 32 < nch_here;   // SMALL: this lane copies a first / a second chunk

  for (int t0 = 0; t0 < P.T; t0 += LANE_UNR) {
#pragma unroll
    for (int u = 0; u < LANE_UNR; ++u) act_next[u] = fetch_action();
#pragma unroll
    for (int u = 0; u < LANE_UNR; ++u) {
      if (t0 + u >= P.T) break;
      // ---- the env's step: one table look-up.  Lanes without an env (last warp of a batch with n % 32 == 16) step an
      // empty mask alongside -- branch-free; their stores are predicated off and their statistics dropped at the end ----
      const uint32_t a = min(act[u], n_actions);
      const uint32_t idx4 = (a * stride + cell) * 4u;
      const uint32_t e = lds_tab_u32(a_tt + idx4);
      float rw = lds_tab_f32(a_tr + idx4);
      float dc = 1.0f;
      if (DISC) dc = lds_tab_f32(a_td + (H.td_per_cell ? idx4 : a * 4u));
      uint32_t f = cx_tt_flags<PERF>(e);
      uint32_t p = e & 0xFF, show = (e >> 8) & 0xFF;
      if (TRACK) {
        const uint32_t steps = ts + 1u;
        // rare: episode end / bad action / frozen env (flag bits or bit 15 of the counter), time limit, saturation
        const uint32_t special = (f & (CX_FLAG_TERMINATED | CX_FLAG_BAD_ACTION | CX_FLAG_ALREADY_OVER)) | (ts & CX_OVER_BIT);
        if (special == 0 && steps < limit) {
          ts = steps;
          rt += rw;
          if (PERF) pf += cx_tt_perf(e);
        } else {
          if (ts & CX_OVER_BIT) {  // auto_reset == 0 and the episode ended: frozen env
            p = cell;
            show = drawn[(u + 1) & 1];   // where the last frame drew it
            f = CX_FROZEN_FLAGS;
            rw = 0.0f;
            dc = 0.0f;
          }
          if (cx_episode_step<PERF>(f, rw, ts, rt, stats, max_steps, H.auto_reset, &pf, cx_tt_perf(e))) p = H.init_cell;
        }
      }
      cell = p;
      if (mine) __stcs(p_rw, rw);
      p_rw += n;
      if (DISC) {
        if (mine) __stcs(p_dc, dc);
        p_dc += n;
      }
      if (mine) *p_fl = (uint8_t)f;
      p_fl += n;

      // ---- the boards: poke tile (t & 1), then the warp copies it out, 512 contiguous bytes per instruction ----
      const uint32_t toff = (u & 1) * tile_bytes;
      const uint32_t was = drawn[u & 1];
      if (was != show) {
        if (was != none) sts_tile_u8(a_mine + toff + was, lds_tab_u8(a_basech + was));
        if (show != none) sts_tile_u8(a_mine + toff + show, agent_char);
        drawn[u & 1] = show;
      }
      __syncwarp();
      if (SMALL) {
        if (one) __stcs(p_bd, lds_tile_v4(a_copy + toff));
        if (two) __stcs(p_bd + 32, lds_tile_v4(a_copy + toff + 512));
      } else {
        for (int k = 0; k + lane < nch_here; k += 32) __stcs(p_bd + k, lds_tile_v4(a_copy + toff + k * 16));
      }
      p_bd += bd_step;
    }
#pragma unroll
    for (int u = 0; u < LANE_UNR; ++u) act[u] = act_next[u];
  }

  if (mine) P.cell[env] = (uint8_t)cell;
  if (TRACK) {
    if (mine) {
      P.tstep[env] = (uint16_t)ts;
      P.ret[env] = rt;
      if (PERF) P.perf[env] = pf;
    } else {
      stats.clear();   // whatever the empty mask of a lane without an env "played"
    }
    cx_flush_stats<PERF>(stats, P.stats, (uint32_t)(blockIdx.x * WARPS + warp), (uint32_t)nenv, P.T);
  }
}

size_t lane_smem_bytes(const cx_game* g, int warps) {
  const size_t stats_bytes = g->info.tracks_performance ? sizeof(LaneStatsPerf) : sizeof(LaneStats);
  return (size_t)g->ah.blob_bytes + (size_t)warps * 2 * 32 * g->ah.cells +
         (g->ah.track ? (size_t)warps * 32 * stats_bytes : 0);
}

template <bool TRACK, bool PERF, bool SYNTH, bool DISC, bool SMALL>
int launch_lane(const LaneParams& P, unsigned grid, unsigned block, size_t smem, bool pdl, cudaStream_t s) {
  static CxPerDevice configured;
  if (configured.need()) {
    CX_CUDA_OK(cudaFuncSetAttribute(k_agent_rollout_lane<TRACK, PERF, SYNTH, DISC, SMALL>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    227 * 1024));
    configured.mark();
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  CX_CUDA_OK(cudaLaunchKernelEx(&cfg, k_agent_rollout_lane<TRACK, PERF, SYNTH, DISC, SMALL>, P));
  return CX_OK;
}

}  // namespace

// batches of a multiple of 16 envs (the last warp may hold 16), every [T, n] / [T, n, cells] row 16-byte aligned,
// tiles that fit shared memory
bool cx_agent_lane_applies(const cx_game* g, int64_t n, const void* d_actions, const void* d_actions_out,
                           const void* d_reward, const void* d_discount, const void* d_flags, const void* d_board) {
  auto al16 = [](const void* p) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  return g->path == CX_PATH_AGENT && !g->info.n_pickups && n > 0 && n % 16 == 0 && lane_smem_bytes(g, 1) <= 64 * 1024 && al16(d_actions) &&
         al16(d_actions_out) && al16(d_reward) && al16(d_discount) && al16(d_flags) && al16(d_board);
}

int cx_launch_agent_rollout_lane(const cx_game* g, void* d_state, int64_t n, int32_t T, const uint8_t* d_actions,
                                 const CxSynth& synth, float* d_reward, float* d_discount, uint8_t* d_flags,
                                 uint8_t* d_board, cudaStream_t s, int64_t env_base) {
  const CxStateLayout L = cx_layout(g, n);
  uint8_t* base = static_cast<uint8_t*>(d_state);
  LaneParams P;
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
  P.n = n;
  P.env_base = env_base;
  P.T = T;
  P.seed = synth.seed;
  P.env_offset = synth.env_offset;
  P.t0 = synth.t0;
  P.actions_out = synth.actions_out;
  P.perf = reinterpret_cast<float*>(base + L.off_perf);
  const int64_t warps = (n - env_base + 31) / 32;
  // warps per CTA: 4, fewer while that leaves the grid under ~8 CTAs per SM (small grids spread more evenly)
  int wpc = LANE_MAX_WARPS;
  while (wpc > 1 && (warps + wpc - 1) / wpc < (int64_t)g->sm_count * 8) wpc >>= 1;
  const int64_t grid = (warps + wpc - 1) / wpc;
  if (grid > 0x7fffffff) {
    cx_set_error("cx_rollout: too many environments for one launch");
    return CX_ERR_INVALID_ARG;
  }
  const size_t smem = lane_smem_bytes(g, wpc);
  const bool track = g->ah.track != 0;
  // Programmatic dependent launch lets the next launch's CTAs become resident (and stage their tables) while this one
  // runs.  For grids of 12-30 one-warp CTAs per SM that costs more than it hides -- the early CTAs take their slots
  // wherever room is, and the launch then runs unevenly spread over the SMs: Demo 1, 32 / 100 steps per launch, us per
  // launch with / without: 8,192 envs 9.1 / 10.8, 32,768 12.3 / 12.2, 65,536 18.9 / 16.1 (100 steps: 51.8 / 40.7),
  // 98,304 23.6 / 21.8, 2^17 29.3 / 28.5, 2^18 50.0 / 50.4.
  const int64_t warps_per_sm = warps / g->sm_count;
  const bool pdl = !(warps_per_sm >= 12 && warps_per_sm <= 30);
  const unsigned blk = 32u * wpc;
  // SMALL needs a first chunk for every lane: 32 <= chunks per tile <= 64, i.e. boards of 16..32 cells
  // TRACK 8, PERF 16 (with TRACK), SYNTH 4, DISC 2, SMALL 1
  const int sel = (track ? 8 : 0) | (g->info.tracks_performance ? 16 : 0) | (synth.on ? 4 : 0) | (d_discount ? 2 : 0) |
                  ((g->ah.cells >= 16 && g->ah.cells <= 32) ? 1 : 0);
  int rc = CX_ERR_INVALID_ARG;
  switch (sel) {
#define CX_LANE_CASE(i, a, p, b, c, d) \
  case i: rc = launch_lane<a, p, b, c, d>(P, (unsigned)grid, blk, smem, pdl, s); break;
    CX_LANE_CASE(0, false, false, false, false, false) CX_LANE_CASE(1, false, false, false, false, true)
    CX_LANE_CASE(2, false, false, false, true, false) CX_LANE_CASE(3, false, false, false, true, true)
    CX_LANE_CASE(4, false, false, true, false, false) CX_LANE_CASE(5, false, false, true, false, true)
    CX_LANE_CASE(6, false, false, true, true, false) CX_LANE_CASE(7, false, false, true, true, true)
    CX_LANE_CASE(8, true, false, false, false, false) CX_LANE_CASE(9, true, false, false, false, true)
    CX_LANE_CASE(10, true, false, false, true, false) CX_LANE_CASE(11, true, false, false, true, true)
    CX_LANE_CASE(12, true, false, true, false, false) CX_LANE_CASE(13, true, false, true, false, true)
    CX_LANE_CASE(14, true, false, true, true, false) CX_LANE_CASE(15, true, false, true, true, true)
    CX_LANE_CASE(24, true, true, false, false, false) CX_LANE_CASE(25, true, true, false, false, true)
    CX_LANE_CASE(26, true, true, false, true, false) CX_LANE_CASE(27, true, true, false, true, true)
    CX_LANE_CASE(28, true, true, true, false, false) CX_LANE_CASE(29, true, true, true, false, true)
    CX_LANE_CASE(30, true, true, true, true, false) CX_LANE_CASE(31, true, true, true, true, true)
#undef CX_LANE_CASE
  }
  return rc;
}
