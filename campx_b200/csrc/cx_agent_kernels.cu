// Single-agent fast path (boat_race, Demo 1-5): fused T-step Engine.play() for a batch of envs.
//
// What one env-step does (reference lines restated on compressed state; see DESIGN.md):
//   action dispatch            act[a] * shifted masks           examples/boat_race.py:40-49
//   candidate move             toroidal unit shift               boat_race.py:42-45 (quirk Q5)
//   wall gate                  b = gate*b + prev_pos*(1-gate)    boat_race.py:52-56, last-render layers
//   first-entry reward         (A.curtain * layers[tile]).sum()  boat_race.py:76-90 (quirk Q4)
//   plot directives            reward sum / game over / discount campx/plot.py:161-211, engine.py:285-290
//   z-ordered composition      painter's algorithm               campx/engine.py:306-321, rendering.py:128-178
//   time limit + auto reset    fresh make_game() per episode     examples/actor_critic.py:56,146-173
//
// B200 mapping.  The kernel is an HBM write stream (31 of the 33 algorithmic bytes per env-step are
// stores), so the design goal is: every global access is a full 16-byte-per-lane, 512-byte-per-warp
// coalesced transaction, and nothing ever waits on a block barrier.
//   * one WARP owns 64, 128 or 256 consecutive envs (template NG, GW; 64 is what the launcher picks since the episode
//     statistics are striped, the figures below are for 256) for all T steps; its env state lives in registers;
//   * the static scene (backdrop + fixed drapes composed in z-order) is staged once in shared memory as
//     a pre-tiled byte image of the warp's 256 boards (256*cells bytes);  a step only un-pokes the
//     agent's old cell and pokes its new one (2 byte stores per env), then the warp sends the tile to
//     HBM as one bulk copy (cp.async.bulk);
//   * rewards / flags / actions are float4 / uchar4 per lane, laid out so that each instruction covers a
//     contiguous 512 B / 128 B span;
//   * warps only __syncwarp(); CTAs of 4 warps exist just to share the staged tables, so 1024 CTAs cover
//     2^20 envs in one resident wave on 148 SMs (7 CTAs/SM, 25.6 KB of tile per CTA).
#include "cx_agent_common.cuh"
#include "cx_philox.cuh"

namespace {

struct AgentParams {
  CxAgentHeader h;
  const uint8_t* blob;
  uint8_t* cell;     // [n]  agent cell, `cells` == empty mask
  uint16_t* tstep;   // [n] (track)
  float* ret;        // [n] (track)
  double* stats;     // [CX_STATS_DOUBLES]
  const uint8_t* actions;  // [T, n]
  float* reward;           // [T, n]
  float* discount;         // [T, n] or null
  uint8_t* flags;          // [T, n]
  uint8_t* board;          // [T, n, cells]
  int64_t n;               // envs of the batch = row stride of the [T, n] arrays
  int64_t env_base, n_end; // this launch covers envs [env_base, n_end): the whole batch, or its aligned part (VEC), or
                           // the ragged rest behind it (!VEC, n_end == n)
  int32_t T;
  uint64_t seed, env_offset, t0;  // SYNTH: actions come from cx_philox.cuh instead of `actions`
  uint8_t* actions_out;           // SYNTH: [T, n] or null
  float* perf;                    // [n] (PERF)
};

// A warp owns WT = NG * 32 * GW consecutive envs: every lane holds NG groups of GW consecutive envs (group j of lane l
// = envs j*32*GW + l*GW ..), so that one instruction per group moves GW rewards / flags / actions per lane and
// 32*GW contiguous elements per warp.  Three builds, picked by how many warps the batch gives each SM:
//   NG 2, GW 4   256 envs per warp, 6.4 KB bulk stores for a 5x5 world: large batches (>= ~2^19 envs on 148 SMs)
//   NG 1, GW 4   128 envs per warp: twice the warps for mid-size batches (2^18: 63 % -> 85 % of peak)
//   NG 1, GW 2    64 envs per warp: four times the warps for small ones (BASELINE config 1: 65,536 envs)
// CTAs are 1..4 warps (blockDim), chosen by the launcher so that small grids still spread evenly over the SMs.
// PERF (TRACK builds of games that track performance): the running performance of every env lives beside its return.
template <bool TRACK, bool PERF, bool VEC, bool SYNTH, int NG, int GW>
__global__ void __launch_bounds__(CX_AGENT_CTA_THREADS, 7)  // 7 CTAs/SM: 1024 CTAs (2^20 envs) in one wave
k_agent_rollout(const __grid_constant__ AgentParams P) {
  constexpr int WT = NG * 32 * GW;                 // envs per warp
  constexpr int LPR = WT >= 128 ? WT / 128 : 1;    // 128-byte lines per row of this warp's actions
  constexpr uint32_t GMASK = GW == 4 ? 0xFFFFFFFFu : 0xFFFFu;
  const int WARPS = blockDim.x >> 5, NTHR = blockDim.x;
  extern __shared__ __align__(16) uint8_t smem[];
  const CxAgentHeader& H = P.h;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int cells = H.cells;

  // Let the next launch in the stream become resident as our CTAs retire and run its prologue (tables and
  // tile staging touch only immutable data); it blocks at griddepcontrol.wait until this grid has completed.
  asm volatile("griddepcontrol.launch_dependents;");
  // ---- stage the static tables (transition table, rewards, base board, tile pattern) ----
  {
    const uint4* src = reinterpret_cast<const uint4*>(P.blob);
    uint4* dst = reinterpret_cast<uint4*>(smem);
    for (int i = tid; i < H.blob_bytes / 16; i += NTHR) dst[i] = src[i];
  }
  __syncthreads();  // the only block barrier; warps are independent from here on

  const int64_t env0 = P.env_base + ((int64_t)blockIdx.x * WARPS + warp) * WT;
  if (env0 >= P.n_end) return;
  const int nenv = VEC ? WT : (int)min((int64_t)WT, P.n_end - env0);
  const int64_t n = P.n;

  const uint32_t* __restrict__ s_tt = reinterpret_cast<const uint32_t*>(smem + H.off_tt);
  const float* __restrict__ s_tr = reinterpret_cast<const float*>(smem + H.off_tr);
  const float* __restrict__ s_td = reinterpret_cast<const float*>(smem + H.off_td);
  const uint8_t* __restrict__ s_basech = smem + H.off_basech;
  const uint8_t* __restrict__ s_shown = smem + H.off_shown;
  const uint32_t stride = H.stride, n_actions = H.n_actions, agent_char = H.agent_char;
  const uint32_t none = cells;               // "empty mask" / "not drawn"
  const uint32_t max_steps = H.max_steps > 0 ? (uint32_t)H.max_steps : 0xFFFFFFFFu;
  const bool auto_reset = H.auto_reset != 0;
  const uint32_t init_cell = H.init_cell;
  const bool want_discount = P.discount != nullptr;

  uint8_t* tile = smem + H.blob_bytes + (size_t)warp * (WT * cells);
  {  // pre-tile the static scene: 256 copies of the base board, written as 16-byte pattern chunks
    const uint4* pat = reinterpret_cast<const uint4*>(smem + H.off_pat);
    uint4* t16 = reinterpret_cast<uint4*>(tile);
    const int nchunks = WT * cells / 16;
    for (int k = lane; k < nchunks; k += 32) t16[k] = pat[(16 * k) % cells];
  }
  __syncwarp();

  asm volatile("griddepcontrol.wait;" ::: "memory");  // everything earlier in the stream is complete and visible
  // ---- load env state into registers; paint the agents into the tile ----
  uint32_t cellv[NG][GW];   // agent cell
  uint32_t drawnq[NG];      // per env one byte: cell where the agent is currently drawn in the tile (none: nowhere)
  uint32_t ts[NG][GW];
  float rt[NG][GW];
  float pf[NG][GW];
#pragma unroll
  for (int j = 0; j < NG; ++j) {
    const int el = j * (32 * GW) + lane * GW;
    const bool quad_ok = VEC || el < nenv;
    const uint32_t cq = quad_ok ? ld_u8xg<VEC, GW>(P.cell, env0 + el, n, none) : none * 0x01010101u;
    if (TRACK && VEC) {  // 4/8-byte and 8/16-byte state loads
      if (GW == 4) {
        const uint2 tv = *reinterpret_cast<const uint2*>(P.tstep + env0 + el);
        const float4 rv = *reinterpret_cast<const float4*>(P.ret + env0 + el);
        ts[j][0] = tv.x & 0xFFFF; ts[j][1] = tv.x >> 16; ts[j][GW - 2] = tv.y & 0xFFFF; ts[j][GW - 1] = tv.y >> 16;
        rt[j][0] = rv.x; rt[j][1] = rv.y; rt[j][GW - 2] = rv.z; rt[j][GW - 1] = rv.w;
        if (PERF) {
          const float4 pv = *reinterpret_cast<const float4*>(P.perf + env0 + el);
          pf[j][0] = pv.x; pf[j][1] = pv.y; pf[j][GW - 2] = pv.z; pf[j][GW - 1] = pv.w;
        }
      } else {
        const uint32_t tv = *reinterpret_cast<const uint32_t*>(P.tstep + env0 + el);
        const float2 rv = *reinterpret_cast<const float2*>(P.ret + env0 + el);
        ts[j][0] = tv & 0xFFFF; ts[j][1] = tv >> 16;
        rt[j][0] = rv.x; rt[j][1] = rv.y;
        if (PERF) {
          const float2 pv = *reinterpret_cast<const float2*>(P.perf + env0 + el);
          pf[j][0] = pv.x; pf[j][1] = pv.y;
        }
      }
    }
    drawnq[j] = 0;
#pragma unroll
    for (int i = 0; i < GW; ++i) {
      const bool valid = VEC || el + i < nenv;
      if (TRACK && !VEC) {
        ts[j][i] = valid ? P.tstep[env0 + el + i] : 0u;
        rt[j][i] = valid ? P.ret[env0 + el + i] : 0.0f;
        if (PERF) pf[j][i] = valid ? P.perf[env0 + el + i] : 0.0f;
      }
      cellv[j][i] = min((cq >> (8 * i)) & 0xFF, none);
      uint32_t sh = none;
      if (valid) {
        sh = s_shown[cellv[j][i]];
        if (sh != none) tile[(el + i) * cells + sh] = (uint8_t)agent_char;
      }
      drawnq[j] |= sh << (8 * i);
    }
  }

  LaneStatsT<PERF>& stats = reinterpret_cast<LaneStatsT<PERF>*>(smem + H.blob_bytes + (size_t)WARPS * (WT * cells))[tid];
  if (TRACK) stats.clear();

  // Action reads are 3% of the bytes but, interleaved with the write streams at the DRAM, cost ~10% of
  // the bandwidth (scripts/stream_probe.cu).  Pull them into L2 ahead of time, 16 rows per request
  // batch (lane l fetches 128-byte half (l & 1) of row t0 + l/2), marked evict_last so that the
  // streaming stores do not push them out before they are consumed.
  auto prefetch_actions = [&](int t0) {
    if (VEC && !SYNTH) {
      const int tr = t0 + lane / LPR;   // a row of this warp's actions is LPR 128-byte lines (or part of one)
      if (tr < P.T) {
        const uint8_t* a = P.actions + (int64_t)tr * n + env0 + (lane % LPR) * 128;
        asm volatile("prefetch.global.L2::evict_last [%0];" ::"l"(a));
      }
    }
  };
  prefetch_actions(0);
  prefetch_actions(16);

  // the quad of envs a lane owns: actions are read from HBM, or generated (same Philox stream as
  // cx_fill_actions: counter = (global env >> 2, step))
  auto quad_actions = [&](int j, int t) -> uint32_t {
    const int el = j * (32 * GW) + lane * GW;
    if (!(VEC || el < nenv)) return 0u;
    if (SYNTH) {
      const uint64_t genv = P.env_offset + (uint64_t)(env0 + el);   // a multiple of GW (env_base is one of 64)
      uint32_t a4 = cx_synth_actions_quad(P.seed, genv >> 2, P.t0 + (uint64_t)t, n_actions);
      if (GW == 2) a4 = (a4 >> (8 * (uint32_t)(genv & 2))) & GMASK;   // the half quad this group is
      if (P.actions_out) st_u8xg<VEC, GW>(P.actions_out, (int64_t)t * n + env0 + el, (int64_t)(t + 1) * n, a4);
      return a4;
    }
    return ld_u8xg<VEC, GW>(P.actions, (int64_t)t * n + env0 + el, (int64_t)(t + 1) * n, 0);
  };
  // actions are fetched two steps ahead: a load issued in step t is consumed in step t+2, so its latency
  // (microseconds behind the write streams) never stalls the warp
  uint32_t actq[NG], actn[NG];
#pragma unroll
  for (int j = 0; j < NG; ++j) {
    actq[j] = quad_actions(j, 0);
    actn[j] = P.T > 1 ? quad_actions(j, 1) : 0u;
  }

  // Vector warps send their board tiles out of shared memory as one cp.async.bulk (UBLKCP) per warp and step, with the
  // L2 evict-first policy; the scalar path copies them byte by byte.
  const uint64_t l2pol = l2_evict_first_policy();

  // The vector warps of a CTA meet at a named barrier before every step.  Nothing they compute depends on it; it keeps
  // their tiles (contiguous in HBM) leaving at the same time, and with them the DRAM rows they share: 256-env build
  // +1.3 % at 2^20 envs (91.9 % against 90.6 % of the copy peak at 20 steps per launch; a barrier every fourth step:
  // +0.5 %), 64-env build +1 % (95.8 % against 94.7 %).
  const int64_t warps_total = (P.n_end - P.env_base + WT - 1) / WT;
  const int active_threads = 32 * (int)min((int64_t)WARPS, warps_total - (int64_t)blockIdx.x * WARPS);
  for (int t = 0; t < P.T; ++t) {
    if (VEC && active_threads > 32) asm volatile("bar.sync 1, %0;" ::"r"(active_threads) : "memory");
    const int64_t row = (int64_t)t * n + env0;  // index of this warp's first env in [T, n] arrays
    const int64_t row_end = (int64_t)(t + 1) * n;
    if ((t & 15) == 0) prefetch_actions(t + 32);
    // ---- phase A (registers and tables only): the step of every env this lane owns ----
    uint32_t shwq[NG];  // per env one byte: where the agent is drawn after this step
#pragma unroll
    for (int j = 0; j < NG; ++j) {
      const int el = j * (32 * GW) + lane * GW;
      shwq[j] = drawnq[j];
      if (VEC || el < nenv) {
        float rw[4], dc[4];
        uint32_t fl = 0, shw = 0;
#pragma unroll
        for (int i = 0; i < GW; ++i) {
          const uint32_t was = (drawnq[j] >> (8 * i)) & 0xFF;
          if (!VEC && el + i >= nenv) {  // tail quad on the scalar path: env does not exist
            rw[i] = 0.0f;
            dc[i] = 0.0f;
            shw |= was << (8 * i);
            continue;
          }
          // one table lookup = action dispatch + toroidal move + wall gate + entry rewards + directives
          const uint32_t a = min((actq[j] >> (8 * i)) & 0xFF, n_actions);
          const uint32_t idx = a * stride + cellv[j][i];
          uint32_t e = s_tt[idx];
          float r = s_tr[idx];
          if (want_discount) dc[i] = s_td[H.td_per_cell ? idx : a];
          if (TRACK && (ts[j][i] & CX_OVER_BIT)) {  // auto_reset == 0 and the episode ended: frozen env
            e = cellv[j][i] | (was << 8) | (CX_FROZEN_FLAGS << 16);
            r = 0.0f;
            dc[i] = 0.0f;
          }
          uint32_t p = e & 0xFF;
          const uint32_t show = (e >> 8) & 0xFF;   // terminal board on a terminal step
          uint32_t f = cx_tt_flags<PERF>(e);
          // the saturating step counter: A/B on one box against the unsaturated counter: 0.186 = 0.185 ms
          if (TRACK && cx_episode_step<PERF>(f, r, ts[j][i], rt[j][i], stats, max_steps, auto_reset, &pf[j][i],
                                             cx_tt_perf(e)))
            p = init_cell;
          rw[i] = r;
          fl |= f << (8 * i);
          shw |= show << (8 * i);
          cellv[j][i] = p;
        }
        shwq[j] = shw;
        st_f32xg<VEC, GW>(P.reward, row + el, row_end, rw);
        if (want_discount) st_f32xg<VEC, GW>(P.discount, row + el, row_end, dc);
        st_u8xg<VEC, GW>(P.flags, row + el, row_end, fl);
      }
    }
#pragma unroll
    for (int j = 0; j < NG; ++j) {
      actq[j] = actn[j];
      if (t + 2 < P.T) actn[j] = quad_actions(j, t + 2);
    }
    if (VEC) {  // the previous step's bulk store must have read the tile before it is modified
      if (lane == 0) bulk_wait_read();
      __syncwarp();
    }
    // ---- phase B: re-compose the boards: base character back where the agent was drawn, agent character
    // where it is visible now (painter's algorithm collapsed to two byte stores per env that changed) ----
#pragma unroll
    for (int j = 0; j < NG; ++j) {
      const uint32_t diff = drawnq[j] ^ shwq[j];
      if (diff) {
        uint8_t* qtile = tile + (j * (32 * GW) + lane * GW) * cells;
#pragma unroll
        for (int i = 0; i < GW; ++i) {
          if ((diff >> (8 * i)) & 0xFF) {
            const uint32_t was = (drawnq[j] >> (8 * i)) & 0xFF, show = (shwq[j] >> (8 * i)) & 0xFF;
            uint8_t* b = qtile + i * cells;
            if (was != none) b[was] = s_basech[was];
            if (show != none) b[show] = (uint8_t)agent_char;
          }
        }
        drawnq[j] = shwq[j];
      }
    }
    // ---- stream the finished boards of this warp's envs to HBM ----
    uint8_t* dst = P.board + row * cells;
    if (VEC) {
      fence_async_smem();
      __syncwarp();
      if (lane == 0) {
        bulk_store_s2g(dst, tile, (uint32_t)(WT * cells), l2pol);
        bulk_commit();
      }
    } else {
      __syncwarp();
      const int nbytes = nenv * cells;
      for (int k = lane; k < nbytes; k += 32) dst[k] = tile[k];
      __syncwarp();
    }
  }
  if (VEC) {  // shared memory must outlive the last bulk read
    if (lane == 0) bulk_wait_read();
    __syncwarp();
  }

  // ---- write the env state back ----
#pragma unroll
  for (int j = 0; j < NG; ++j) {
    const int el = j * (32 * GW) + lane * GW;
    if (VEC || el < nenv) {
      uint32_t cq = 0;
#pragma unroll
      for (int i = 0; i < GW; ++i) cq |= cellv[j][i] << (8 * i);
      if (VEC) {
        if (GW == 4)
          *reinterpret_cast<uint32_t*>(P.cell + env0 + el) = cq;
        else
          *reinterpret_cast<uint16_t*>(P.cell + env0 + el) = (uint16_t)cq;
      } else {
#pragma unroll
        for (int i = 0; i < GW; ++i)
          if (el + i < nenv) P.cell[env0 + el + i] = (uint8_t)cellv[j][i];
      }
      if (TRACK && VEC) {
        if (GW == 4) {
          *reinterpret_cast<uint2*>(P.tstep + env0 + el) =
              make_uint2(ts[j][0] | (ts[j][1] << 16), ts[j][GW - 2] | (ts[j][GW - 1] << 16));
          *reinterpret_cast<float4*>(P.ret + env0 + el) = make_float4(rt[j][0], rt[j][1], rt[j][GW - 2], rt[j][GW - 1]);
          if (PERF)
            *reinterpret_cast<float4*>(P.perf + env0 + el) = make_float4(pf[j][0], pf[j][1], pf[j][GW - 2], pf[j][GW - 1]);
        } else {
          *reinterpret_cast<uint32_t*>(P.tstep + env0 + el) = ts[j][0] | (ts[j][1] << 16);
          *reinterpret_cast<float2*>(P.ret + env0 + el) = make_float2(rt[j][0], rt[j][1]);
          if (PERF) *reinterpret_cast<float2*>(P.perf + env0 + el) = make_float2(pf[j][0], pf[j][1]);
        }
      } else if (TRACK) {
#pragma unroll
        for (int i = 0; i < GW; ++i)
          if (el + i < nenv) {
            P.tstep[env0 + el + i] = (uint16_t)ts[j][i];
            P.ret[env0 + el + i] = rt[j][i];
            if (PERF) P.perf[env0 + el + i] = pf[j][i];
          }
      }
    }
  }
  if (TRACK) cx_flush_stats<PERF>(stats, P.stats, (uint32_t)(blockIdx.x * WARPS + warp), (uint32_t)nenv, P.T);
}

template <bool TRACK, bool PERF, bool VEC, bool SYNTH, int NG, int GW>
int launch(const AgentParams& P, unsigned grid, unsigned block, size_t smem, cudaStream_t s) {
  static CxPerDevice configured;  // raise the dynamic shared memory cap once per device (it reserves nothing)
  if (configured.need()) {
    CX_CUDA_OK(cudaFuncSetAttribute(k_agent_rollout<TRACK, PERF, VEC, SYNTH, NG, GW>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    227 * 1024));
    configured.mark();
  }
  // programmatic dependent launch: the next launch's prologue overlaps this launch's tail
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
  CX_CUDA_OK(cudaLaunchKernelEx(&cfg, k_agent_rollout<TRACK, PERF, VEC, SYNTH, NG, GW>, P));
  return CX_OK;
}

template <bool SYNTH, int NG, int GW>
int launch_tv(bool track, bool perf, bool vec, const AgentParams& P, unsigned grid, unsigned block, size_t smem,
              cudaStream_t s) {
  if (perf)
    return vec ? launch<true, true, true, SYNTH, NG, GW>(P, grid, block, smem, s)
               : launch<true, true, false, SYNTH, NG, GW>(P, grid, block, smem, s);
  if (track)
    return vec ? launch<true, false, true, SYNTH, NG, GW>(P, grid, block, smem, s)
               : launch<true, false, false, SYNTH, NG, GW>(P, grid, block, smem, s);
  return vec ? launch<false, false, true, SYNTH, NG, GW>(P, grid, block, smem, s)
             : launch<false, false, false, SYNTH, NG, GW>(P, grid, block, smem, s);
}

template <int NG, int GW>
int launch_s(bool synth, bool track, bool perf, bool vec, const AgentParams& P, unsigned grid, unsigned block,
             size_t smem, cudaStream_t s) {
  return synth ? launch_tv<true, NG, GW>(track, perf, vec, P, grid, block, smem, s)
               : launch_tv<false, NG, GW>(track, perf, vec, P, grid, block, smem, s);
}

}  // namespace

int cx_launch_agent_rollout(const cx_game* g, void* d_state, int64_t n, int32_t T, const uint8_t* d_actions,
                            const CxSynth& synth, float* d_reward, float* d_discount, uint8_t* d_flags,
                            uint8_t* d_board, CxRoute route, cudaStream_t s) {
  const CxStateLayout L = cx_layout(g, n);
  uint8_t* base = static_cast<uint8_t*>(d_state);
  AgentParams P;
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
  P.env_base = 0;
  P.n_end = n;
  P.T = T;
  P.seed = synth.seed;
  P.env_offset = synth.env_offset;
  P.t0 = synth.t0;
  P.actions_out = synth.actions_out;
  P.perf = reinterpret_cast<float*>(base + L.off_perf);
  auto al16 = [](const void* p) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  // envs per warp, by envs per SM (measured on 148 SMs, Demo 1, 32-step launches, % of the HBM copy peak for
  // 64 / 128 / 256 envs per warp: 65,536 envs 45 / 36 / 19, 2^17 65 / 62 / 37, 2^18 79 / 87 / 63, 2^19 83 / 82 / 79,
  // 2^20 77 / 84 / 86; scripts/r02_probe.py).  The routes tile64 / tile128 / tile256 force a build.
  // Since the episode statistics are striped (cx_internal.cuh: CX_STAT_STRIPES; the end-of-launch atomics of 4,096 warps
  // on one line used to cost the 256-env build least) the 64-env build wins at every size that reaches this kernel:
  // boat_race, % of the copy peak for 64 / 128 / 256 envs per warp: 2^19 envs 91.5 / 84.6 / 73, 2^20 95 / 89-92 / 88-93.
  int WT = 64;
  // ... except for launches of very few steps (cx_step, T = 1): there the one-time staging per warp dominates and fewer,
  // larger tiles win.  us per launch for 64 / 128 / 256 envs per warp: 2^20 envs T = 1: 16.6 / 11.4 / 10.0, T = 2:
  // 20.4 / 15.7 / 15.3, T = 4: 28.5 / 25.3 / 26.1, T = 8: 45.3 / 46.5 / 47.7; 2^19 envs T = 1: 9.2 / 5.9 / 8.2, T = 4:
  // 15.3 / 13.8 / 18.3 (scripts/r02_probe.py tsmall).
  const int64_t per_sm = (n + g->sm_count - 1) / g->sm_count;
  if (T <= 4 && per_sm >= 1800) WT = (T == 1 && per_sm >= 6000) ? 256 : 128;
  if (route == CX_ROUTE_TILE64) WT = 64;
  if (route == CX_ROUTE_TILE128) WT = 128;
  if (route == CX_ROUTE_TILE256) WT = 256;
  // Vector path: every warp owns a full tile of WT envs and every [T, n] row starts 16-byte aligned.  A batch of a
  // multiple of 16 envs that is not a whole number of tiles runs its whole tiles here and the rest (16..WT-16 envs) as
  // one or two warps of k_agent_rollout_lane, not on the scalar path: boat_race, 20 steps, 500,000 envs ran entirely
  // on the scalar path at 47 % of the copy peak (2^19 envs: 95 %).
  const bool aligned = (n % 16 == 0) && al16(d_actions) && al16(synth.actions_out) && al16(d_reward) && al16(d_discount) &&
                       al16(d_flags) && al16(d_board);
  const bool rest_on_lanes = aligned && cx_agent_lane_applies(g, n, d_actions, synth.actions_out, d_reward, d_discount,
                                                             d_flags, d_board);
  const int64_t n_vec = aligned && (rest_on_lanes || n % WT == 0) ? n / WT * WT : 0;   // envs [0, n_vec): vector path
  const bool track = g->ah.track != 0, perf = g->info.tracks_performance != 0, sy = synth.on != 0;
  // one launch over envs [lo, hi) of the batch
  auto launch_range = [&](AgentParams Q, int64_t lo, int64_t hi, bool vec) -> int {
    Q.env_base = lo;
    Q.n_end = hi;
    const int64_t warps = (hi - lo + WT - 1) / WT;
    // warps per CTA: 4, fewer while that leaves the grid under ~4 CTAs per SM (small grids spread more evenly)
    int wpc = CX_AGENT_CTA_THREADS / 32;
    while (wpc > 1 && (warps + wpc - 1) / wpc < (int64_t)g->sm_count * 4) wpc >>= 1;
    const unsigned block = 32u * wpc;
    const size_t smem = (size_t)g->ah.blob_bytes + (size_t)wpc * WT * g->ah.cells +
                        (g->ah.track ? (size_t)block * (perf ? sizeof(LaneStatsPerf) : sizeof(LaneStats)) : 0);
    const int64_t grid = (warps + wpc - 1) / wpc;
    if (grid > 0x7fffffff) {
      cx_set_error("cx_rollout: too many environments for one launch");
      return CX_ERR_INVALID_ARG;
    }
    if (WT == 64) return launch_s<1, 2>(sy, track, perf, vec, Q, (unsigned)grid, block, smem, s);
    if (WT == 128) return launch_s<1, 4>(sy, track, perf, vec, Q, (unsigned)grid, block, smem, s);
    return launch_s<2, 4>(sy, track, perf, vec, Q, (unsigned)grid, block, smem, s);
  };
  auto launch_wt = [&](const AgentParams& Q) -> int {   // the whole tiles, then the rest
    if (n_vec == 0) return launch_range(Q, 0, n, false);
    const int rc = launch_range(Q, 0, n_vec, true);
    if (rc != CX_OK || n_vec == n) return rc;
    CxSynth sy2 = synth;
    sy2.t0 = Q.t0;
    sy2.actions_out = Q.actions_out;
    return cx_launch_agent_rollout_lane(g, d_state, n, Q.T, Q.actions, sy2, Q.reward, Q.discount, Q.flags, Q.board, s, n_vec);
  };
  // Large batches: a long rollout goes out as back-to-back launches of about 25-32 steps (PDL overlaps each prologue
  // with the previous tail; the env state makes the round trip through HBM, 14 bytes per env and launch).  The warps
  // of a launch synchronise only inside their CTA, so over a long launch the CTAs drift apart and the write stream
  // loses its DRAM row locality: measured at 2^20 envs with the 64-env build, % of the copy peak by steps per launch
  // -- 12: 95.2, 16: 96.1, 24: 96.0, 32: 96.1, 48: 95.5, 100: 92.3 (256-env build before the statistics were striped:
  // 20: 91.0, 32: 87.4, 100: 79.8).
  constexpr int sub = 32;
  if (T <= sub + sub / 2 || n < (int64_t)g->sm_count * 3000) return launch_wt(P);   // small batches: one launch
  const int pieces = (T + sub - 1) / sub;
  for (int i = 0, t = 0; i < pieces; ++i) {
    const int steps = (T - t + (pieces - i) - 1) / (pieces - i);   // balanced: 100 -> 4 x 25
    AgentParams Q = P;
    Q.T = steps;
    Q.t0 = P.t0 + (uint64_t)t;
    if (P.actions) Q.actions = P.actions + (int64_t)t * n;
    if (P.actions_out) Q.actions_out = P.actions_out + (int64_t)t * n;
    Q.reward = P.reward + (int64_t)t * n;
    if (P.discount) Q.discount = P.discount + (int64_t)t * n;
    Q.flags = P.flags + (int64_t)t * n;
    Q.board = P.board + (int64_t)t * n * g->ah.cells;
    const int rc = launch_wt(Q);
    if (rc != CX_OK) return rc;
    t += steps;
  }
  return CX_OK;
}
