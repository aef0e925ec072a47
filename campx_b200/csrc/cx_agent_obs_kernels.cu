// Single-agent fast path with the FULL observation: fused T-step Engine.play() that writes, per env-step,
// the board AND the layered board (campx/rendering.py:181-219: layers[ch] = board == ord(ch), stacked in
// canonical channel order) -- the tensor the reference's RL loops feed to the policy
// (examples/actor_critic.py:147,173: state = board.layered_board.view(-1).float()).
//
// Why a second kernel: deriving the layers from a finished board (cx_layers_from_board) re-reads the board
// from HBM and costs a second launch; here they leave the SM together.  Algorithmic bytes per env-step
// (boat_race): action 1 + reward 4 + flags 1 + board 25 + layered 7*25 = 206 B.
//
// B200 mapping.  The layered board of a single-agent game is, like its board, a static image plus the
// agent: moving the agent from cell `was` to cell `show` changes four bytes
//     layer[agent][was] = 0, layer[base(was)][was] = 1, layer[base(show)][show] = 0, layer[agent][show] = 1
// so one WARP keeps the boards (32 x cells bytes) and layered boards (32 x chars x cells bytes) of 32
// consecutive envs in shared memory for all T steps, lane = env, pokes 2 + 4 bytes per env-step and hands
// both tiles to the TMA engine: two cp.async.bulk (UBLKCP) stores per warp and step, 800 B + 5600 B for
// boat_race, contiguous in HBM because the outputs are env-major.  Rewards / flags / actions are one
// 128 B / 32 B / 32 B transaction per warp.  The step itself is the same (action, cell) table lookup as
// k_agent_rollout (cx_agent_kernels.cu), so the two kernels cannot disagree on the game rules.
//
// The same kernel, with the layered board switched off, is the step kernel of single-agent games whose boards
// are too large for k_agent_rollout's 256-env warp tiles (97..254 cells): at >= 100 bytes per env-step a
// lane-per-env warp saturates HBM as well.  It also takes ragged batches (N not a multiple of 32) and
// unaligned buffers (coalesced byte stores instead of the bulk stores) and in-kernel Philox actions.
//
// Games with collectible items (CX_KIND_PICKUP) run only here, in the PICK build: each lane keeps its env's u64 of
// remaining items (CxPickHeader) and every ring slot remembers which items it shows; an item whose bit differs is
// poked between its present and absent bytes (board and layered tile) when the slot comes up.  Key-locked doors
// (CX_KIND_DOOR) are a function of the items: a step looks its (action, cell) up in the table of the doors its start
// shows, and the cells of the doors a frame shows closed are bits of the same shown word as the items.
#include "cx_agent_common.cuh"
#include "cx_philox.cuh"

namespace {

struct ObsParams {
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
  uint8_t* layered;        // [T, n, chars, cells] or null
  int64_t n;
  int32_t T;
  int32_t bulk;            // every [T, n, ...] row of board / layered starts 16-byte aligned: TMA bulk stores
  int32_t synth;           // actions from cx_philox.cuh instead of `actions`
  uint64_t seed, env_offset, t0;
  uint8_t* actions_out;    // synth: [T, n] or null
  float* perf;             // [n] (PERF)
  uint64_t* pick;          // [n] items each env still holds (PICK)
  CxPickHeader pk;         // (PICK)
};

constexpr int OBS_WARPS = 4;
constexpr int OBS_THREADS = OBS_WARPS * 32;
constexpr int OBS_TILE = 32;  // envs per warp: lane = env

// RING: tiles per warp, 1 or 2.  A warp may not touch a tile again before the bulk store that shipped it has READ it; with one
// tile that wait (TMA issue -> shared-memory read, ~1 us) sits on every step's critical path, which is what bounds
// small batches (65,536 envs = 14 warps per SM: there is nothing else to run meanwhile).  With RING tiles used round
// robin the warp waits for the store issued RING steps ago (`cp.async.bulk.wait_group.read RING-1`), i.e. almost
// never, and a step's chain is table lookup -> 2 byte pokes -> fence -> issue.  PERF (TRACK builds of games that
// track performance): the running performance beside the return.  PICK: games with pickups (see the top of the file).
template <bool TRACK, bool PERF, int RING, bool PICK>
__global__ void __launch_bounds__(OBS_THREADS) k_agent_rollout_obs(const __grid_constant__ ObsParams P) {
  extern __shared__ __align__(16) uint8_t smem[];
  const CxAgentHeader& H = P.h;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int cells = H.cells, lay_bytes = H.n_chars * H.cells;

  asm volatile("griddepcontrol.launch_dependents;");
  {
    const uint4* src = reinterpret_cast<const uint4*>(P.blob);
    uint4* dst = reinterpret_cast<uint4*>(smem);
    for (int i = tid; i < H.blob_bytes_ext / 16; i += OBS_THREADS) dst[i] = src[i];
    if constexpr (PICK) {  // the item tables go right behind the extension
      const uint4* psrc = reinterpret_cast<const uint4*>(P.blob + P.pk.off);
      uint4* pdst = reinterpret_cast<uint4*>(smem + H.blob_bytes_ext);
      for (int i = tid; i < P.pk.bytes / 16; i += OBS_THREADS) pdst[i] = psrc[i];
    }
  }
  __syncthreads();  // the only block barrier

  const int64_t env0 = ((int64_t)blockIdx.x * OBS_WARPS + warp) * OBS_TILE;
  if (env0 >= P.n) return;
  const int64_t n = P.n, env = env0 + lane;
  const int nenv = (int)min((int64_t)OBS_TILE, n - env0);
  const bool mine = lane < nenv;
  const bool layers = P.layered != nullptr;

  const uint32_t* __restrict__ s_tt = reinterpret_cast<const uint32_t*>(smem + H.off_tt);
  const float* __restrict__ s_tr = reinterpret_cast<const float*>(smem + H.off_tr);
  const float* __restrict__ s_td = reinterpret_cast<const float*>(smem + H.off_td);
  const uint8_t* __restrict__ s_basech = smem + H.off_basech;
  const uint8_t* __restrict__ s_shown = smem + H.off_shown;
  const uint8_t* __restrict__ s_basek = smem + H.off_basek;
  const uint8_t* __restrict__ s_baselay = smem + H.off_baselay;
  const uint32_t stride = H.stride, n_actions = H.n_actions, agent_char = H.agent_char, agent_k = H.agent_k;
  const uint32_t none = cells;
  const uint32_t max_steps = H.max_steps > 0 ? (uint32_t)H.max_steps : 0xFFFFFFFFu;
  const bool auto_reset = H.auto_reset != 0, want_discount = P.discount != nullptr;

  // per warp: RING x { [board tile 32*cells][layered tile 32*chars*cells (if wanted)] }, all multiples of 16 bytes
  const int per_env = cells + (layers ? lay_bytes : 0);
  const int slot_bytes = OBS_TILE * per_env;
  const int tiles_at = H.blob_bytes_ext + (PICK ? P.pk.bytes : 0);
  uint8_t* wbase = smem + tiles_at + (size_t)warp * RING * slot_bytes;
  for (int r = 0; r < RING; ++r) {                              // every lane stages its own env's static scene
    uint8_t* myb = wbase + r * slot_bytes + lane * cells;
    uint8_t* myl = wbase + r * slot_bytes + OBS_TILE * cells + lane * lay_bytes;
    for (int c = 0; c < cells; ++c) myb[c] = s_basech[c];
    if (layers)
      for (int j = 0; j < lay_bytes; ++j) myl[j] = s_baselay[j];
  }
  __syncwarp();

  asm volatile("griddepcontrol.wait;" ::: "memory");
  // Occluded layers (the reference's default, rendering.py:204-209) follow the BOARD: the agent's plane is set where
  // it is drawn and the plane of the character it covers is cleared there.  Unoccluded layers
  // (cx_game_desc::unoccluded_layers, rendering.py:227-353) follow the CURTAINS: only the agent's own plane changes,
  // at the agent's real cell, drawn or not; the static planes (backdrop cells, whole static curtains) never do.
  const bool unocc = H.unoccluded != 0;
  auto draw = [&](int r, uint32_t c) {  // paint the agent at visible cell c of ring slot r
    uint8_t* myb = wbase + r * slot_bytes + lane * cells;
    myb[c] = (uint8_t)agent_char;
    if (layers && !unocc) {
      uint8_t* myl = wbase + r * slot_bytes + OBS_TILE * cells + lane * lay_bytes;
      const uint32_t k = s_basek[c];
      if (k != 0xFF) myl[k * cells + c] = 0;
      myl[agent_k * cells + c] = 1;
    }
  };
  auto erase = [&](int r, uint32_t c) {  // back to the static scene at cell c
    uint8_t* myb = wbase + r * slot_bytes + lane * cells;
    myb[c] = s_basech[c];
    if (layers && !unocc) {
      uint8_t* myl = wbase + r * slot_bytes + OBS_TILE * cells + lane * lay_bytes;
      myl[agent_k * cells + c] = 0;
      const uint32_t k = s_basek[c];
      if (k != 0xFF) myl[k * cells + c] = 1;
    }
  };
  auto agent_plane = [&](int r, uint32_t c, uint8_t v) {  // unoccluded: the agent's curtain is its one cell
    (wbase + r * slot_bytes + OBS_TILE * cells + lane * lay_bytes)[agent_k * cells + c] = v;
  };

  // PICK: the static scene (basech / basek / baselay) shows every item and every door closed; slot r shows the items
  // and closed door cells in shown_items[r] (CxPickHeader).
  const uint8_t* __restrict__ s_item_at = smem + H.blob_bytes_ext + P.pk.item_at;
  const uint64_t* __restrict__ s_drape_cells =
      reinterpret_cast<const uint64_t*>(smem + H.blob_bytes_ext + P.pk.drape_cells);
  const CxPickItem* __restrict__ s_items = reinterpret_cast<const CxPickItem*>(smem + H.blob_bytes_ext + P.pk.items);
  const CxPickDrape* __restrict__ s_drapes =
      reinterpret_cast<const CxPickDrape*>(smem + H.blob_bytes_ext + P.pk.drapes);
  uint64_t items = 0, shown_items[RING];
  if constexpr (PICK) items = mine ? P.pick[env] : P.pk.all;
  // PICK: the doors of `items` -- the open ones, the shown-word bits of the closed door cells, and the offsets of the
  // open doors' step tables from the agent header's.  They change only when a key drape gives up its last item (it
  // opens its doors) and at an auto reset (every door closes), so a step that takes nothing does no door work.
  uint32_t open = 0, tt_off = 0, tr_off = 0, td_off = 0;
  uint64_t closed = 0;
  auto door_tables = [&]() {
    tt_off = open ? P.pk.tt_first + (open - 1) * P.pk.tt_size : 0;
    tr_off = open ? P.pk.tr_first + (open - 1) * P.pk.tt_size : 0;
    td_off = open ? P.pk.td_first + (open - 1) * P.pk.td_size : 0;
  };
  if constexpr (PICK) {
    open = cx_doors(P.pk, items, &closed);
    door_tables();
  }
  auto poke_item = [&](int r, uint32_t i, bool present) {  // item i of ring slot r (the agent is not drawn on it)
    const CxPickItem it = s_items[i];
    const uint32_t c = it.cell, kp = s_basek[c];
    (wbase + r * slot_bytes + lane * cells)[c] = present ? s_basech[c] : it.under_ch;
    if (layers) {
      uint8_t* myl = wbase + r * slot_bytes + OBS_TILE * cells + lane * lay_bytes;
      const uint32_t k_off = present ? it.under_k : kp, k_on = present ? kp : it.under_k;
      if (k_off != 0xFF) myl[k_off * cells + c] = 0;
      if (k_on != 0xFF) myl[k_on * cells + c] = 1;
    }
  };
  auto sync_items = [&](int r, uint64_t want) {  // bring slot r to the items `want`
    for (uint64_t m = shown_items[r] ^ want; m; m &= m - 1) {
      const uint32_t i = __ffsll((long long)m) - 1;
      poke_item(r, i, (want >> i) & 1);
    }
    shown_items[r] = want;
  };
  auto draw_agent = [&](int r, uint32_t c) {  // draw over the items slot r shows (a taken one left its under_k set)
    draw(r, c);
    if constexpr (PICK) {
      const uint32_t i = s_item_at[c];
      if (layers && i != CX_NO_ITEM && !((shown_items[r] >> i) & 1)) {
        const uint32_t k = s_items[i].under_k;
        if (k != 0xFF) (wbase + r * slot_bytes + OBS_TILE * cells + lane * lay_bytes)[k * cells + c] = 0;
      }
    }
  };
  auto erase_agent = [&](int r, uint32_t c) {  // erase, with the items slot r shows
    erase(r, c);
    if constexpr (PICK) {
      const uint32_t i = s_item_at[c];
      if (i != CX_NO_ITEM && !((shown_items[r] >> i) & 1)) poke_item(r, i, false);
    }
  };

  uint32_t cell = mine ? min((uint32_t)P.cell[env], none) : none;
  uint32_t shown = s_shown[cell];   // where the agent is drawn in the most recent frame
  uint32_t drawn[RING];             // ... and in each ring slot (a slot is RING frames behind when it comes up again)
  uint32_t lcell[RING];             // unoccluded layers: the cell set in the agent's plane of each ring slot
#pragma unroll
  for (int r = 0; r < RING; ++r) {
    drawn[r] = shown;
    lcell[r] = none;
    if constexpr (PICK) {  // the items this env has already taken, and the doors that opened, leave every slot
      shown_items[r] = P.pk.scene_all;
      sync_items(r, items | closed);
    }
    if (shown != none) draw_agent(r, shown);
    if (layers && unocc && cell != none) {
      agent_plane(r, cell, 1);
      lcell[r] = cell;
    }
  }
  uint32_t ts = 0;
  float rt = 0.0f, pf = 0.0f;
  if (TRACK && mine) {
    ts = P.tstep[env];
    rt = P.ret[env];
    if (PERF) pf = P.perf[env];
  }
  LaneStatsT<PERF>& stats =
      reinterpret_cast<LaneStatsT<PERF>*>(smem + tiles_at + (size_t)OBS_WARPS * RING * slot_bytes)[tid];
  if (TRACK) stats.clear();

  // whole tiles over TMA when the rows are 16-byte aligned and the warp owns 32 envs; else byte stores
  const bool bulk = P.bulk && nenv == OBS_TILE;
  auto fetch_action = [&](int t) -> uint32_t {
    if (!mine || t >= P.T) return 0u;
    if (P.synth) {
      const uint32_t a = cx_synth_action(P.seed, P.env_offset + (uint64_t)env, P.t0 + (uint64_t)t, n_actions);
      if (P.actions_out) P.actions_out[(int64_t)t * n + env] = (uint8_t)a;
      return a;
    }
    return P.actions[(int64_t)t * n + env];
  };
  const uint64_t l2pol = l2_evict_first_policy();
  // the loop is unrolled by UNR steps so that ring slots and the action registers are indexed statically; actions
  // are fetched one whole group (UNR steps) ahead of their use
  constexpr int UNR = 4;
  static_assert(UNR % RING == 0, "ring slots are indexed by the unrolled step");
  uint32_t act[UNR], act_next[UNR];
#pragma unroll
  for (int u = 0; u < UNR; ++u) act[u] = fetch_action(u);

  for (int t0 = 0; t0 < P.T; t0 += UNR) {
#pragma unroll
    for (int u = 0; u < UNR; ++u) act_next[u] = fetch_action(t0 + UNR + u);
#pragma unroll
    for (int u = 0; u < UNR; ++u) {
      const int t = t0 + u;
      if (t >= P.T) break;
      const int r = u % RING;
      const int64_t row = (int64_t)t * n + env0;
      // ---- phase A: the env's step (same table as k_agent_rollout) ----
      const uint32_t a = min(act[u], n_actions);
      const uint32_t idx = a * stride + cell;
      uint32_t e;
      float rw, dc;
      if constexpr (PICK) {  // the doors this step's last render shows open select their own tables
        e = s_tt[idx + tt_off];
        rw = s_tr[idx + tr_off];
        dc = want_discount ? s_td[(H.td_per_cell ? idx : a) + td_off] : 1.0f;
      } else {
        e = s_tt[idx];
        rw = s_tr[idx];
        dc = want_discount ? s_td[H.td_per_cell ? idx : a] : 1.0f;
      }
      if (TRACK && (ts & CX_OVER_BIT)) {
        e = cell | (shown << 8) | (CX_FROZEN_FLAGS << 16);
        rw = 0.0f;
        dc = 0.0f;
      }
      uint32_t p = e & 0xFF;
      const uint32_t show = mine ? (e >> 8) & 0xFF : none;
      const uint32_t stood = mine ? p : none;   // the agent's cell in this step's frame (before any auto reset)
      uint32_t f = cx_tt_flags<PERF>(e);
      uint64_t frame_items = 0;   // PICK: the shown word of this step's frame (before an auto reset)
      if constexpr (PICK) {
        // one look-up at the watched cell: the agent's cell after the move when the pickups update after it, before
        // the move otherwise (the entry-reward query); a bad action or a frozen env takes nothing
        const uint32_t i = s_item_at[P.pk.after ? p : cell];
        if (mine && i != CX_NO_ITEM && ((items >> i) & 1) && !(f & (CX_FLAG_BAD_ACTION | CX_FLAG_ALREADY_OVER))) {
          items &= ~(1ull << i);
          const CxPickDrape& D = s_drapes[s_items[i].drape];
          rw += D.reward[a];      // the table's sum of the entities before it, or 0 (REWARD_NONE)
          f &= ~(uint32_t)CX_FLAG_REWARD_NONE;
          if (D.terminates && !(items & D.items)) {
            f |= CX_FLAG_TERMINATED;
            dc = D.emptied_value;
          }
          if (D.opens && !(items & D.items)) {   // a key drape's last item: its doors open (cx_doors)
            open |= D.opens;
            closed &= ~s_drape_cells[s_items[i].drape];
            door_tables();
          }
        }
        frame_items = items | closed;
      }
      if (TRACK && mine && cx_episode_step<PERF>(f, rw, ts, rt, stats, max_steps, auto_reset, &pf, cx_tt_perf(e))) {
        p = H.init_cell;
        if constexpr (PICK) {   // an auto reset puts every item back, and closes every door
          items = P.pk.all;
          if (open) {
            open = 0;
            closed = P.pk.scene_all & ~P.pk.all;
            door_tables();
          }
        }
      }
      if (mine) {
        cell = p;
        __stcs(P.reward + row + lane, rw);
        if (want_discount) __stcs(P.discount + row + lane, dc);
        P.flags[row + lane] = (uint8_t)f;
      }
      shown = show;

      // ---- phase B: bring ring slot r up to date (2 + 4 byte stores when the agent moved) and send it out ----
      if (bulk) {
        if (lane == 0) bulk_wait_read_pending<RING - 1>();  // the store that last shipped slot r has read it
        __syncwarp();
      }
      if constexpr (PICK) {
        if (shown_items[r] != frame_items) {   // the agent comes off first: pokes assume it is not drawn there
          if (drawn[r] != none) erase_agent(r, drawn[r]);
          drawn[r] = none;
          sync_items(r, frame_items);
        }
        if (drawn[r] != show) {
          if (drawn[r] != none) erase_agent(r, drawn[r]);
          if (show != none) draw_agent(r, show);
          drawn[r] = show;
        }
      } else if (drawn[r] != show) {
        if (drawn[r] != none) erase(r, drawn[r]);
        if (show != none) draw(r, show);
        drawn[r] = show;
      }
      if (layers && unocc && lcell[r] != stood) {
        if (lcell[r] != none) agent_plane(r, lcell[r], 0);
        if (stood != none) agent_plane(r, stood, 1);
        lcell[r] = stood;
      }
      const uint8_t* btile = wbase + r * slot_bytes;
      const uint8_t* ltile = btile + OBS_TILE * cells;
      uint8_t* bdst = P.board + row * cells;
      if (bulk) {
        fence_async_smem();
        __syncwarp();
        if (lane == 0) {
          bulk_store_s2g(bdst, btile, (uint32_t)(OBS_TILE * cells), l2pol);
          if (layers) bulk_store_s2g(P.layered + row * lay_bytes, ltile, (uint32_t)(OBS_TILE * lay_bytes), l2pol);
          bulk_commit();
        }
      } else {
        __syncwarp();
        for (int k = lane; k < nenv * cells; k += 32) bdst[k] = btile[k];
        if (layers) {
          uint8_t* ldst = P.layered + row * lay_bytes;
          for (int k = lane; k < nenv * lay_bytes; k += 32) ldst[k] = ltile[k];
        }
        __syncwarp();
      }
    }
#pragma unroll
    for (int u = 0; u < UNR; ++u) act[u] = act_next[u];
  }
  if (lane == 0) bulk_wait_read();
  __syncwarp();
  if (mine) {
    P.cell[env] = (uint8_t)cell;
    if (TRACK) {
      P.tstep[env] = (uint16_t)ts;
      P.ret[env] = rt;
      if (PERF) P.perf[env] = pf;
    }
    if constexpr (PICK) P.pick[env] = items;
  }
  if (TRACK)  // all 32 lanes reduce (lanes without an env contribute empty statistics)
    cx_flush_stats<PERF>(stats, P.stats, (uint32_t)(blockIdx.x * OBS_WARPS + warp), (uint32_t)nenv, P.T);
}

size_t obs_smem_bytes(const cx_game* g, bool layers, int ring = 1) {
  const size_t per_env = (size_t)g->ah.cells * (1 + (layers ? g->ah.n_chars : 0));
  return (size_t)g->ah.blob_bytes_ext + (size_t)g->ph.bytes + (size_t)OBS_WARPS * OBS_TILE * per_env * ring +
         (g->ah.track ? OBS_THREADS * (g->info.tracks_performance ? sizeof(LaneStatsPerf) : sizeof(LaneStats)) : 0);
}

template <bool TRACK, bool PERF, int RING, bool PICK>
int launch_obs(const ObsParams& P, unsigned grid, size_t smem, cudaStream_t s) {
  static CxPerDevice configured;  // the dynamic shared memory cap is a per-device function attribute
  if (configured.need()) {
    CX_CUDA_OK(cudaFuncSetAttribute(k_agent_rollout_obs<TRACK, PERF, RING, PICK>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    227 * 1024));
    configured.mark();
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(OBS_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  CX_CUDA_OK(cudaLaunchKernelEx(&cfg, k_agent_rollout_obs<TRACK, PERF, RING, PICK>, P));
  return CX_OK;
}

template <bool TRACK, bool PERF, bool PICK = false>
int launch_obs_ring(int ring, const ObsParams& P, unsigned grid, size_t smem, cudaStream_t s) {
  return ring >= 2 ? launch_obs<TRACK, PERF, 2, PICK>(P, grid, smem, s) : launch_obs<TRACK, PERF, 1, PICK>(P, grid, smem, s);
}

}  // namespace

// Shared memory decides whether the lane-per-env kernel can hold a CTA's tiles (boards up to 254 cells always
// fit without the layered tile; with it, up to about 1500 bytes of layered board per env).
bool cx_agent_obs_applies(const cx_game* g, bool layers) {
  return g->path == CX_PATH_AGENT && obs_smem_bytes(g, layers) <= 200 * 1024;
}

size_t cx_agent_obs_smem_bytes(const cx_game* g) { return obs_smem_bytes(g, false); }

int cx_launch_agent_rollout_obs(const cx_game* g, void* d_state, int64_t n, int32_t T, const uint8_t* d_actions,
                                const CxSynth& synth, float* d_reward, float* d_discount, uint8_t* d_flags,
                                uint8_t* d_board, uint8_t* d_layered, cudaStream_t s) {
  const CxStateLayout L = cx_layout(g, n);
  uint8_t* base = static_cast<uint8_t*>(d_state);
  ObsParams P;
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
  P.T = T;
  P.synth = synth.on;
  P.seed = synth.seed;
  P.env_offset = synth.env_offset;
  P.t0 = synth.t0;
  P.actions_out = synth.actions_out;
  P.perf = reinterpret_cast<float*>(base + L.off_perf);
  P.pick = reinterpret_cast<uint64_t*>(base + L.off_pick);
  P.pk = g->ph;
  // bulk (TMA) stores: every [T, n, ...] row and every warp tile must start 16-byte aligned
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  const int64_t lay_bytes = (int64_t)g->ah.n_chars * g->ah.cells;
  P.bulk = al16(d_board) && (n * g->ah.cells) % 16 == 0 &&
           (!d_layered || (al16(d_layered) && (n * lay_bytes) % 16 == 0));
  const int64_t warps = (n + OBS_TILE - 1) / OBS_TILE;
  const int64_t grid = (warps + OBS_WARPS - 1) / OBS_WARPS;
  if (grid > 0x7fffffff) {
    cx_set_error("cx_rollout: too many environments for one launch");
    return CX_ERR_INVALID_ARG;
  }
  // ring depth: two tiles per warp for small batches (measured on 148 SMs: board-only 65,536 envs 33 % -> 39 % of
  // peak, layered 4,096 envs 14.5 % -> 17.7 %; four tiles never beat two), one tile from 65,536 envs up, where the
  // other resident warps hide the wait and the extra staging only costs (2^18 envs: 62 % -> 58 %)
  const bool lay = d_layered != nullptr;
  int ring = 1;
  if (P.bulk && T > 1 && n < 65536 && obs_smem_bytes(g, lay, 2) <= (size_t)(lay ? 56 : 32) * 1024) ring = 2;
  const size_t smem = obs_smem_bytes(g, lay, ring);
  if (smem > 227 * 1024) {
    cx_set_error("cx_rollout: board too large for the lane-per-env kernel with %d tiles per warp", ring);
    return CX_ERR_INVALID_ARG;
  }
  if (g->info.tracks_performance) return launch_obs_ring<true, true>(ring, P, (unsigned)grid, smem, s);
  if (g->info.n_pickups)   // (never together with performance: cx_game_create refuses that)
    return g->ah.track ? launch_obs_ring<true, false, true>(ring, P, (unsigned)grid, smem, s)
                       : launch_obs_ring<false, false, true>(ring, P, (unsigned)grid, smem, s);
  return g->ah.track ? launch_obs_ring<true, false>(ring, P, (unsigned)grid, smem, s)
                     : launch_obs_ring<false, false>(ring, P, (unsigned)grid, smem, s);
}
