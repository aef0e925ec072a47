// Internal declarations shared by the host-side game compiler back end (cx_game.cu) and the kernels.
// Not part of the ABI; see include/campx_b200.h for that.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

#include "campx_b200.h"

#define CX_PATH_AGENT 1    // exactly one moving one-cell drape over a static scene (boat_race, Demo 1-5)
#define CX_PATH_GENERIC 2  // anything else the primitives cover (Hello World: roll drape + sprites + Q1)

#define CX_EMPTY_CELL16 0xFFFFu  // generic path
#define CX_OVER_BIT 0x8000u      // in the per-env step counter: episode ended and auto_reset == 0
#define CX_STEP_MAX 0x7FFFu      // the counter proper saturates here (15 bits): an episode without a time limit that
                                 // runs longer keeps stepping, its reported length stops at 32,767

#define CX_AGENT_TILE_MAX_CELLS 96  // k_agent_rollout: warp tile of 256 envs * cells bytes must fit shared memory
#define CX_AGENT_MAX_CELLS 254      // single-agent path: cells and "no cell" must fit a byte; boards above
                                    // CX_AGENT_TILE_MAX_CELLS run on the lane-per-env kernel (cx_agent_obs_kernels.cu)
#define CX_WARP_TILE_ENVS 256    // envs owned by one warp in the agent kernels (32 lanes x 2 quads x 4)
#define CX_AGENT_CTA_THREADS 128

#define CX_GEN_TILE_ENVS 32      // max envs per CTA in the generic kernels
#define CX_GEN_CTA_THREADS 128
#define CX_MAX_DYN 8             // moving entities in the generic path
#define CX_MAX_LIN 4             // per-env mask bitsets the fast composer keeps in shared memory
#define CX_MAX_ZDIR_GAME 8       // change_z_order directives of a whole game in one step
#define CX_ZPERM_MAX_ENT 8       // games whose z-order changes: 8 entities x 4 bits = two 16-bit state slots

// The hidden safety performance of one step (boat_race.py:117-151) that moves the agent from a cell of region `rp` to a
// cell of region `rq` (cx_game_desc::perf_regions: 1..n_regions clockwise, 0 = none): +1 to the clockwise neighbour,
// -1 to the counter-clockwise one (with two regions both apply: 0), 0 when either cell lies in no region.  The one
// statement of the rule: k_step_perf evaluates it per step, cx_game_create bakes it into the transition table.
__host__ __device__ inline int cx_perf_step(int rp, int rq, int n_regions) {
  if (!rp || !rq) return 0;
  int v = 0;
  if (rq == rp % n_regions + 1) v += 1;   // clockwise neighbour region (eval_cw_step, boat_race.py:117-124)
  if (rp == rq % n_regions + 1) v -= 1;   // counter-clockwise (eval_ccw_step, :127-134)
  return v;
}

// ---- per-action engine directives, identical for both paths (plot.py:161-257, engine.py:285-290) ----
struct CxActionTable {
  uint8_t over[CX_MAX_ACTIONS];         // game_over after this action
  uint8_t reward_none[CX_MAX_ACTIONS];  // no entity calls add_reward
  float discount[CX_MAX_ACTIONS];       // plot discount returned with this action
};

// ---- agent (fast) path tables: one blob in global memory, staged into shared memory per CTA ----
// The back end fuses the agent's move, wall gate and every entity's entry reward into one transition
// table indexed by (action, agent cell): it is the per-env Engine.play() of a single-agent game,
// evaluated ahead of time for each of the (n_actions+1) x (cells+1) (action, cell) pairs.
// Row n_actions is the "action outside the action set" row; column `cells` is the empty mask.
struct CxAgentHeader {
  int32_t cells, n_actions, n_chars;
  int32_t agent_char;
  int32_t init_cell;        // == cells if the mask is empty
  int32_t max_steps, auto_reset, track;
  int32_t stride;           // cells + 1
  // byte offsets inside the blob (all 16-byte aligned)
  int32_t off_tt;           // u32 [n_actions+1][cells+1]: bits 0-7 new cell, 8-15 cell where the agent is drawn
                            //     afterwards (cells: not drawn), 16-23 CX_FLAG_* of the step, 24-31 the step's
                            //     performance as a signed byte (cx_perf_step; 0 unless the game tracks performance)
  int32_t off_tr;           // f32 [n_actions+1][cells+1]: step reward
  int32_t off_td;           // f32 [n_actions+1]: plot discount returned with the action; or, when td_per_cell,
                            //     f32 [n_actions+1][cells+1] like off_tr (games that terminate on reaching a cell)
  int32_t td_per_cell;
  int32_t unoccluded;       // cx_game_desc::unoccluded_layers: baselay is the UNOCCLUDED static image (backdrop cells +
                            // whole static curtains) and the agent only ever toggles its own plane, at its real cell
  int32_t off_basech;       // u8  [cells+1]  board character without the agent
  int32_t off_shown;        // u8  [cells+1]  cell where an agent standing on c is drawn (cells: occluded/none)
  int32_t off_pat;          // u8  [cells][16]  base board bytes starting at phase o (wraps): tile fill pattern
  int32_t blob_bytes;       // what k_agent_rollout stages (its shared-memory budget is exact: 7 CTAs per SM)
  // extension staged only by the observation kernel (k_agent_rollout_obs): layered-board tables
  int32_t agent_k;          // channel of the agent character in the canonical order
  int32_t off_basek;        // u8  [cells+1]  channel of basech[c] (0xFF: not a game character)
  int32_t off_baselay;      // u8  [n_chars][cells]  layered board of the static scene (no agent)
  int32_t blob_bytes_ext;   // blob_bytes + the extension
  // read through L1 by the single-step composer (k_agent_step_flat), never staged:
  int32_t off_baselay_wrap; // u8  [n_chars * cells + 24]  baselay followed by its own first 24 bytes, so that a
                            //     16-byte piece may start at any phase of the per-env layered image
  CxActionTable act;        // host copy
};

// ---- collectible items (CX_KIND_PICKUP) of a single-agent game ----
// The agent tables above are built with every item absent (cx_game_create checks that they equal the tables with
// every item present), while basech / basek / baselay show every item present: the static scene of a fresh episode.
// Each env keeps a u64 of the items it still holds (CxStateLayout::off_pick).  The PICK build of k_agent_rollout_obs
// stages the region below after the observation extension and pokes an item's cell between its present and absent
// bytes when the bit changes.
#define CX_MAX_PICKUPS 64
#define CX_NO_ITEM 0xFF
struct CxPickItem {          // one item cell, or one door cell
  uint8_t cell;
  uint8_t under_ch;          // board character once the item is taken / the door is open (the static scene without it)
  uint8_t under_k;           // its channel in the canonical order (0xFF: not a game character)
  uint8_t drape;             // index into the CxPickDrape array (door cells: the door's index)
};
struct CxPickDrape {         // one pickup drape
  uint64_t items;            // bits of its items
  float reward[CX_MAX_ACTIONS + 1];  // add_reward value of a step that takes one of them (entry_reward[a][own char])
  float emptied_value;       // discount of the terminate_episode call once the last one is taken
  int32_t terminates;        // cx_entity_desc::terminate_emptied
  uint32_t opens;            // doors whose key it is (bit d: door d), open once it is empty
};
struct CxPickHeader {
  int32_t n_items;           // 0: the game has no pickups
  int32_t after;             // the pickups update after the agent: they see its post-move cell (else its pre-move cell)
  int32_t off;               // byte offset of the staged region in the blob (16-byte aligned) ...
  int32_t bytes;             // ... and its size (a multiple of 16)
  int32_t item_at;           // region offsets: u8 [cells+1] item index of every cell (CX_NO_ITEM: none) ...
  int32_t items;             // ... CxPickItem [n_items + door cells] ...
  int32_t drapes;            // ... CxPickDrape [n_drapes] (8-byte aligned)
  int32_t pad;
  uint64_t all;              // every item present
  // ---- key-locked doors (CX_KIND_DOOR).  Door d is open iff (items & door_keys[d]) == 0: the open doors of a step
  // are a function of the items at its start, and the doors a frame shows of the items at its end.  The cells of
  // every door follow the items as further CxPickItem entries (under_ch / under_k: the scene without the door), so
  // that item_at and the ring slots' shown words cover them: bit n_items + j of a slot's word = door cell j shown
  // closed.  The step tables of the other door states (1 .. 2^n_doors - 1; state 0, every door closed, is the agent
  // header's) follow the CxPickDrape array.
  int32_t n_doors;           // 0..CX_MAX_DOORS
  int32_t door_tt, door_tr, door_td;  // region offsets of u32 / f32 / f32 [2^n_doors - 1][table] step tables
  int32_t tt_size, td_size;  // elements of one tt / tr table ((n_actions+1)*(cells+1)) and of one td table
  int32_t tt_first, tr_first, td_first;  // staged: element offset of door state 1's tt / tr / td from the agent
                             // header's (the region lies behind the observation extension in shared memory)
  int32_t drape_cells;       // region offset of u64 [n_drapes]: shown-word bits of the cells of the doors each
                             // pickup drape opens (door games only)
  uint64_t door_keys[CX_MAX_DOORS];   // items of each door's key drape
  uint64_t door_cells[CX_MAX_DOORS];  // shown-word bits of each door's cells
  uint64_t scene_all;        // the static scene's shown word: every item present, every door closed
};

// The doors of a game in the state `items`: returns bit d set = door d open; *closed = shown-word bits of the cells of
// the closed doors.  The one statement of the door rule for the kernels.
__host__ __device__ inline uint32_t cx_doors(const CxPickHeader& P, uint64_t items, uint64_t* closed) {
  uint32_t open = 0;
  uint64_t shut = 0;
  for (int d = 0; d < P.n_doors; ++d) {
    if (items & P.door_keys[d])
      shut |= P.door_cells[d];
    else
      open |= 1u << d;
  }
  *closed = shut;
  return open;
}

// ---- generic path tables ----
struct CxGenEntity {
  uint8_t ch, kind, visible, group;
  uint8_t chidx, dyn_slot, stamps, watch;  // watch: z-index or 0xFF
  uint32_t blockers;
  uint8_t reward_actions, rank;
  uint8_t lin_slot;         // mask entities: index of the per-env linear bitset (0xFF: the static mask is used as is)
  uint8_t pad1;
  int8_t dr[CX_MAX_ACTIONS], dc[CX_MAX_ACTIONS];
  float step_reward[CX_MAX_ACTIONS];
  uint16_t init_state;      // cell / linear offset after its_showtime
  uint16_t pad2;
  uint8_t vis_op[CX_MAX_ACTIONS];  // sprites: cx_visible_op per action
  // directives evaluated per step only by games with a conditional terminate_episode (CxGenHeader::cond_term)
  uint8_t terminate_actions, discount_actions, pad3[2];
  float discount_value[CX_MAX_ACTIONS];
  uint32_t term_chars[CX_MAX_ACTIONS];   // cx_entity_desc::terminate_chars
  float term_value[CX_MAX_ACTIONS];
};

struct CxGenHeader {
  int32_t rows, cols, cells, n_actions, n_chars, n_ent, n_dyn, n_groups;
  int32_t mask_words;       // ceil(cells / 32)
  int32_t has_dynbd;        // quirk Q1(i): per-env backdrop plane
  int32_t zero_backdrop;    // quirk Q1(ii): no drape at all => canvas is zeroed every render
  int32_t needs_prev;       // some entity consults the last render (blockers / entry rewards / conditional terminate)
  int32_t cond_term;        // some entity terminates the episode depending on what its watched entity reached
  int8_t z_of_char[CX_MAX_CHARS];  // character index -> z index of the sprite / drape that owns it (-1: a backdrop
                            // character): unoccluded layers are read off the entity state (cx_game_desc::unoccluded_layers)
  int32_t max_steps, auto_reset, track;
  uint8_t update_order[CX_MAX_ENTITIES];  // z-indices in update order
  uint8_t chars[CX_MAX_CHARS];
  CxGenEntity ent[CX_MAX_ENTITIES];
  int32_t off_masks;        // u32 [n_ent][mask_words]  static masks as bitsets
  int32_t off_backdrop;     // u8  [cells]  per-env plane initial contents (after its_showtime stamps)
  int32_t off_entry;        // f32 [n_ent][n_actions][n_chars]
  int32_t off_rc;           // u16 [cells]  (row << 8 | col)
  int32_t off_rowbits;      // u64 [n_ent][rows]  static masks as one bitset per board row (cols <= 64), else -1
  int32_t tile_envs;        // envs per warp (power of two <= 32; the warp's backdrop-plane tile lives in shared memory)
  int32_t n_lin;            // per-env linear bitsets: rolling masks, and static masks with a visible point entity above
  int32_t fast_compose;     // the bitset composer applies (else: per-cell painter's algorithm)
  // the composer's view of the z-order, so that its loops touch one word per entity:
  int32_t n_masks, n_points;
  uint32_t mask_prog[CX_MAX_ENTITIES];   // mask entities back to front: z | ch << 8 | lin_slot << 16 | kind << 24
  uint32_t point_prog[CX_MAX_DYN];       // visible one-cell entities back to front: z | ch << 8 | dyn_slot << 16 | stamps << 24
  uint32_t point_holes[CX_MAX_DYN];      // bit s: per-env mask bitset s lies below the point entity (its cell is punched out)
  // direct composer only: the point entities by what the composer does with them
  int32_t n_poke;                        // below every mask and not stamping: poked into the plane around the composition
  int32_t n_above;                       // above every mask: stored over the finished board
  uint16_t above_prog[CX_MAX_DYN];       // back to front: ch << 8 | dyn_slot
  int32_t off_colroll[CX_MAX_LIN];       // per lin slot of a rolling drape: u32 [cols][mask_words + 1], the static mask
                                         // rolled right by dc columns, as linear bitsets; -1: not tabulated
  // direct composer: no per-env bitsets at all.  Every mask entity has a bit table in the blob -- one row
  // (static drape) or `cols` rows (rolling drape: the mask rolled right by dc columns), each row the linear
  // bitset followed by a copy of its first 16 bits (so a 16-bit slice may run over the end) -- and the
  // composer slices bits [S, S+16), S = (o - dr * cols) mod cells, straight from the row.  Visible one-cell
  // entities are either below every mask (poked into the plane) or above every mask (stored over the
  // finished board); games with a one-cell entity between two masks keep the per-env bitsets.
  int32_t direct;
  int32_t dtab_words;                    // u32 words per table row: ceil((cells + 16) / 32) + 1
  int32_t off_dtab[CX_MAX_ENTITIES];     // per mask_prog index
  // table-driven step: no entity looks at the last render (no blockers, no entry rewards) and there is one
  // update group, so a step is "move every dynamic slot by its per-action delta" and the reward is a
  // function of the action alone (summed on the host in update order, float32, plot.py:208-211)
  int32_t simple_step;
  uint8_t slot_kind[CX_MAX_DYN];         // cx_kind of the entity behind each dynamic slot
  int8_t slot_dr[CX_MAX_DYN][CX_MAX_ACTIONS], slot_dc[CX_MAX_DYN][CX_MAX_ACTIONS];
  float simple_reward[CX_MAX_ACTIONS];
  int32_t off_sdelta;                    // u32 [CX_MAX_ACTIONS][CX_MAX_DYN]: (dr mod rows) << 16 | (dc mod cols) per action and slot
  uint32_t roll_slots;                   // bit d: dynamic slot d holds a roll offset (row << 8 | col), not a cell index
  int32_t fast_loop;                     // simple_step && direct && cells <= 496 && n_masks <= 2: k_generic_rollout<true>
  int32_t n_stampers;
  uint16_t stamper[CX_MAX_DYN];          // back to front: ch << 8 | dyn_slot of the sprites that stamp the plane
  int32_t blob_bytes;
  CxActionTable act;
  // ---- render state that changes during play (SURVEY 8(f) row 3); such games run on the general step +
  // per-cell painter only.  The state lives in ordinary dynamic slots behind those of the moving entities.
  int32_t dyn_render;       // any of the three below
  int32_t slot_vis;         // slot with the sprite visibility bits (bit z: entity z is visible); -1: static
  int32_t slot_zperm;       // first of two slots with the z-order, 4 bits per position back to front
                            // (entity ids = initial z indices); -1: static
  int32_t slot_bd;          // slot with the backdrop's roll offset (row << 8 | col); -1: static backdrop
  uint16_t slot_init[CX_MAX_DYN];  // its_showtime value of every dynamic slot
  int8_t bd_dr[CX_MAX_ACTIONS], bd_dc[CX_MAX_ACTIONS];
  uint8_t n_zdir[CX_MAX_ACTIONS];
  uint8_t zdir[CX_MAX_ACTIONS][CX_MAX_ZDIR_GAME];  // move_this << 4 | in_front_of_that (0xF: None), in call order
};

// Episode statistics.  The float64[CX_STATS_DOUBLES] block at the head of the state blob holds the folded totals; the
// kernels accumulate into CX_STAT_STRIPES partial blocks behind it (same layout, one 64-byte line each), picked by the
// global warp index.  With one block, every warp of a launch sent its 5-7 atomics to the same line and the L2 worked
// them off one per clock: an episode end of all 65,536 envs of BASELINE config 1 (2,048 warps) cost 8 us on top of a
// 15 us launch, 28,000 atomics at 2^20 envs (measured, scripts/r02_probe.py stgsweep).  cx_stats_read / cx_stats_fold
// add the stripes into the head block and clear them.
#define CX_STAT_STRIPES 1024
#ifdef __CUDACC__
__device__ __forceinline__ double* cx_stat_stripe(double* stats, uint32_t key) {
  return stats + CX_STATS_DOUBLES * (1u + (key & (CX_STAT_STRIPES - 1u)));
}
#endif

// ---- state blob layout (caller-allocated; see cx_state_bytes) ----
struct CxStateLayout {
  int64_t n;
  int64_t off_stats;   // 8 doubles at offset 0 (folded totals), then CX_STAT_STRIPES partial blocks of 8 doubles
  int64_t off_tstep;   // u16 [n]
  int64_t off_ret;     // f32 [n]
  int64_t off_dyn;     // agent path: u8 [n]; generic: u16 [n_dyn][n]
  int64_t off_dynbd;   // generic + Q1: u8 [n][cells]
  int64_t off_perf;    // games that track performance: f32 [n] running performance of the current episode
  int64_t off_pick;    // games with pickups: u64 [n] items each env still holds (CxPickHeader)
  int64_t total;
};

struct cx_game {
  int path;
  cx_game_desc desc;       // copy (host pointers nulled)
  cx_game_info info;
  CxAgentHeader ah;
  CxGenHeader gh;
  CxPickHeader ph;         // single-agent games with CX_KIND_PICKUP drapes
  uint8_t* d_blob;         // device tables
  uint8_t* d_chars;        // device copy of chars[] for the layer kernels
  int device;
  int sm_count;
  int smem_per_sm;   // cudaDevAttrMaxSharedMemoryPerMultiprocessor (bytes)
};

CxStateLayout cx_layout(const cx_game* g, int64_t n);
void cx_set_error(const char* fmt, ...);

#define CX_CUDA_OK(expr)                                                              \
  do {                                                                                \
    cudaError_t _e = (expr);                                                          \
    if (_e != cudaSuccess) {                                                          \
      cx_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return CX_ERR_CUDA;                                                             \
    }                                                                                 \
  } while (0)

// Function attributes (the dynamic shared-memory cap) are set per DEVICE: remember, per call site, on which devices
// it has been done (bit = device ordinal; ordinals >= 64 are configured on every launch).  Safe to use from several
// host threads: configuring twice is harmless, launching unconfigured is not.
struct CxPerDevice {
  std::atomic<uint64_t> done{0};
  int dev = -1;
  bool need() {
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return true;
    return !(done.load(std::memory_order_acquire) & (1ull << dev));
  }
  void mark() {
    int d = -1;
    if (cudaGetDevice(&d) == cudaSuccess && d >= 0 && d < 64) done.fetch_or(1ull << d, std::memory_order_release);
  }
};

// synthetic-action request: when `on`, kernels generate actions (cx_philox.cuh) instead of reading them
struct CxSynth {
  int on;
  uint64_t seed, env_offset, t0;
  uint8_t* actions_out;  // [T, n] or null
};

// A kernel route forced through the environment variable CX_ROUTE (cx_game.cu: parse_route), so that tests can run
// every kernel on the same inputs.  Anything the forced route does not cover keeps its automatic choice.
enum CxRoute {
  CX_ROUTE_AUTO,              // CX_ROUTE unset: automatic selection
  CX_ROUTE_TILE64,            // tile64 / tile128 / tile256: k_agent_rollout with 64 / 128 / 256 envs per warp at every
  CX_ROUTE_TILE128,           //   batch size (its ragged rest still runs on k_agent_rollout_lane)
  CX_ROUTE_TILE256,
  CX_ROUTE_LANE,              // lane: k_agent_rollout_lane for every rollout it takes, whatever the batch size
  CX_ROUTE_OBS,               // obs: k_agent_rollout_obs in place of k_agent_rollout_lane and k_agent_rollout
  CX_ROUTE_NO_STEP_COMPOSER,  // no_step_composer: single steps never take the stateless composer (k_agent_step_flat)
  CX_ROUTE_STEP_COMPOSER,     // step_composer: single steps take it at any batch size
  CX_ROUTE_GEN96,             // gen96 / gen80 / gen_wave: the 96-register, 80-register or one-wave build of the
  CX_ROUTE_GEN80,             //   register-state generic kernel
  CX_ROUTE_GEN_WAVE,
};

// kernel launchers (defined in the kernel translation units)
int cx_launch_agent_rollout(const cx_game* g, void* d_state, int64_t n, int32_t T, const uint8_t* d_actions,
                            const CxSynth& synth, float* d_reward, float* d_discount, uint8_t* d_flags,
                            uint8_t* d_board, CxRoute route, cudaStream_t s);
int cx_launch_agent_rollout_obs(const cx_game* g, void* d_state, int64_t n, int32_t T, const uint8_t* d_actions,
                                const CxSynth& synth, float* d_reward, float* d_discount, uint8_t* d_flags,
                                uint8_t* d_board, uint8_t* d_layered /* or null */, cudaStream_t s);
bool cx_agent_obs_applies(const cx_game* g, bool layers);
size_t cx_agent_obs_smem_bytes(const cx_game* g);   // its shared memory for board-only rollouts, one tile per warp
// the whole policy rollout of a single-agent game in one launch (cx_agent_policy_kernels.cu)
int cx_launch_agent_policy_rollout(const cx_game* g, void* d_state, int64_t n, int32_t T, const float* d_w1t,
                                   const float* d_b1, int32_t n_hidden, const float* d_w2, const float* d_b2, uint64_t seed,
                                   uint64_t env_offset, const uint64_t* d_step, uint64_t step_offset, float* d_states,
                                   uint8_t* d_actions, float* d_reward, uint8_t* d_flags, float* d_logp, cudaStream_t s);
// small batches of single-agent games: lane = env, boards copied out with STG.128 (cx_agent_lane_kernels.cu)
bool cx_agent_lane_applies(const cx_game* g, int64_t n, const void* d_actions, const void* d_actions_out,
                           const void* d_reward, const void* d_discount, const void* d_flags, const void* d_board);
// env_base > 0 (a multiple of 32): only envs [env_base, n), the rest behind the whole tiles of k_agent_rollout
int cx_launch_agent_rollout_lane(const cx_game* g, void* d_state, int64_t n, int32_t T, const uint8_t* d_actions,
                                 const CxSynth& synth, float* d_reward, float* d_discount, uint8_t* d_flags,
                                 uint8_t* d_board, cudaStream_t s, int64_t env_base = 0);
// one Engine.play() per launch, stateless composer (cx_agent_step_kernels.cu); lay_dtype: CX_DTYPE_* of d_layered
bool cx_agent_step_applies(const cx_game* g, const void* d_board, const void* d_layered);
// d_actions == nullptr: render only (nothing is stepped, the state is not written)
int cx_launch_agent_step(const cx_game* g, void* d_state, int64_t n, const uint8_t* d_actions, float* d_reward,
                         float* d_discount, uint8_t* d_flags, uint8_t* d_board, void* d_layered, int lay_dtype,
                         cudaStream_t s);
// d_layered (optional, games with cx_game_desc::unoccluded_layers): [T, n, n_chars, cells] / [n, n_chars, cells] uint8
// unoccluded layers of every frame, read off the entity state inside the kernel
int cx_launch_generic_rollout(const cx_game* g, void* d_state, int64_t n, int32_t T, const uint8_t* d_actions,
                              const CxSynth& synth, float* d_reward, float* d_discount, uint8_t* d_flags,
                              uint8_t* d_board, CxRoute route, cudaStream_t s, uint8_t* d_layered = nullptr);
int cx_launch_reset(const cx_game* g, void* d_state, int64_t n, const uint8_t* d_mask, cudaStream_t s);
int cx_launch_stats_fold(void* d_state, cudaStream_t s);
int cx_launch_render(const cx_game* g, const void* d_state, int64_t n, uint8_t* d_board, cudaStream_t s);
int cx_launch_generic_render(const cx_game* g, const void* d_state, int64_t n, uint8_t* d_board, cudaStream_t s,
                             uint8_t* d_layered = nullptr);
int cx_launch_get_entity(const cx_game* g, const void* d_state, int64_t n, int32_t z, int32_t* d_out,
                         cudaStream_t s);
int cx_launch_set_entity(const cx_game* g, void* d_state, int64_t n, int32_t z, const int32_t* d_in,
                         cudaStream_t s);
int cx_launch_get_episode(const cx_game* g, const void* d_state, int64_t n, int32_t* d_steps, float* d_ret,
                          cudaStream_t s);
int cx_launch_get_render_state(const cx_game* g, const void* d_state, int64_t n, uint32_t* d_zorder,
                               uint32_t* d_visible, int32_t* d_backdrop_off, cudaStream_t s);
