// Generic path: any game made of the four entity primitives (static drape, one-cell drape, rolling
// drape, sprite), several moving entities, several update groups, and the backdrop-stamping quirk Q1.
// Used by Hello World (13x36: RollingDrape + 4 SlidingSprites, `Hello World Example.ipynb` cells 3-4).
//
// Reference lines restated per env-step:
//   update order / groups      campx/engine.py:184-208 (re-render after every group)
//   RollingDrape / SlidingSprite   Hello World notebook cell 3 (np.roll of the mask; (row,col) += d mod size)
//   one-cell drape with wall gate  examples/boat_race.py:35-59
//   entry rewards              boat_race.py:76-90, Demo 3 cell 3
//   painter's algorithm        engine.py:306-321 + rendering.py:111,128,150,173-178 -- including the
//                              storage aliasing: sprites painted before the first drape write into the
//                              backdrop itself (per-env backdrop plane), and a game without any drape
//                              has its canvas zeroed at every render
//   plot directives            campx/plot.py:161-257, engine.py:285-290
//
// B200 mapping.  One WARP owns `tile_envs` (8..32) consecutive envs for all T fused steps and keeps
// their BACKDROP PLANES (static scenery + quirk-Q1 sprite stamps; loaded once per launch, written back
// once) as one byte tile in shared memory.  Warps never wait on a block barrier after the tables are
// staged.  A step is
//   phase 1   lane = env: entity state update in update order (a few bytes in shared memory), stamps
//             into the plane tile;
//   phase 1b  whole warp: the masks that differ per env (rolled drapes; static drapes with a one-cell
//             entity above them) are rebuilt as LINEAR bitsets (bit = cell index) in shared memory: a
//             roll is a 64-bit rotate per board row, re-packed 32 cells per lane;
//   phase 1c  lane = env: cells of one-cell entities are punched out of the masks below them and their
//             characters poked into the plane tile (un-poked after the step), so that ...
//   phase 2   ... composing is only "plane bytes, overlaid by each mask entity in z-order": one lane per
//             16-byte chunk of the board tile: LDS.128 of the plane, per mask entity a 16-bit slice of its
//             bitset (funnel shift), expanded to byte masks (multiply trick) and merged with LOP3, then
//             STG.128 (st.global.cs) straight from registers.  Chunks that straddle two envs (cells is
//             not a multiple of 16) take a second pass with two slices per mask.
// DIRECT composer (CxGenHeader::direct: at most 2 mask entities on boards of at most 496 cells; Hello World): phases
// 1b/1c disappear.  A rolled mask is a slice of a host-built table (row dc = the static mask rolled by dc columns as
// a linear bitset with wrap-around bits; the row roll is a rotation by dr * cols bits, i.e. an offset into that row),
// lane l of iteration k composes chunk 32 k + l of the warp's tile, so every warp store is one aligned 512-byte run
// of whole lines, and one-cell entities above the masks are byte-stored over the finished board.  Games whose
// entities never consult the last render keep their entity state in registers (k_generic_rollout<true, ...>).
// Per env-step HBM traffic is the observation contract only (board + reward + flags + discount + action);
// entity state and the plane move once per launch.  Games with more than CX_MAX_LIN per-env masks, rolling
// drapes wider than 64 columns, or unaligned buffers use the per-cell painter's algorithm instead.
#include "cx_episode.cuh"
#include "cx_philox.cuh"

namespace {

constexpr int kChunkUnroll = 2;  // chunks of the composer loop in flight per lane (ILP)
constexpr int kMinCtas = 5;      // resident CTAs per SM the register allocation aims for (5 x 128 threads x 96 registers);
                                 // the register-state kernel is also built for one CTA more, see cx_launch_generic_rollout
constexpr int kFlatUnroll = 5;   // 512-byte groups of the flat composer in flight per warp
constexpr int NT = CX_GEN_CTA_THREADS;
constexpr int kWaveThreads = 448;  // fat CTAs of the one-wave build: 2 x 448 threads x 72 registers per SM

struct GenParams {
  CxGenHeader h;
  const uint8_t* blob;
  uint16_t* dyn;     // [n_dyn][n]
  uint16_t* tstep;   // [n]
  float* ret;        // [n]
  uint8_t* dynbd;    // [n][cells]
  double* stats;
  const uint8_t* actions;
  float* reward;
  float* discount;
  uint8_t* flags;
  uint8_t* board;
  uint8_t* layered;               // [T, n, n_chars, cells] unoccluded layers (cx_game_desc::unoccluded_layers) or null
  int64_t n;
  int32_t T;
  int32_t vec;
  int32_t synth;                  // actions generated in the kernel (cx_philox.cuh)
  uint64_t seed, env_offset, t0;
  uint8_t* actions_out;
};

struct Ctx {
  const CxGenHeader* H;
  const uint32_t* masks;
  const uint8_t* backdrop;
  const float* entry;
  const uint16_t* rc;
  const uint64_t* rowbits;
  const uint8_t* chidx;  // [256] char code -> game char index (0xFF: not a game char)
  const uint8_t* smem;   // staged tables blob
  const uint4* act;      // [n_actions] {simple_reward bits, discount bits, directive flags, 0}: one LDS.128 per step
};

// per-warp view of the shared-memory working set
struct WarpMem {
  uint8_t* plane;              // [G][cells] backdrop planes, tile-contiguous like the board rows in HBM
  uint32_t* lin;               // [G][n_lin][mask_words + 1] per-env mask bitsets (last word stays 0)
  uint16_t (*dyn)[CX_MAX_DYN]; // [G] entity state
  uint16_t (*prev)[CX_MAX_DYN];
};

__device__ __forceinline__ bool mask_bit(const Ctx& X, int z, int cell) {
  return (X.masks[z * X.H->mask_words + (cell >> 5)] >> (cell & 31)) & 1u;
}

// ---- render state that changes during play (CxGenHeader::dyn_render) ----------------------------------------
// z-order of this env: 4 bits per position back to front (engine.py:242-281 rebuilds the OrderedDict)
__device__ __forceinline__ uint32_t zperm_of(const CxGenHeader& H, const uint16_t* st) {
  return H.slot_zperm >= 0 ? (uint32_t)st[H.slot_zperm] | ((uint32_t)st[H.slot_zperm + 1] << 16) : 0x76543210u;
}
__device__ __forceinline__ int z_at(const CxGenHeader& H, uint32_t perm, int p) {
  return H.slot_zperm >= 0 ? (int)((perm >> (4 * p)) & 15u) : p;
}
// Sprite.visible (things.py:390-392; engine.py:315 paints visible sprites only)
__device__ __forceinline__ bool visible_now(const CxGenHeader& H, const uint16_t* st, int z) {
  return H.slot_vis >= 0 ? ((st[H.slot_vis] >> z) & 1u) != 0 : H.ent[z].visible != 0;
}
// Backdrop character at `cell`: the per-env plane, or the static scenery rolled by the backdrop's offset
// (Backdrop.update, things.py:103-148, fitted as a toroidal roll of its curtain)
__device__ __forceinline__ uint8_t backdrop_at(const Ctx& X, const uint16_t* st, const uint8_t* plane, int cell) {
  const CxGenHeader& H = *X.H;
  if (H.slot_bd < 0) return plane[cell];
  const uint32_t off = st[H.slot_bd], rcv = X.rc[cell];
  int r = (int)(rcv >> 8) - (int)(off >> 8), c = (int)(rcv & 255) - (int)(off & 255);
  if (r < 0) r += H.rows;
  if (c < 0) c += H.cols;
  return X.backdrop[r * H.cols + c];
}
// the_plot.change_z_order(move_this, in_front_of_that): engine.py:262-279
__device__ __forceinline__ uint32_t apply_zdir(uint32_t perm, int n_ent, uint32_t mv, uint32_t fr) {
  uint32_t out = 0;
  int k = 0;
  if (fr == 0xFu) out |= mv << (4 * k++);  // in_front_of_that is None: all the way to the back
  for (int p = 0; p < n_ent; ++p) {
    const uint32_t z = (perm >> (4 * p)) & 15u;
    if (z == mv) continue;
    out |= z << (4 * k++);
    if (z == fr) out |= mv << (4 * k++);
  }
  return out;
}

// Painter's algorithm at ONE cell on top of backdrop byte v (engine.py:310-321).  Used for the few
// point queries of the last render (wall gate, entry rewards) and by the wide-board fallback.
__device__ __forceinline__ uint8_t overlay(const Ctx& X, const uint16_t* st, int cell, uint8_t v) {
  const CxGenHeader& H = *X.H;
  const uint32_t perm = zperm_of(H, st);
  for (int p = 0; p < H.n_ent; ++p) {
    const int z = z_at(H, perm, p);
    const CxGenEntity& e = H.ent[z];
    bool covers;
    switch (e.kind) {
      case CX_KIND_STATIC:
        covers = mask_bit(X, z, cell);
        break;
      case CX_KIND_ROLL: {
        const uint32_t off = st[e.dyn_slot], rcv = X.rc[cell];
        int r = (int)(rcv >> 8) - (int)(off >> 8), c = (int)(rcv & 255) - (int)(off & 255);
        if (r < 0) r += H.rows;
        if (c < 0) c += H.cols;
        covers = mask_bit(X, z, r * H.cols + c);
        break;
      }
      case CX_KIND_SPRITE:
        covers = visible_now(H, st, z) && st[e.dyn_slot] == cell;
        break;
      default:  // CELL drape: one cell
        covers = st[e.dyn_slot] == cell;
    }
    if (covers) v = e.ch;
  }
  return v;
}

// rendering.py:150 through the alias of :128 -- sprites behind the first drape paint into the backdrop
__device__ __forceinline__ void stamp(const Ctx& X, const uint16_t* st, uint8_t* plane) {
  const CxGenHeader& H = *X.H;
  if (H.dyn_render) {  // who lies behind the first drape, and is visible, depends on this env's state
    if (!H.has_dynbd) return;
    const uint32_t perm = zperm_of(H, st);
    for (int p = 0; p < H.n_ent; ++p) {
      const int z = z_at(H, perm, p);
      const CxGenEntity& e = H.ent[z];
      if (e.kind != CX_KIND_SPRITE) break;  // rendering.py:178: the first drape re-seats the canvas
      if (visible_now(H, st, z)) plane[st[e.dyn_slot]] = e.ch;
    }
    return;
  }
  for (int i = 0; i < H.n_stampers; ++i) {
    const uint32_t sp = H.stamper[i];
    plane[st[sp & 0xFF]] = (uint8_t)(sp >> 8);
  }
}

__device__ __forceinline__ uint32_t wrap_move(const CxGenHeader& H, uint32_t r, uint32_t c, int dr, int dc,
                                              uint32_t* rr, uint32_t* cc) {
  int nr = (int)r + dr, nc = (int)c + dc;  // |dr| < rows, |dc| < cols (checked by cx_game_create)
  if (nr >= H.rows) nr -= H.rows;
  if (nc >= H.cols) nc -= H.cols;
  if (nr < 0) nr += H.rows;
  if (nc < 0) nc += H.cols;
  *rr = nr;
  *cc = nc;
  return nr * H.cols + nc;
}

// One env, one Engine.play(): entity updates in schedule order with a render after every update group.
// st: current state (updated in place); prev: scratch snapshot of the state at the last render;
// plane: this env's backdrop plane (shared memory).
__device__ void generic_env_step(const Ctx& X, uint32_t a, uint16_t* st, uint16_t* prev, uint8_t* plane,
                                 float& reward, uint32_t& flags, float& disc) {
  const CxGenHeader& H = *X.H;
  if (a >= (uint32_t)H.n_actions) {
    reward = 0.0f;
    disc = 1.0f;
    flags = CX_FLAG_BAD_ACTION | CX_FLAG_REWARD_NONE;
    return;
  }
  for (int d = 0; d < H.n_dyn; ++d) prev[d] = st[d];
  if (H.slot_bd >= 0) {  // engine.py:190: the backdrop updates first; entities still see the last render
    const uint32_t off = st[H.slot_bd];
    uint32_t rr, cc;
    wrap_move(H, off >> 8, off & 255, H.bd_dr[a], H.bd_dc[a], &rr, &cc);
    st[H.slot_bd] = (uint16_t)((rr << 8) | cc);
  }
  float summed = 0.0f;
  bool first = true;
  bool over = H.act.over[a] != 0;      // directives: per-action tables, unless some terminate_episode call depends
  float pdisc = H.act.discount[a];     // on where a watched entity stands (then replayed in update order below)
  if (H.cond_term) {
    over = false;
    pdisc = 1.0f;
  }
  int group = H.n_ent > 0 ? H.ent[H.update_order[0]].group : 0;
  for (int i = 0; i < H.n_ent; ++i) {
    const int z = H.update_order[i];
    const CxGenEntity& e = H.ent[z];
    if (e.group != group) {  // engine.py:208: the board is re-rendered before the next group updates
      stamp(X, st, plane);
      for (int d = 0; d < H.n_dyn; ++d) prev[d] = st[d];
      group = e.group;
    }
    const int dr = e.dr[a], dc = e.dc[a];
    if (e.kind == CX_KIND_CELL) {
      const uint32_t p = st[e.dyn_slot];
      if (p != CX_EMPTY_CELL16) {
        uint32_t rr, cc;
        const uint32_t rcv = X.rc[p];
        uint32_t t = wrap_move(H, rcv >> 8, rcv & 255, dr, dc, &rr, &cc);
        if (e.blockers) {
          const uint8_t k = X.chidx[overlay(X, prev, (int)t, backdrop_at(X, prev, plane, (int)t))];
          if (k != 0xFF && ((e.blockers >> k) & 1u)) {
            // fall back to the agent layer of the last render (boat_race.py:55-56)
            const uint32_t pp = prev[e.dyn_slot];
            const bool vis = pp != CX_EMPTY_CELL16 &&
                             overlay(X, prev, (int)pp, backdrop_at(X, prev, plane, (int)pp)) == e.ch;
            t = vis ? pp : CX_EMPTY_CELL16;
          }
        }
        st[e.dyn_slot] = (uint16_t)t;
      }
    } else if (e.kind == CX_KIND_SPRITE) {
      const uint32_t rcv = X.rc[st[e.dyn_slot]];
      uint32_t rr, cc;
      const uint32_t t = wrap_move(H, rcv >> 8, rcv & 255, dr, dc, &rr, &cc);
      // MazeWalker: a target the last render showed a blocker at is refused, and the sprite stays (visibility: KEEP)
      const uint8_t k = e.blockers ? X.chidx[overlay(X, prev, (int)t, backdrop_at(X, prev, plane, (int)t))] : 0xFF;
      if (k == 0xFF || !((e.blockers >> k) & 1u)) st[e.dyn_slot] = (uint16_t)t;
      if (H.slot_vis >= 0 && e.vis_op[a] != CX_VIS_KEEP) {
        const uint32_t bit = 1u << z, bits = st[H.slot_vis], op = e.vis_op[a];
        st[H.slot_vis] = (uint16_t)(op == CX_VIS_SHOW ? bits | bit : op == CX_VIS_HIDE ? bits & ~bit : bits ^ bit);
      }
    } else if (e.kind == CX_KIND_ROLL) {
      const uint32_t off = st[e.dyn_slot];
      uint32_t rr, cc;
      wrap_move(H, off >> 8, off & 255, dr, dc, &rr, &cc);
      st[e.dyn_slot] = (uint16_t)((rr << 8) | cc);
    }
    if ((e.reward_actions >> a) & 1u) {
      float r = e.step_reward[a];
      if (e.watch != 0xFF) {
        const uint32_t wc = st[H.ent[e.watch].dyn_slot];  // things[...] is current, not last-render, state
        if (wc != CX_EMPTY_CELL16) {
          const uint8_t k = X.chidx[overlay(X, prev, (int)wc, backdrop_at(X, prev, plane, (int)wc))];
          if (k != 0xFF) r = __fadd_rn(r, X.entry[(z * H.n_actions + a) * H.n_chars + k]);
        }
      }
      summed = first ? r : __fadd_rn(r, summed);  // plot.py:208-211
      first = false;
    }
    if (H.cond_term) {  // plot.py:161-184,232-257: the last call of the step wins
      if ((e.discount_actions >> a) & 1u) pdisc = e.discount_value[a];
      if ((e.terminate_actions >> a) & 1u) {
        over = true;
        pdisc = e.discount_value[a];
      }
      if (e.term_chars[a] && e.watch != 0xFF) {
        const uint32_t wc = st[H.ent[e.watch].dyn_slot];
        if (wc != CX_EMPTY_CELL16) {
          const uint8_t k = X.chidx[overlay(X, prev, (int)wc, backdrop_at(X, prev, plane, (int)wc))];
          if (k != 0xFF && ((e.term_chars[a] >> k) & 1u)) {
            over = true;
            pdisc = e.term_value[a];
          }
        }
      }
    }
  }
  stamp(X, st, plane);  // the render that produces this step's observation
  if (H.slot_zperm >= 0 && H.n_zdir[a]) {  // engine.py:242-281, then the re-render of engine.py:163
    uint32_t perm = zperm_of(H, st);
    for (int i = 0; i < H.n_zdir[a]; ++i) perm = apply_zdir(perm, H.n_ent, H.zdir[a][i] >> 4, H.zdir[a][i] & 15u);
    st[H.slot_zperm] = (uint16_t)perm;
    st[H.slot_zperm + 1] = (uint16_t)(perm >> 16);
    stamp(X, st, plane);
  }
  reward = summed;
  disc = pdisc;
  flags = (over ? CX_FLAG_TERMINATED : 0) | (H.act.reward_none[a] ? CX_FLAG_REWARD_NONE : 0);
}

// Engine.play() of a game whose entities never consult the last render (CxGenHeader::simple_step): every
// dynamic slot moves by its per-action toroidal delta; reward, discount and directives depend on the action
// alone.  Same results as generic_env_step.
__device__ __forceinline__ void simple_env_step(const Ctx& X, uint32_t a, uint16_t* st, uint8_t* plane, float& reward,
                                                uint32_t& flags, float& disc) {
  const CxGenHeader& H = *X.H;
  if (a >= (uint32_t)H.n_actions) {
    reward = 0.0f;
    disc = 1.0f;
    flags = CX_FLAG_BAD_ACTION | CX_FLAG_REWARD_NONE;
    return;
  }
  const int R = H.rows, C = H.cols;
  for (int d = 0; d < H.n_dyn; ++d) {
    const uint32_t s = st[d];
    const int dr = H.slot_dr[d][a], dc = H.slot_dc[d][a];
    uint32_t rc;
    const bool roll = H.slot_kind[d] == CX_KIND_ROLL;
    if (roll) {
      rc = s;
    } else {
      if (s == CX_EMPTY_CELL16) continue;
      rc = X.rc[s];
    }
    int r = (int)(rc >> 8) + dr, c = (int)(rc & 255u) + dc;  // |dr| < rows, |dc| < cols
    r += r < 0 ? R : 0;
    c += c < 0 ? C : 0;
    r -= r >= R ? R : 0;
    c -= c >= C ? C : 0;
    st[d] = (uint16_t)(roll ? (r << 8) | c : r * C + c);
  }
  stamp(X, st, plane);
  const uint4 at = X.act[a];
  reward = __uint_as_float(at.x);
  disc = __uint_as_float(at.y);
  flags = at.z;
}

// simple_env_step with the entity state in registers (k_generic_rollout<true>): sreg[d] = row << 16 | col for
// every kind (0xFFFFFFFF: empty one-cell mask).  The per-action deltas are tabulated as non-negative residues
// ((dr mod rows) << 16 | (dc mod cols)), so a move is ONE add for both coordinates and one fused add-min per
// coordinate for the toroidal wrap (x in [0, 2n-2]: min(x, x - n) as unsigned), with no table look-up in the
// dependency chain; the slots are independent instruction streams.  st[] (shared memory) receives the
// representation the composer reads: cell index, or roll offset (row << 8 | col) for rolling drapes.
__device__ __forceinline__ void fast_env_step(const Ctx& X, uint32_t a, uint32_t (&sreg)[CX_MAX_DYN], uint16_t* st,
                                              uint8_t* plane, float& reward, uint32_t& flags, float& disc) {
  const CxGenHeader& H = *X.H;
  if (a >= (uint32_t)H.n_actions) {
    reward = 0.0f;
    disc = 1.0f;
    flags = CX_FLAG_BAD_ACTION | CX_FLAG_REWARD_NONE;
    return;
  }
  const uint32_t R = H.rows, C = H.cols;
  const uint4* dl = reinterpret_cast<const uint4*>(X.smem + H.off_sdelta + a * (CX_MAX_DYN * 4));
  const uint4 d0 = dl[0];
  uint4 d1 = make_uint4(0u, 0u, 0u, 0u);
  if (H.n_dyn > 4) d1 = dl[1];
  const uint32_t w[CX_MAX_DYN] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
#pragma unroll
  for (int d = 0; d < CX_MAX_DYN; ++d) {
    if (d < H.n_dyn) {
      const uint32_t s = sreg[d];
      const uint32_t t = s + w[d];
      uint32_t r = t >> 16, c = t & 0xFFFFu;
      r = min(r, r - R);
      c = min(c, c - C);
      if (s != 0xFFFFFFFFu) {
        sreg[d] = (r << 16) | c;
        st[d] = (uint16_t)(((H.roll_slots >> d) & 1u) ? (r << 8) | c : r * C + c);
      }
    }
  }
  stamp(X, st, plane);
  const uint4 at = X.act[a];
  reward = __uint_as_float(at.x);
  disc = __uint_as_float(at.y);
  flags = at.z;
}
__device__ __forceinline__ void fast_load_state(const Ctx& X, const uint16_t* st, uint32_t (&sreg)[CX_MAX_DYN]) {
  const CxGenHeader& H = *X.H;
#pragma unroll
  for (int d = 0; d < CX_MAX_DYN; ++d) {
    sreg[d] = 0xFFFFFFFFu;
    if (d < H.n_dyn) {
      const uint32_t v = st[d];
      const bool roll = (H.roll_slots >> d) & 1u;
      if (roll || v != CX_EMPTY_CELL16) {
        const uint32_t rc = roll ? v : (uint32_t)X.rc[v];
        sreg[d] = ((rc >> 8) << 16) | (rc & 255u);
      }
    }
  }
}

__device__ __forceinline__ void setup_ctx(Ctx& X, const GenParams& P, uint8_t* smem, uint8_t* s_chidx, const uint4* s_act) {
  X.act = s_act;
  X.H = &P.h;
  X.masks = reinterpret_cast<const uint32_t*>(smem + P.h.off_masks);
  X.backdrop = smem + P.h.off_backdrop;
  X.entry = reinterpret_cast<const float*>(smem + P.h.off_entry);
  X.rc = reinterpret_cast<const uint16_t*>(smem + P.h.off_rc);
  X.rowbits = P.h.off_rowbits >= 0 ? reinterpret_cast<const uint64_t*>(smem + P.h.off_rowbits) : nullptr;
  X.chidx = s_chidx;
  X.smem = smem;
}

__device__ __forceinline__ void stage_tables(const GenParams& P, uint8_t* smem, uint8_t* s_chidx, uint4* s_act) {
  if (threadIdx.x < CX_MAX_ACTIONS) {  // per-action directives: indexed by a lane-varying action in the step
    const int a = threadIdx.x;
    s_act[a] = make_uint4(__float_as_uint(P.h.simple_reward[a]), __float_as_uint(P.h.act.discount[a]),
                          (P.h.act.over[a] ? CX_FLAG_TERMINATED : 0u) | (P.h.act.reward_none[a] ? CX_FLAG_REWARD_NONE : 0u), 0u);
  }
  const uint4* src = reinterpret_cast<const uint4*>(P.blob);
  uint4* dst = reinterpret_cast<uint4*>(smem);
  for (int i = threadIdx.x; i < P.h.blob_bytes / 16; i += blockDim.x) dst[i] = src[i];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) {
    uint8_t k = 0xFF;
    for (int j = 0; j < P.h.n_chars; ++j)
      if (P.h.chars[j] == i) k = (uint8_t)j;
    s_chidx[i] = k;
  }
}

// x / d by multiplication with ceil(2^32 / d): exact while x * d < 2^32 (tiles are < 2^17 bytes, d <= 4096)
__device__ __forceinline__ uint32_t div_inverse(uint32_t d) { return d == 1u ? 0u : 0xFFFFFFFFu / d + 1u; }
__device__ __forceinline__ uint32_t fast_div(uint32_t x, uint32_t inv) { return inv ? __umulhi(x, inv) : x; }

// phase 1b: rebuild the per-env linear bitsets (32 cells per lane and task)
__device__ __forceinline__ void build_linear_masks(const Ctx& X, const WarpMem& W, int nenv, int lane) {
  const CxGenHeader& H = *X.H;
  if (H.n_lin == 0) return;
  const int mw = H.mask_words, lw = mw + 1, R = H.rows, C = H.cols;
  const uint32_t inv_mw = div_inverse((uint32_t)mw);
  const uint64_t full = C >= 64 ? ~0ull : ((1ull << C) - 1ull);
  for (int i = 0; i < H.n_masks; ++i) {
    const uint32_t prog = H.mask_prog[i];
    const uint32_t z = prog & 0xFF, ls = (prog >> 16) & 0xFF, kind = prog >> 24;
    if (ls == 0xFF) continue;
    const uint32_t slot = H.ent[z].dyn_slot;
    const uint64_t* rows = X.rowbits + z * R;
    const int32_t off_cr = kind == CX_KIND_ROLL ? H.off_colroll[ls] : -1;
    const uint32_t* colroll = reinterpret_cast<const uint32_t*>(X.smem + (off_cr >= 0 ? off_cr : 0));
    for (int task = lane; task < nenv * mw; task += 32) {
      const int e = (int)fast_div((uint32_t)task, inv_mw), j = task - e * mw;
      uint32_t w;
      if (kind == CX_KIND_STATIC) {
        w = X.masks[z * mw + j];
      } else if (off_cr >= 0) {
        // rolled mask = (static mask rolled by dc columns: tabulated) rotated by dr * cols bits
        const uint32_t s = W.dyn[e][slot];
        const uint32_t* src = colroll + (s & 255u) * lw;
        int S = 32 * j - (int)(s >> 8) * C;          // first source bit of this word
        if (S < 0) S += H.cells;
        w = __funnelshift_r(src[S >> 5], src[(S >> 5) + 1], S & 31);
        const int n1 = H.cells - S;                  // bits left before the bitset wraps around
        if (n1 < 32) w = (w & ((1u << n1) - 1u)) | (src[0] << n1);
      } else {  // rolled mask (np.roll: content moves down/right by the accumulated offset): gather cells
                // 32j .. 32j+31 from the rotated board rows
        const uint32_t s = W.dyn[e][slot], k = s & 255u;
        const uint32_t rcv = X.rc[32 * j];
        int r = (int)(rcv >> 8), c = (int)(rcv & 255), got = 0;
        int sr = r - (int)(s >> 8);
        if (sr < 0) sr += R;
        w = 0;
        while (got < 32 && r < R) {
          const uint64_t x = rows[sr];
          const uint64_t bits = (k ? ((x << k) | (x >> (C - k))) & full : x) >> c;
          w |= (uint32_t)(bits << got);
          got += C - c;
          c = 0;
          ++r;
          if (++sr == R) sr = 0;
        }
      }
      W.lin[(e * H.n_lin + ls) * lw + j] = w;
    }
  }
}

// phase 1c (lane = env): one-cell entities.  Their cells are punched out of every per-env mask BELOW them
// in z-order and their characters poked into the plane in z-order, so that the composer only deals with
// masks.  Returns the plane bytes that were overwritten (one per dynamic slot) for unpoke_points().
__device__ __forceinline__ uint64_t poke_points(const Ctx& X, const WarpMem& W, int e) {
  const CxGenHeader& H = *X.H;
  const int lw = H.mask_words + 1;
  uint8_t* plane = W.plane + e * H.cells;
  uint32_t* lin = W.lin + e * H.n_lin * lw;
  uint64_t saved = 0;
  for (int i = 0; i < H.n_points; ++i) {
    const uint32_t prog = H.point_prog[i], slot = (prog >> 16) & 0xFF;
    const uint32_t s = W.dyn[e][slot];
    if (s == CX_EMPTY_CELL16) continue;
    for (uint32_t holes = H.point_holes[i]; holes; holes &= holes - 1)
      lin[(__ffs(holes) - 1) * lw + (s >> 5)] &= ~(1u << (s & 31));
    if (!(prog >> 24)) {  // stamping sprites are in the plane for good (quirk Q1)
      saved |= (uint64_t)plane[s] << (8 * slot);
      plane[s] = (uint8_t)(prog >> 8);
    }
  }
  return saved;
}
__device__ __forceinline__ void unpoke_points(const Ctx& X, const WarpMem& W, int e, uint64_t saved) {
  const CxGenHeader& H = *X.H;
  uint8_t* plane = W.plane + e * H.cells;
  for (int i = H.n_points - 1; i >= 0; --i) {  // reverse order: restores what was under stacked entities
    const uint32_t prog = H.point_prog[i], slot = (prog >> 16) & 0xFF;
    if (prog >> 24) continue;
    const uint32_t s = W.dyn[e][slot];
    if (s != CX_EMPTY_CELL16) plane[s] = (uint8_t)(saved >> (8 * slot));
  }
}

// 4 mask bits -> 4 byte masks (0x00 / 0xFF): the multiply moves bit i to the top of byte i (no carries),
// the byte permute replicates each byte's top bit
// (prmt selector nibble 8|i = "sign of byte i"; __byte_perm masks that bit off, hence the inline PTX)
__device__ __forceinline__ uint32_t expand4(uint32_t nib) {
  uint32_t m;
  asm("prmt.b32 %0, %1, 0, 0xBA98;" : "=r"(m) : "r"(nib * 0x10204080u));
  return m;
}

// branch-free on purpose: the chunk loop is straight-line code, so two chunks per lane interleave (ILP).
// Only bits 0-15 of `slice` are used.  Nibbles at bits 4-7 are expanded in place with their own multiplier
// (bit 4+i -> bit 7+8i), which saves the shifts.
__device__ __forceinline__ uint32_t expand4_hi(uint32_t nib_at_4) {
  uint32_t m;
  asm("prmt.b32 %0, %1, 0, 0xBA98;" : "=r"(m) : "r"(nib_at_4 * 0x01020408u));
  return m;
}
__device__ __forceinline__ void overlay16(uint4& v, uint32_t slice, uint32_t ch4) {
  const uint32_t hi = slice >> 8;
  uint32_t m;
  m = expand4(slice & 0x0Fu);     v.x = (v.x & ~m) | (ch4 & m);
  m = expand4_hi(slice & 0xF0u);  v.y = (v.y & ~m) | (ch4 & m);
  m = expand4(hi & 0x0Fu);        v.z = (v.z & ~m) | (ch4 & m);
  m = expand4_hi(hi & 0xF0u);     v.w = (v.w & ~m) | (ch4 & m);
}

// bits [o, o+16) of a linear bitset (one word of slack behind the last is readable)
__device__ __forceinline__ uint32_t slice16(const uint32_t* bits, uint32_t o) {
  const uint32_t j = o >> 5;
  return __funnelshift_r(bits[j], bits[j + 1], o & 31u) & 0xFFFFu;
}

// phase 2: compose this warp's board tile chunk by chunk and stream it to `dst` (16-byte aligned)
__device__ __forceinline__ void compose_stream(const Ctx& X, const WarpMem& W, int nenv, uint8_t* dst, int lane) {
  const CxGenHeader& H = *X.H;
  const uint32_t cells = H.cells, mw = H.mask_words, lw = mw + 1, env_words = H.n_lin * lw;
  const uint32_t inv_cells = div_inverse(cells);
  const int nchunks = nenv * (int)cells / 16, n_masks = H.n_masks;
  const uint4* p16 = reinterpret_cast<const uint4*>(W.plane);
  uint4* d16 = reinterpret_cast<uint4*>(dst);
  // pass A: chunks inside one env.  The first four mask entities' programs live in registers.
  constexpr int HOIST = 4;
  uint32_t prog[HOIST];
#pragma unroll
  for (int i = 0; i < HOIST; ++i) prog[i] = i < n_masks ? H.mask_prog[i] : 0u;
  uint32_t ch4[HOIST], lsw[HOIST];
  const uint32_t* sbits[HOIST];
#pragma unroll
  for (int i = 0; i < HOIST; ++i) {
    const uint32_t ls = (prog[i] >> 16) & 0xFF;
    ch4[i] = ((prog[i] >> 8) & 0xFF) * 0x01010101u;
    lsw[i] = ls * lw;
    sbits[i] = ls == 0xFF ? X.masks + (prog[i] & 0xFF) * mw : nullptr;  // shared static mask, or per-env bitset
  }
#pragma unroll kChunkUnroll
  for (int k = lane; k < nchunks; k += 32) {
    const uint32_t b = 16u * k, e = fast_div(b, inv_cells), o = b - e * cells;
    uint4 v = p16[k];
    const uint32_t* lin_e = W.lin + e * env_words;
#pragma unroll
    for (int i = 0; i < HOIST; ++i) {
      if (i < n_masks) {
        const uint32_t* bits = sbits[i] ? sbits[i] : lin_e + lsw[i];
        overlay16(v, slice16(bits, o), ch4[i]);
      }
    }
    for (int i = HOIST; i < n_masks; ++i) {
      const uint32_t pg = H.mask_prog[i], ls = (pg >> 16) & 0xFF;
      const uint32_t* bits = ls == 0xFF ? X.masks + (pg & 0xFF) * mw : lin_e + ls * lw;
      overlay16(v, slice16(bits, o), ((pg >> 8) & 0xFF) * 0x01010101u);
    }
    if (o + 16u <= cells) __stcs(d16 + k, v);  // else: the chunk straddles two envs -> pass B
  }
  // pass B: the chunk across the boundary between env i-1 and env i (lane i), if there is one
  if ((cells & 15u) != 0) {
    for (int i = lane + 1; i < nenv; i += 32) {
      const uint32_t b = (uint32_t)i * cells;
      if ((b & 15u) == 0) continue;
      const uint32_t k = b >> 4, cnt = b - 16u * k;       // cnt cells of env i-1, 16-cnt cells of env i
      const uint32_t o = cells - cnt, lo_mask = (1u << cnt) - 1u;
      uint4 v = p16[k];
      for (int m = 0; m < n_masks; ++m) {
        const uint32_t prog = H.mask_prog[m], ls = (prog >> 16) & 0xFF;
        uint32_t sl;
        if (ls == 0xFF) {
          const uint32_t* bits = X.masks + (prog & 0xFF) * mw;
          sl = (slice16(bits, o) & lo_mask) | ((bits[0] << cnt) & 0xFFFFu);
        } else {
          const uint32_t* b0 = W.lin + (i - 1) * env_words + ls * lw;
          sl = (slice16(b0, o) & lo_mask) | ((b0[env_words] << cnt) & 0xFFFFu);
        }
        overlay16(v, sl, ((prog >> 8) & 0xFF) * 0x01010101u);
      }
      __stcs(d16 + k, v);
    }
  }
}

// ---- direct composer (CxGenHeader::direct) ------------------------------------------------------------
// bits [S, S+16) of a table row; rows carry 16 wrap-around bits and a slack word behind the bitset
struct DirectMask {
  const uint32_t* row;  // table row of this env (static drape: the only row; rolling drape: row dc)
  uint32_t rot;         // (cells - dr * cols) mod cells: first source bit of cell 0
};
__device__ __forceinline__ DirectMask direct_mask(const Ctx& X, const WarpMem& W, int i, int e) {
  const CxGenHeader& H = *X.H;
  const uint32_t prog = H.mask_prog[i];
  DirectMask m;
  m.row = reinterpret_cast<const uint32_t*>(X.smem + H.off_dtab[i]);
  m.rot = 0;
  if ((prog >> 24) == CX_KIND_ROLL) {
    const uint32_t s = W.dyn[e][H.ent[prog & 0xFF].dyn_slot];
    m.row += (s & 255u) * H.dtab_words;
    const uint32_t back = (s >> 8) * H.cols;
    m.rot = back ? H.cells - back : 0u;
  }
  return m;
}
__device__ __forceinline__ uint32_t direct_slice(const DirectMask& m, uint32_t o, uint32_t cells) {
  uint32_t S = o + m.rot;
  S = min(S, S - cells);  // S mod cells (unsigned wrap makes S - cells huge while S < cells)
  const uint32_t j = S >> 5;
  return __funnelshift_r(m.row[j], m.row[j + 1], S & 31u);  // bits 16-31: don't care
}

// Boards of at most 496 cells, exactly NM masks.  Flat chunk mapping: lane l of iteration k composes chunk 32 k + l
// of the warp's board tile, so every warp store is one 512-byte, 512-byte-aligned run of whole lines (a mapping
// that follows the envs -- 29 of 32 lanes storing from a 16-byte-aligned start, 5 partial lines per store --
// measured 4.4 TB/s against 5.6 TB/s for aligned runs, see profiles/r01_ncu_generic_rollout.md).
// The env of a chunk is one multiplication with the inverse of `cells`; its table row and rotation come from the
// lane that owns the env (SHFL with a per-lane source).  Chunks that straddle two envs are left to lane = env below.
template <int NM, int U>
__device__ __forceinline__ void compose_direct_flat(const Ctx& X, const WarpMem& W, int nenv, uint8_t* dst, int lane) {
  const CxGenHeader& H = *X.H;
  const uint32_t cells = H.cells;
  const uint4* p16 = reinterpret_cast<const uint4*>(W.plane);
  uint4* d16 = reinterpret_cast<uint4*>(dst);
  uint32_t pk[NM > 0 ? NM : 1], ch4[NM > 0 ? NM : 1];
#pragma unroll
  for (int i = 0; i < NM; ++i) {
    ch4[i] = ((H.mask_prog[i] >> 8) & 0xFF) * 0x01010101u;
    pk[i] = 0;
    if (lane < nenv) {
      const DirectMask m = direct_mask(X, W, i, lane);
      pk[i] = m.rot | ((uint32_t)(reinterpret_cast<const uint8_t*>(m.row) - X.smem) << 12);
    }
  }
  const uint32_t nchunks = (uint32_t)nenv * cells >> 4;     // the tile holds whole chunks (gen_vec_ok)
  const uint32_t inv_cells = div_inverse(cells);
#pragma unroll U
  for (uint32_t c0 = 0; c0 < nchunks; c0 += 32) {
    const uint32_t c = c0 + lane;
    const bool valid = c < nchunks;
    const uint32_t cc = valid ? c : 0u, b = 16u * cc;
    const uint32_t e = fast_div(b, inv_cells), o = b - e * cells;
    uint4 v = p16[cc];
#pragma unroll
    for (int i = 0; i < NM; ++i) {
      const uint32_t q = __shfl_sync(0xffffffffu, pk[i], e);
      DirectMask m;
      m.row = reinterpret_cast<const uint32_t*>(X.smem + (q >> 12));
      m.rot = q & 0xFFFu;
      overlay16(v, direct_slice(m, o, cells), ch4[i]);
    }
    if (valid && o + 16u <= cells) d16[c] = v;  // default policy: measured 3 % faster than st.global.cs here
  }
  // the chunk across the boundary between env i-1 and env i (lane i), if there is one
  if ((cells & 15u) != 0) {
    uint32_t pk_prev[NM > 0 ? NM : 1];
#pragma unroll
    for (int i = 0; i < NM; ++i) pk_prev[i] = __shfl_up_sync(0xffffffffu, pk[i], 1);
    const uint32_t b = (uint32_t)lane * cells;
    if (lane >= 1 && lane < nenv && (b & 15u) != 0) {
      const uint32_t k = b >> 4, cnt = b - 16u * k;       // cnt cells of env lane-1, 16-cnt cells of env lane
      const uint32_t o = cells - cnt, lo_mask = (1u << cnt) - 1u;
      uint4 v = p16[k];
#pragma unroll
      for (int i = 0; i < NM; ++i) {
        DirectMask m0, m1;
        m0.row = reinterpret_cast<const uint32_t*>(X.smem + (pk_prev[i] >> 12));
        m0.rot = pk_prev[i] & 0xFFFu;
        m1.row = reinterpret_cast<const uint32_t*>(X.smem + (pk[i] >> 12));
        m1.rot = pk[i] & 0xFFFu;
        overlay16(v, (direct_slice(m0, o, cells) & lo_mask) | (direct_slice(m1, 0u, cells) << cnt), ch4[i]);
      }
      d16[k] = v;
    }
  }
}

template <int U>
__device__ __forceinline__ void compose_direct(const Ctx& X, const WarpMem& W, int nenv, uint8_t* dst, int lane) {
  const CxGenHeader& H = *X.H;
  const uint32_t cells = H.cells;
  const int n_masks = H.n_masks;
  const uint4* p16 = reinterpret_cast<const uint4*>(W.plane);
  uint4* d16 = reinterpret_cast<uint4*>(dst);
  constexpr int HOIST = 2;
  uint32_t ch4[HOIST];
#pragma unroll
  for (int i = 0; i < HOIST; ++i) ch4[i] = i < n_masks ? ((H.mask_prog[i] >> 8) & 0xFF) * 0x01010101u : 0u;
  // pass A: one env per iteration (its table rows and rotations are warp-uniform), one lane per 16-byte chunk
  // that lies inside the env
  const bool small = cells <= 496u && n_masks <= 2;
  if (small) {
    if (n_masks == 0) compose_direct_flat<0, U>(X, W, nenv, dst, lane);
    else if (n_masks == 1) compose_direct_flat<1, U>(X, W, nenv, dst, lane);
    else compose_direct_flat<2, U>(X, W, nenv, dst, lane);
    return;
  }
#pragma unroll 2
  for (int e = 0; e < nenv; ++e) {
    const uint32_t b0 = (uint32_t)e * cells;
    const uint32_t c_lo = (b0 + 15u) >> 4, c_hi = (b0 + cells) >> 4;
    DirectMask dm[HOIST];
#pragma unroll
    for (int i = 0; i < HOIST; ++i)
      if (i < n_masks) dm[i] = direct_mask(X, W, i, e);
    for (uint32_t c = c_lo + lane; c < c_hi; c += 32) {
      const uint32_t o = 16u * c - b0;
      uint4 v = p16[c];
#pragma unroll
      for (int i = 0; i < HOIST; ++i)
        if (i < n_masks) overlay16(v, direct_slice(dm[i], o, cells), ch4[i]);
      for (int i = HOIST; i < n_masks; ++i) {
        const DirectMask m = direct_mask(X, W, i, e);
        overlay16(v, direct_slice(m, o, cells), ((H.mask_prog[i] >> 8) & 0xFF) * 0x01010101u);
      }
      __stcs(d16 + c, v);
    }
  }
  // pass B: the chunk across the boundary between env i-1 and env i (lane i), if there is one
  if ((cells & 15u) != 0) {
    for (int i = lane + 1; i < nenv; i += 32) {
      const uint32_t b = (uint32_t)i * cells;
      if ((b & 15u) == 0) continue;
      const uint32_t k = b >> 4, cnt = b - 16u * k;       // cnt cells of env i-1, 16-cnt cells of env i
      const uint32_t o = cells - cnt, lo_mask = (1u << cnt) - 1u;
      uint4 v = p16[k];
      for (int m = 0; m < n_masks; ++m) {
        const DirectMask m0 = direct_mask(X, W, m, i - 1), m1 = direct_mask(X, W, m, i);
        const uint32_t sl = (direct_slice(m0, o, cells) & lo_mask) | (direct_slice(m1, 0u, cells) << cnt);
        overlay16(v, sl, ((H.mask_prog[m] >> 8) & 0xFF) * 0x01010101u);
      }
      __stcs(d16 + k, v);
    }
  }
}

// one-cell entities of the direct composer: those below every mask are poked into the plane before the
// composition (and restored afterwards), those above every mask are stored over the finished board
__device__ __forceinline__ uint64_t poke_below(const Ctx& X, const WarpMem& W, int e) {
  const CxGenHeader& H = *X.H;
  uint8_t* plane = W.plane + e * H.cells;
  uint64_t saved = 0;
  for (int i = 0; i < H.n_points; ++i) {
    const uint32_t prog = H.point_prog[i], slot = (prog >> 16) & 0xFF;
    if (prog >> 24) continue;  // stamped for good (1) or above the masks (2)
    const uint32_t s = W.dyn[e][slot];
    if (s == CX_EMPTY_CELL16) continue;
    saved |= (uint64_t)plane[s] << (8 * slot);
    plane[s] = (uint8_t)(prog >> 8);
  }
  return saved;
}
__device__ __forceinline__ void store_above(const Ctx& X, const WarpMem& W, int e, uint8_t* dst) {
  const CxGenHeader& H = *X.H;
  for (int i = 0; i < H.n_above; ++i) {
    const uint32_t prog = H.above_prog[i];
    const uint32_t s = W.dyn[e][prog & 0xFF];
    if (s != CX_EMPTY_CELL16) dst[(uint32_t)e * H.cells + s] = (uint8_t)(prog >> 8);
  }
}

// Unoccluded layers of a warp's envs (cx_game_desc::unoccluded_layers, the intent of rendering.py:227-353), read off
// the entity state the frame was rendered from: layers[ch] = the whole curtain of drape ch (rolled / one cell), or
// where the BACKDROP holds ch -- the per-env plane, quirk-Q1 stamps included, rendering.py:283-286 -- plus, for a
// visible sprite, its cell (:309).  One byte per (env, character, cell), written cell by cell: the correctness route of
// games that need the generic kernels (the single-agent kernels emit these layers as part of their tiles).
__device__ __forceinline__ void emit_unoccluded_layers(const Ctx& X, const WarpMem& W, int nenv, uint8_t* dst, int lane) {
  const CxGenHeader& H = *X.H;
  const uint32_t cells = H.cells, per = (uint32_t)H.n_chars * cells;
  const uint32_t inv_cells = div_inverse(cells);
  for (uint32_t e = 0; e < (uint32_t)nenv; ++e) {
    const uint16_t* st = W.dyn[e];
    const uint8_t* plane = W.plane + e * cells;
    for (uint32_t i = lane; i < per; i += 32) {
      const uint32_t k = fast_div(i, inv_cells), c = i - k * cells;
      const int z = H.z_of_char[k];
      bool v;
      if (z >= 0 && H.ent[z].kind != CX_KIND_SPRITE) {
        const CxGenEntity& en = H.ent[z];
        if (en.kind == CX_KIND_STATIC) {
          v = mask_bit(X, z, (int)c);
        } else if (en.kind == CX_KIND_ROLL) {
          const uint32_t off = st[en.dyn_slot], rcv = X.rc[c];
          int r = (int)(rcv >> 8) - (int)(off >> 8), cc = (int)(rcv & 255) - (int)(off & 255);
          if (r < 0) r += H.rows;
          if (cc < 0) cc += H.cols;
          v = mask_bit(X, z, r * H.cols + cc);
        } else {
          v = st[en.dyn_slot] == c;
        }
      } else {
        v = backdrop_at(X, st, plane, (int)c) == H.chars[k];
        if (z >= 0 && visible_now(H, st, z) && st[H.ent[z].dyn_slot] == c) v = true;
      }
      dst[e * per + i] = v ? 1 : 0;
    }
  }
}

// Whole step-end composition of a warp's envs.  `fast`: bitset composer with 16-byte stores; otherwise the
// per-cell painter's algorithm with byte stores (any geometry, any alignment).
template <int U>
__device__ __forceinline__ void compose_warp(const Ctx& X, const WarpMem& W, int nenv, uint8_t* dst, bool fast,
                                             int lane) {
  const CxGenHeader& H = *X.H;
  if (fast && H.direct) {
    const bool pokes = H.n_poke > 0;  // warp-uniform
    uint64_t saved = 0;
    if (pokes) {
      if (lane < nenv) saved = poke_below(X, W, lane);
      __syncwarp();
    }
    compose_direct<U>(X, W, nenv, dst, lane);
    if (H.n_above > 0) {
      __syncwarp();  // orders the chunk stores before the byte stores of other lanes to the same addresses
      if (lane < nenv) store_above(X, W, lane, dst);
    }
    if (pokes) {
      __syncwarp();
      if (lane < nenv) unpoke_points(X, W, lane, saved);
    }
  } else if (fast) {
    build_linear_masks(X, W, nenv, lane);
    __syncwarp();
    uint64_t saved = 0;
    if (lane < nenv) saved = poke_points(X, W, lane);
    __syncwarp();
    compose_stream(X, W, nenv, dst, lane);
    __syncwarp();
    if (lane < nenv) unpoke_points(X, W, lane, saved);
  } else {
    const int cells = H.cells;
    const uint32_t inv_cells = div_inverse((uint32_t)cells);
    for (int b = lane; b < nenv * cells; b += 32) {
      const int e = (int)fast_div((uint32_t)b, inv_cells), cell = b - e * cells;
      dst[b] = overlay(X, W.dyn[e], cell, backdrop_at(X, W.dyn[e], W.plane + e * cells, cell));
    }
  }
  __syncwarp();
}

// dynamic shared memory: [tables blob][per warp: plane tile (16-byte multiple) | per-env mask bitsets | entity
// state u16 [G][CX_MAX_DYN] | its snapshot at the last render (only games that consult it)]
__device__ __host__ __forceinline__ size_t warp_state_bytes(const CxGenHeader& H) {
  return (size_t)H.tile_envs * CX_MAX_DYN * 2 * (H.needs_prev || !H.simple_step ? 2 : 1);
}
__device__ __host__ __forceinline__ size_t warp_mem_bytes(const CxGenHeader& H) {
  const size_t tile = ((size_t)H.tile_envs * H.cells + 15) / 16 * 16;
  const size_t lin = ((size_t)H.tile_envs * H.n_lin * (H.mask_words + 1) * 4 + 15) / 16 * 16;
  return tile + lin + (warp_state_bytes(H) + 15) / 16 * 16;
}

__device__ __forceinline__ WarpMem warp_mem(const CxGenHeader& H, uint8_t* smem, int warp, int lane) {
  WarpMem W;
  const size_t tile = ((size_t)H.tile_envs * H.cells + 15) / 16 * 16;
  const size_t lin = ((size_t)H.tile_envs * H.n_lin * (H.mask_words + 1) * 4 + 15) / 16 * 16;
  W.plane = smem + H.blob_bytes + (size_t)warp * warp_mem_bytes(H);
  W.lin = reinterpret_cast<uint32_t*>(W.plane + tile);
  W.dyn = reinterpret_cast<uint16_t (*)[CX_MAX_DYN]>(W.plane + tile + lin);
  W.prev = W.dyn + H.tile_envs;  // only dereferenced by generic_env_step (space reserved when it can run)
  const int nwords = H.tile_envs * H.n_lin * (H.mask_words + 1);
  for (int i = lane; i < nwords; i += 32) W.lin[i] = 0u;  // incl. the slack word behind every bitset
  return W;
}

template <bool FAST, int BLK, int OCC>
__global__ void __launch_bounds__(BLK, OCC) k_generic_rollout(const __grid_constant__ GenParams P) {
  extern __shared__ __align__(16) uint8_t smem[];
  __shared__ uint8_t s_chidx[256];
  __shared__ uint4 s_act[CX_MAX_ACTIONS];
  const CxGenHeader& H = P.h;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, wpc = blockDim.x >> 5;
  const int G = H.tile_envs, cells = H.cells;
  stage_tables(P, smem, s_chidx, s_act);
  Ctx X;
  setup_ctx(X, P, smem, s_chidx, s_act);
  __syncthreads();  // tables staged; warps are independent from here on

  const int64_t env0 = ((int64_t)blockIdx.x * wpc + warp) * G;
  if (env0 >= P.n) return;
  const int nenv = (int)min((int64_t)G, P.n - env0);
  const WarpMem W = warp_mem(H, smem, warp, lane);
  uint8_t* plane = W.plane;
  uint16_t (*dyn)[CX_MAX_DYN] = W.dyn;
  const bool fast = P.vec && H.fast_compose;
  const bool mine = lane < nenv;
  const int64_t env = env0 + lane;
  uint32_t ts = 0;
  float rt = 0.0f;
  if (mine) {
    for (int d = 0; d < H.n_dyn; ++d) dyn[lane][d] = P.dyn[(int64_t)d * P.n + env];
    if (H.track) {
      ts = P.tstep[env];
      rt = P.ret[env];
    }
  }
  // backdrop plane of the tile: per-env plane from HBM (quirk Q1 games) or the static scenery
  if (H.has_dynbd && P.vec) {
    const uint4* s16 = reinterpret_cast<const uint4*>(P.dynbd + env0 * cells);
    uint4* d16 = reinterpret_cast<uint4*>(plane);
    for (int k = lane; k < nenv * cells / 16; k += 32) d16[k] = s16[k];
  } else {
    const uint32_t inv_cells = div_inverse((uint32_t)cells);
    for (int b = lane; b < nenv * cells; b += 32) {
      const int e = (int)fast_div((uint32_t)b, inv_cells);
      plane[b] = H.has_dynbd ? P.dynbd[env0 * cells + b] : X.backdrop[b - e * cells];
    }
  }
  __syncwarp();
  uint32_t sreg[CX_MAX_DYN];
  if (FAST && mine) fast_load_state(X, dyn[lane], sreg);

  LaneStats stats;
  stats.clear();
  const uint32_t max_steps = H.max_steps > 0 ? (uint32_t)H.max_steps : 0xFFFFFFFFu;

  uint32_t a_next = 0;  // this lane's action for the coming step, loaded one step ahead of its use
  if (mine && !P.synth) a_next = P.actions[env0 + lane];
  for (int t = 0; t < P.T; ++t) {
    const int64_t row = (int64_t)t * P.n + env0;
    bool reset_me = false;
    if (mine) {
      uint32_t a;
      if (P.synth) {
        a = cx_synth_action(P.seed, P.env_offset + (uint64_t)env, P.t0 + (uint64_t)t, (uint32_t)H.n_actions);
        if (P.actions_out) P.actions_out[row + lane] = (uint8_t)a;
      } else {
        a = a_next;
        if (t + 1 < P.T) a_next = P.actions[row + P.n + lane];
      }
      float rw, dc;
      uint32_t f;
      if (H.track && (ts & CX_OVER_BIT)) {
        rw = 0.0f;
        dc = 0.0f;
        f = CX_FROZEN_FLAGS;
      } else {
        if (FAST)
          fast_env_step(X, a, sreg, dyn[lane], plane + lane * cells, rw, f, dc);
        else if (H.simple_step)
          simple_env_step(X, a, dyn[lane], plane + lane * cells, rw, f, dc);
        else
          generic_env_step(X, a, dyn[lane], W.prev[lane], plane + lane * cells, rw, f, dc);
      }
      // a restarting env's state is reset after this step's (terminal) board has been composed
      if (H.track) reset_me = cx_episode_step(f, rw, ts, rt, stats, max_steps, H.auto_reset);
      P.reward[row + lane] = rw;
      if (P.discount) P.discount[row + lane] = dc;
      P.flags[row + lane] = (uint8_t)f;
    }
    __syncwarp();  // entity state and backdrop stamps of the warp's envs are visible

    // ---- phases 1b, 1c, 2: compose the boards and stream them out ----
    compose_warp<OCC >= 6 ? 3 : kFlatUnroll>(X, W, nenv, P.board + row * cells, fast, lane);
    if (P.layered) {  // unoccluded layers of this frame, before any auto reset touches the state
      emit_unoccluded_layers(X, W, nenv, P.layered + row * (int64_t)H.n_chars * cells, lane);
      __syncwarp();
    }

    // ---- auto reset: back to the its_showtime state (fresh make_game(), actor_critic.py:146) ----
    uint32_t rmask = __ballot_sync(0xffffffffu, reset_me);
    if (rmask) {
      if (reset_me) {
        for (int d = 0; d < H.n_dyn; ++d) dyn[lane][d] = H.slot_init[d];
        if (FAST) fast_load_state(X, dyn[lane], sreg);
      }
      if (H.has_dynbd) {
        while (rmask) {  // the plane of each finished env goes back to the its_showtime backdrop
          const int e = __ffs(rmask) - 1;
          rmask &= rmask - 1;
          uint8_t* pl = plane + e * cells;
          if ((cells & 3) == 0) {
            const uint32_t* s32 = reinterpret_cast<const uint32_t*>(X.backdrop);
            uint32_t* d32 = reinterpret_cast<uint32_t*>(pl);
            for (int b = lane; b < cells / 4; b += 32) d32[b] = s32[b];
          } else {
            for (int b = lane; b < cells; b += 32) pl[b] = X.backdrop[b];
          }
        }
      }
    }
    __syncwarp();
  }

  if (mine) {
    for (int d = 0; d < H.n_dyn; ++d) P.dyn[(int64_t)d * P.n + env] = dyn[lane][d];
    if (H.track) {
      P.tstep[env] = (uint16_t)ts;
      P.ret[env] = rt;
    }
  }
  if (H.has_dynbd) {
    if (P.vec) {
      const uint4* s16 = reinterpret_cast<const uint4*>(plane);
      uint4* d16 = reinterpret_cast<uint4*>(P.dynbd + env0 * cells);
      for (int k = lane; k < nenv * cells / 16; k += 32) d16[k] = s16[k];
    } else {
      for (int b = lane; b < nenv * cells; b += 32) P.dynbd[env0 * cells + b] = plane[b];
    }
  }
  if (H.track) cx_flush_stats(stats, P.stats, (uint32_t)(blockIdx.x * wpc + warp), (uint32_t)nenv, P.T);
}

// Render the current state of every env (first frame after its_showtime / reset).
__global__ void __launch_bounds__(NT) k_generic_render(const __grid_constant__ GenParams P) {
  extern __shared__ __align__(16) uint8_t smem[];
  __shared__ uint8_t s_chidx[256];
  __shared__ uint4 s_act[CX_MAX_ACTIONS];
  const CxGenHeader& H = P.h;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, wpc = blockDim.x >> 5;
  const int G = H.tile_envs, cells = H.cells;
  stage_tables(P, smem, s_chidx, s_act);
  Ctx X;
  setup_ctx(X, P, smem, s_chidx, s_act);
  __syncthreads();
  const int64_t env0 = ((int64_t)blockIdx.x * wpc + warp) * G;
  if (env0 >= P.n) return;
  const int nenv = (int)min((int64_t)G, P.n - env0);
  const WarpMem W = warp_mem(H, smem, warp, lane);
  if (lane < nenv)
    for (int d = 0; d < H.n_dyn; ++d) W.dyn[lane][d] = P.dyn[(int64_t)d * P.n + env0 + lane];
  const uint32_t inv_cells = div_inverse((uint32_t)cells);
  for (int b = lane; b < nenv * cells; b += 32) {
    const int e = (int)fast_div((uint32_t)b, inv_cells);
    W.plane[b] = H.has_dynbd ? P.dynbd[env0 * cells + b] : X.backdrop[b - e * cells];
  }
  __syncwarp();
  compose_warp<kFlatUnroll>(X, W, nenv, P.board + env0 * cells, P.vec && H.fast_compose, lane);
  if (P.layered) emit_unoccluded_layers(X, W, nenv, P.layered + env0 * (int64_t)H.n_chars * cells, lane);
}

GenParams make_params(const cx_game* g, void* d_state, int64_t n) {
  const CxStateLayout L = cx_layout(g, n);
  uint8_t* base = static_cast<uint8_t*>(d_state);
  GenParams P;
  memset(&P, 0, sizeof(P));
  P.h = g->gh;
  P.blob = g->d_blob;
  P.dyn = reinterpret_cast<uint16_t*>(base + L.off_dyn);
  P.tstep = reinterpret_cast<uint16_t*>(base + L.off_tstep);
  P.ret = reinterpret_cast<float*>(base + L.off_ret);
  P.dynbd = base + L.off_dynbd;
  P.stats = reinterpret_cast<double*>(base + L.off_stats);
  P.n = n;
  return P;
}

size_t gen_warp_bytes(const cx_game* g) { return warp_mem_bytes(g->gh); }
// warps per CTA: share the staged tables between warps while keeping a CTA below ~100 KB of shared memory
int gen_warps_per_cta(const cx_game* g) {
  int w = NT / 32;
  while (w > 1 && (size_t)g->gh.blob_bytes + (size_t)w * gen_warp_bytes(g) > 100 * 1024) w >>= 1;
  return w;
}
size_t gen_smem_bytes(const cx_game* g, int wpc) {
  return (size_t)g->gh.blob_bytes + (size_t)wpc * gen_warp_bytes(g);
}
// 16-byte chunks: every tile and every [T, n] board row starts 16-byte aligned and holds whole chunks
bool gen_vec_ok(const cx_game* g, int64_t n, const void* d_board) {
  const int G = g->gh.tile_envs;
  return ((int64_t)G * g->gh.cells % 16 == 0) && (n % G == 0) && ((n * g->gh.cells) % 16 == 0) &&
         (reinterpret_cast<uintptr_t>(d_board) & 15) == 0;
}

int configure_once() {
  static CxPerDevice configured;
  if (configured.need()) {
    CX_CUDA_OK(cudaFuncSetAttribute(k_generic_rollout<false, NT, kMinCtas>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    CX_CUDA_OK(cudaFuncSetAttribute(k_generic_rollout<true, NT, kMinCtas>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    CX_CUDA_OK(cudaFuncSetAttribute(k_generic_rollout<true, NT, kMinCtas + 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    CX_CUDA_OK(cudaFuncSetAttribute(k_generic_rollout<true, kWaveThreads, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    // two 112 KB CTAs per SM need the largest shared-memory carveout (a hint the driver would otherwise derive per launch)
    CX_CUDA_OK(cudaFuncSetAttribute(k_generic_rollout<true, kWaveThreads, 2>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                    (int)cudaSharedmemCarveoutMaxShared));
    CX_CUDA_OK(cudaFuncSetAttribute(k_generic_render, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    configured.mark();
  }
  return CX_OK;
}

}  // namespace

int cx_launch_generic_rollout(const cx_game* g, void* d_state, int64_t n, int32_t T, const uint8_t* d_actions,
                              const CxSynth& synth, float* d_reward, float* d_discount, uint8_t* d_flags,
                              uint8_t* d_board, CxRoute route, cudaStream_t s, uint8_t* d_layered) {
  GenParams P = make_params(g, d_state, n);
  P.actions = d_actions;
  P.synth = synth.on;
  P.seed = synth.seed;
  P.env_offset = synth.env_offset;
  P.t0 = synth.t0;
  P.actions_out = synth.actions_out;
  P.reward = d_reward;
  P.discount = d_discount;
  P.flags = d_flags;
  P.board = d_board;
  P.layered = d_layered;
  P.T = T;
  const int G = g->gh.tile_envs;
  P.vec = gen_vec_ok(g, n, d_board);
  const int wpc = gen_warps_per_cta(g);
  const int64_t warps = (n + G - 1) / G;
  const int64_t grid = (warps + wpc - 1) / wpc;
  if (grid > 0x7fffffff) {
    cx_set_error("cx_rollout: too many environments for one launch");
    return CX_ERR_INVALID_ARG;
  }
  int rc = configure_once();
  if (rc) return rc;
  if (g->gh.fast_loop && P.vec) {
    // Three builds of the register-state kernel, chosen by how the batch fills the machine:
    //  * a batch that needs slightly more warps per SM than 4-warp CTAs keep resident (Hello World, 65,536 envs: 27.7
    //    against 20-24) would run 1.2-1.4 waves; two fat CTAs per SM (up to 14 warps each, 72 registers) hold it in
    //    ONE wave instead;
    //  * kMinCtas + 1 resident CTAs per SM (80 registers) once the grid is at least two waves deep;
    //  * kMinCtas CTAs (96 registers) otherwise.
    // The routes gen96 / gen80 / gen_wave force the 96-register, the 80-register and the one-wave build (the latter with
    // 14-warp CTAs, as far as they fit shared memory).
    const int64_t per_sm = (warps + g->sm_count - 1) / g->sm_count;
    int fat = (int)((per_sm + 1) / 2);  // warps per CTA with two CTAs per SM
    if (route == CX_ROUTE_GEN_WAVE) fat = kWaveThreads / 32;
    const bool auto_build = route != CX_ROUTE_GEN96 && route != CX_ROUTE_GEN80 && route != CX_ROUTE_GEN_WAVE;
    if ((route == CX_ROUTE_GEN_WAVE || (auto_build && per_sm > (int64_t)wpc * kMinCtas)) && fat * 32 <= kWaveThreads &&
        2 * (gen_smem_bytes(g, fat) + 1024 + 512) <= (size_t)g->smem_per_sm) {
      const int64_t fgrid = (warps + fat - 1) / fat;
      k_generic_rollout<true, kWaveThreads, 2><<<(unsigned)fgrid, fat * 32, gen_smem_bytes(g, fat), s>>>(P);
    } else if (route == CX_ROUTE_GEN80 ||
               (route != CX_ROUTE_GEN96 && grid >= 2 * (int64_t)g->sm_count * (kMinCtas + 1))) {
      k_generic_rollout<true, NT, kMinCtas + 1><<<(unsigned)grid, wpc * 32, gen_smem_bytes(g, wpc), s>>>(P);
    } else {
      k_generic_rollout<true, NT, kMinCtas><<<(unsigned)grid, wpc * 32, gen_smem_bytes(g, wpc), s>>>(P);
    }
  }
  else
    k_generic_rollout<false, NT, kMinCtas><<<(unsigned)grid, wpc * 32, gen_smem_bytes(g, wpc), s>>>(P);
  CX_CUDA_OK(cudaGetLastError());
  return CX_OK;
}

int cx_launch_generic_render(const cx_game* g, const void* d_state, int64_t n, uint8_t* d_board, cudaStream_t s,
                             uint8_t* d_layered) {
  GenParams P = make_params(g, const_cast<void*>(d_state), n);
  P.board = d_board;
  P.layered = d_layered;
  P.vec = gen_vec_ok(g, n, d_board);
  const int G = g->gh.tile_envs;
  const int wpc = gen_warps_per_cta(g);
  const int64_t warps = (n + G - 1) / G;
  const int64_t grid = (warps + wpc - 1) / wpc;
  int rc = configure_once();
  if (rc) return rc;
  k_generic_render<<<(unsigned)grid, wpc * 32, gen_smem_bytes(g, wpc), s>>>(P);
  CX_CUDA_OK(cudaGetLastError());
  return CX_OK;
}
