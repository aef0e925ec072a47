// Host side of libcampx_b200.so: the native back end of the game compiler.
//
// cx_game_create() takes the primitive-level game description produced by the Python front end at
// Engine.its_showtime() (campx_b200/compiler) and lowers it to the device tables the kernels consume:
// z-ordered static composition (engine.py:295-324), toroidal move tables (boat_race.py:42-49), wall /
// blocker masks (boat_race.py:52-56), first-entry reward tables summed in update order with float32
// arithmetic exactly as Plot.add_reward does (plot.py:186-211, boat_race.py:76-90), and the per-action
// engine directives (plot.py:161-257; engine.py:285-290).
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "cx_internal.cuh"

static thread_local char g_err[512] = "";

void cx_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

extern "C" const char* cx_last_error(void) { return g_err; }
extern "C" int cx_abi_version(void) { return CX_ABI_VERSION; }
extern "C" int cx_abi_sizeof(int which) {
  switch (which) {
    case 0: return (int)sizeof(cx_entity_desc);
    case 1: return (int)sizeof(cx_game_desc);
    case 2: return (int)sizeof(cx_game_info);
    default: return -1;
  }
}

static inline int64_t align_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

CxStateLayout cx_layout(const cx_game* g, int64_t n) {
  CxStateLayout L;
  memset(&L, 0, sizeof(L));
  L.n = n;
  int64_t off = 0;
  L.off_stats = off;
  off = align_up(off + (1 + CX_STAT_STRIPES) * CX_STATS_DOUBLES * (int64_t)sizeof(double), 256);
  L.off_tstep = off;
  if (g->info.tracks) off = align_up(off + n * 2, 256);
  L.off_ret = off;
  if (g->info.tracks) off = align_up(off + n * 4, 256);
  L.off_dyn = off;
  if (g->path == CX_PATH_AGENT)
    off = align_up(off + n, 256);
  else
    off = align_up(off + (int64_t)g->gh.n_dyn * n * 2, 256);
  L.off_dynbd = off;
  if (g->path == CX_PATH_GENERIC && g->gh.has_dynbd) off = align_up(off + n * (int64_t)g->gh.cells, 256);
  L.off_perf = off;   // last, so that the layout of a game without performance is what it was before
  if (g->info.tracks_performance) off = align_up(off + n * 4, 256);
  L.off_pick = off;   // behind everything else for the same reason
  if (g->info.n_pickups) off = align_up(off + n * 8, 256);
  L.total = off < 256 ? 256 : off;
  return L;
}

static int char_index(const cx_game_desc* d, int ch) {
  for (int k = 0; k < d->n_chars; ++k)
    if (d->chars[k] == ch) return k;
  return -1;
}

static int popcount_mask(const uint8_t* m, int cells, int* first) {
  int c = 0;
  *first = -1;
  for (int i = 0; i < cells; ++i)
    if (m[i]) {
      if (*first < 0) *first = i;
      ++c;
    }
  return c;
}

// plot directives per action, replayed in update order (engine.py:195-204 then :285-290)
static void build_action_table(const cx_game_desc* d, const int* order, CxActionTable* t) {
  memset(t, 0, sizeof(*t));
  for (int a = 0; a < CX_MAX_ACTIONS; ++a) {
    bool over = false, any_reward = false;
    float disc = 1.0f;  // plot.py:100
    if (a < d->n_actions) {
      for (int i = 0; i < d->n_entities; ++i) {
        const cx_entity_desc& e = d->entities[order[i]];
        if (e.kind == CX_KIND_PICKUP) continue;   // pays and terminates only when it takes an item (the kernel)
        if (e.reward_actions >> a & 1) any_reward = true;
        if (e.discount_actions >> a & 1) disc = e.discount_value[a];
        if (e.terminate_actions >> a & 1) {
          over = true;
          disc = e.discount_value[a];
        }
      }
    }
    t->over[a] = over;
    t->reward_none[a] = !any_reward;
    t->discount[a] = disc;
  }
}

static int validate(const cx_game_desc* d) {
  if (!d) {
    cx_set_error("cx_game_create: desc is NULL");
    return CX_ERR_INVALID_ARG;
  }
  if (d->abi_version != CX_ABI_VERSION) {
    cx_set_error("cx_game_create: abi_version %d, library is %d", d->abi_version, CX_ABI_VERSION);
    return CX_ERR_INVALID_ARG;
  }
  if (d->rows < 1 || d->cols < 1 || d->rows > 255 || d->cols > 255 || (int64_t)d->rows * d->cols > CX_MAX_CELLS) {
    cx_set_error("cx_game_create: board %dx%d out of range (<=255 per side, <=%d cells)", d->rows, d->cols,
                 CX_MAX_CELLS);
    return CX_ERR_INVALID_ARG;
  }
  if (d->n_chars < 1 || d->n_chars > CX_MAX_CHARS) {
    cx_set_error("cx_game_create: n_chars %d out of range 1..%d", d->n_chars, CX_MAX_CHARS);
    return CX_ERR_INVALID_ARG;
  }
  if (d->n_actions < 1 || d->n_actions > CX_MAX_ACTIONS) {
    cx_set_error("cx_game_create: n_actions %d out of range 1..%d", d->n_actions, CX_MAX_ACTIONS);
    return CX_ERR_INVALID_ARG;
  }
  if (d->n_entities < 0 || d->n_entities > CX_MAX_ENTITIES) {
    cx_set_error("cx_game_create: n_entities %d out of range 0..%d", d->n_entities, CX_MAX_ENTITIES);
    return CX_ERR_INVALID_ARG;
  }
  if (d->n_groups < 0 || d->n_groups > CX_MAX_GROUPS) {
    cx_set_error("cx_game_create: n_groups %d out of range 0..%d", d->n_groups, CX_MAX_GROUPS);
    return CX_ERR_INVALID_ARG;
  }
  if (!d->backdrop || (d->n_entities > 0 && !d->masks)) {
    cx_set_error("cx_game_create: backdrop/masks pointers are NULL");
    return CX_ERR_INVALID_ARG;
  }
  if (d->max_episode_steps < 0 || d->max_episode_steps > 32767) {
    cx_set_error("cx_game_create: max_episode_steps %d out of range 0..32767", d->max_episode_steps);
    return CX_ERR_INVALID_ARG;
  }
  if (d->n_perf_regions != 0) {
    if (d->n_perf_regions < 2 || d->n_perf_regions > 255 || !d->perf_regions) {
      cx_set_error("cx_game_create: n_perf_regions %d must be 0 or 2..255, with perf_regions given",
                   d->n_perf_regions);
      return CX_ERR_INVALID_ARG;
    }
    if (!d->track_returns) {
      cx_set_error("cx_game_create: performance is kept with the per-env episode state: set track_returns");
      return CX_ERR_INVALID_ARG;
    }
    for (int i = 0; i < d->rows * d->cols; ++i)
      if (d->perf_regions[i] > d->n_perf_regions) {
        cx_set_error("cx_game_create: perf_regions[%d] = %d exceeds n_perf_regions %d", i, d->perf_regions[i],
                     d->n_perf_regions);
        return CX_ERR_INVALID_ARG;
      }
  }
  for (int k = 1; k < d->n_chars; ++k)
    if (d->chars[k] <= d->chars[k - 1]) {
      cx_set_error("cx_game_create: chars[] must be strictly increasing (canonical channel order)");
      return CX_ERR_INVALID_ARG;
    }
  const int cells = d->rows * d->cols;
  for (int i = 0; i < cells; ++i)
    if (d->backdrop[i] != 0 && char_index(d, d->backdrop[i]) < 0) {
      cx_set_error("cx_game_create: backdrop cell %d holds character %d which is not in chars[]", i,
                   d->backdrop[i]);
      return CX_ERR_INVALID_ARG;
    }
  std::vector<int> seen_rank(d->n_entities, 0);
  for (int z = 0; z < d->n_entities; ++z) {
    const cx_entity_desc& e = d->entities[z];
    if (char_index(d, e.character) < 0) {
      cx_set_error("cx_game_create: entity %d character %d is not in chars[]", z, e.character);
      return CX_ERR_INVALID_ARG;
    }
    for (int y = 0; y < z; ++y)
      if (d->entities[y].character == e.character) {
        cx_set_error("cx_game_create: character %d used by two entities", e.character);  // engine.py:343-350
        return CX_ERR_INVALID_ARG;
      }
    if (e.kind > CX_KIND_DOOR) {
      cx_set_error("cx_game_create: entity %d has unknown kind %d", z, e.kind);
      return CX_ERR_INVALID_ARG;
    }
    if (e.kind == CX_KIND_DOOR && (e.door_key < 0 || e.door_key >= d->n_entities ||
                                   d->entities[e.door_key].kind != CX_KIND_PICKUP)) {
      cx_set_error("cx_game_create: door entity %d names z-index %d as its key, which is not a pickup drape", z,
                   e.door_key);
      return CX_ERR_INVALID_ARG;
    }
    if (e.update_rank >= d->n_entities || seen_rank[e.update_rank]++) {
      cx_set_error("cx_game_create: update_rank of entity %d is not a permutation index", z);
      return CX_ERR_INVALID_ARG;
    }
    if (e.update_group >= (d->n_groups > 0 ? d->n_groups : 1)) {
      cx_set_error("cx_game_create: entity %d update_group %d >= n_groups %d", z, e.update_group, d->n_groups);
      return CX_ERR_INVALID_ARG;
    }
    if (e.watch >= d->n_entities) {
      cx_set_error("cx_game_create: entity %d watches z-index %d which does not exist", z, e.watch);
      return CX_ERR_INVALID_ARG;
    }
    if (e.watch >= 0) {
      const int wk = d->entities[e.watch].kind;
      if (wk != CX_KIND_CELL && wk != CX_KIND_SPRITE) {
        cx_set_error("cx_game_create: entity %d watches entity %d which is not a CELL or SPRITE", z, e.watch);
        return CX_ERR_UNSUPPORTED;
      }
    }
    if (e.kind == CX_KIND_SPRITE) {
      if (e.init_row < 0 || e.init_row >= d->rows || e.init_col < 0 || e.init_col >= d->cols) {
        cx_set_error("Position (%d, %d) does not fall inside a %dx%d game board.", e.init_row, e.init_col,
                     d->rows, d->cols);  // engine.py:50-53
        return CX_ERR_INVALID_ARG;
      }
      // a blocked sprite keeps its visibility: every case of the wall gate is then "stay" or "move"
      for (int a = 0; a < d->n_actions && e.blockers; ++a)
        if (e.visible_op[a] != CX_VIS_KEEP) {
          cx_set_error("cx_game_create: sprite %d has blockers and changes its visibility (action %d); a blocked "
                       "sprite must keep it", z, a);
          return CX_ERR_UNSUPPORTED;
        }
    }
    if (e.kind == CX_KIND_PICKUP && e.terminate_emptied && !(e.emptied_value >= 0.0f && e.emptied_value <= 1.0f)) {
      cx_set_error("Pcontinue must be in range [0,1]");  // plot.py:176-177
      return CX_ERR_INVALID_ARG;
    }
    if (e.kind == CX_KIND_CELL) {
      int first;
      if (popcount_mask(d->masks + (size_t)z * cells, cells, &first) > 1) {
        cx_set_error("cx_game_create: CELL entity %d has more than one mask cell", z);
        return CX_ERR_UNSUPPORTED;
      }
    }
    for (int a = 0; a < d->n_actions; ++a) {
      if (e.visible_op[a] > CX_VIS_TOGGLE || (e.visible_op[a] != CX_VIS_KEEP && e.kind != CX_KIND_SPRITE)) {
        cx_set_error("cx_game_create: entity %d action %d has visible_op %d (sprites only, 0..3)", z, a,
                     e.visible_op[a]);
        return CX_ERR_INVALID_ARG;
      }
      if (e.n_zdirs[a] > CX_MAX_ZDIRS) {
        cx_set_error("cx_game_create: entity %d action %d has %d z-order directives (max %d)", z, a, e.n_zdirs[a],
                     CX_MAX_ZDIRS);
        return CX_ERR_INVALID_ARG;
      }
      for (int k = 0; k < e.n_zdirs[a]; ++k) {
        const int mv = e.z_move[a][k], fr = e.z_front[a][k];
        if (mv < 0 || mv >= d->n_entities || fr < -1 || fr >= d->n_entities) {
          // engine.py:247-262: "A z-order change directive said to move a Sprite or Drape ... no such ... exists"
          cx_set_error("cx_game_create: z-order directive of entity %d names an entity that does not exist", z);
          return CX_ERR_INVALID_ARG;
        }
        if (mv == fr) {  // engine.py:270-279 would drop the entity from the game altogether
          cx_set_error("cx_game_create: z-order directive moves entity %d in front of itself", mv);
          return CX_ERR_UNSUPPORTED;
        }
      }
      if (abs((int)e.move_dr[a]) >= d->rows + (d->rows == 1) || abs((int)e.move_dc[a]) >= d->cols + (d->cols == 1)) {
        cx_set_error("cx_game_create: entity %d action %d moves by (%d, %d), not less than the board size", z, a,
                     e.move_dr[a], e.move_dc[a]);
        return CX_ERR_INVALID_ARG;
      }
      if (e.terminate_chars[a]) {
        if (e.watch < 0) {
          cx_set_error("cx_game_create: entity %d has terminate_chars but watches no entity", z);
          return CX_ERR_INVALID_ARG;
        }
        if (!(e.terminate_value[a] >= 0.0f && e.terminate_value[a] <= 1.0f)) {
          cx_set_error("Pcontinue must be in range [0,1]");  // plot.py:176-177
          return CX_ERR_INVALID_ARG;
        }
      }
      const float dv = e.discount_value[a];
      if (((e.terminate_actions | e.discount_actions) >> a & 1) && !(dv >= 0.0f && dv <= 1.0f)) {
        cx_set_error("Pcontinue must be in range [0,1]");  // plot.py:176-177,250-251
        return CX_ERR_INVALID_ARG;
      }
    }
  }
  for (int a = 0; a < d->n_actions; ++a)
    if (abs((int)d->backdrop_dr[a]) >= d->rows + (d->rows == 1) || abs((int)d->backdrop_dc[a]) >= d->cols + (d->cols == 1)) {
      cx_set_error("cx_game_create: action %d rolls the backdrop by (%d, %d), not less than the board size", a,
                   d->backdrop_dr[a], d->backdrop_dc[a]);
      return CX_ERR_INVALID_ARG;
    }
  // update groups must be ordered consistently with ranks (engine.py:520-521 sorts groups; ranks follow)
  for (int z = 0; z < d->n_entities; ++z)
    for (int y = 0; y < d->n_entities; ++y)
      if (d->entities[z].update_rank < d->entities[y].update_rank &&
          d->entities[z].update_group > d->entities[y].update_group) {
        cx_set_error("cx_game_create: update ranks are not grouped by update_group");
        return CX_ERR_INVALID_ARG;
      }
  return CX_OK;
}

struct Blob {
  std::vector<uint8_t> bytes;
  int32_t reserve(size_t n) {
    size_t off = (bytes.size() + 15) / 16 * 16;
    bytes.resize(off + n, 0);
    return (int32_t)off;
  }
  void pad() { bytes.resize((bytes.size() + 15) / 16 * 16, 0); }
};

// z-order directives, sprite visibility directives or a rolling backdrop: render state that changes during play
static void dynamic_render_needs(const cx_game_desc* d, bool* vis, bool* zord, bool* bd) {
  *vis = *zord = *bd = false;
  for (int a = 0; a < d->n_actions; ++a) {
    if (d->backdrop_dr[a] || d->backdrop_dc[a]) *bd = true;
    for (int z = 0; z < d->n_entities; ++z) {
      if (d->entities[z].visible_op[a] != CX_VIS_KEEP) *vis = true;
      if (d->entities[z].n_zdirs[a]) *zord = true;
    }
  }
}

// One mover over a static scene: a one-cell drape, or a visible sprite behind at least one drape in z-order (it then
// neither stamps the backdrop, quirk Q1, nor has its canvas zeroed, and the tables' "drawn cell" is its painted cell).
static bool agent_path_applies(const cx_game_desc* d, int* agent_z) {
  const int cells = d->rows * d->cols;
  if (cells > CX_AGENT_MAX_CELLS || d->n_groups > 1) return false;
  bool vis, zord, bd;
  dynamic_render_needs(d, &vis, &zord, &bd);
  if (vis || zord || bd) return false;
  int moving = -1, count = 0;
  for (int z = 0; z < d->n_entities; ++z) {
    const cx_entity_desc& e = d->entities[z];
    if (e.kind == CX_KIND_ROLL) return false;
    if (e.kind == CX_KIND_SPRITE && (!e.visible || z == 0)) return false;
    if (e.kind == CX_KIND_CELL || e.kind == CX_KIND_SPRITE) {
      moving = z;
      ++count;
    }
  }
  if (count != 1) return false;
  for (int z = 0; z < d->n_entities; ++z)
    if (d->entities[z].watch >= 0 && d->entities[z].watch != moving) return false;
  *agent_z = moving;
  return true;
}

// One Engine.play() of a single-agent game for agent cell p (cells == empty mask) and action a, on the
// host: examples/boat_race.py:40-59 (move + wall gate against the last render), :76-90 (entry rewards of
// every entity, summed in update order with float32 arithmetic as plot.py:208-211 does).  A sprite agent
// (PyColab's MazeWalker) stays at p when blocked, whether or not the last render showed it there.
struct AgentStep {
  int q;          // new cell (cells: empty)
  float reward;
  bool over;      // the_plot.terminate_episode() was called (plot.py:161-184)
  float discount; // discount returned with the step (engine.py:285-290)
};

static AgentStep agent_step_host(const cx_game_desc* d, int agent_z, const int* order, const uint8_t* basech,
                                 const uint8_t* vis, int a, int p) {
  const int R = d->rows, C = d->cols, cells = R * C, L = d->n_chars;
  const cx_entity_desc& ag = d->entities[agent_z];
  const int agent_idx = char_index(d, ag.character);
  auto idx_of = [&](int ch) { return ch == 0 ? L : char_index(d, ch); };
  int ko = L, kn = L, q = p;  // L == "no cell"
  if (p < cells) {
    const bool visp = vis[p] != 0;                 // the agent was visible in the last render
    const int r = p / C, c = p % C;
    const int t = (((r + ag.move_dr[a]) % R + R) % R) * C + ((c + ag.move_dc[a]) % C + C) % C;
    const bool onto_self = (t == p) && visp;       // the last render showed the agent itself there
    const int seen_t = onto_self ? agent_idx : idx_of(basech[t]);
    const bool blocked = seen_t < L && ((ag.blockers >> seen_t) & 1u);
    ko = visp ? agent_idx : idx_of(basech[p]);
    if (blocked) {                                 // b = prev_pos: the agent layer of the last render,
      if (ag.kind == CX_KIND_SPRITE) {             // empty when the agent was occluded (boat_race.py:55-56);
        kn = ko;                                   // a sprite keeps its position
      } else if (visp) {
        kn = agent_idx;
      } else {
        q = cells;
      }
    } else {
      q = t;
      kn = seen_t;
    }
  }
  bool first_add = true;
  float summed = 0.0f;
  for (int i = 0; i < d->n_entities; ++i) {
    const cx_entity_desc& e = d->entities[order[i]];
    if (!(e.reward_actions >> a & 1) || e.kind == CX_KIND_PICKUP) continue;
    volatile float rr = e.step_reward[a];
    if (e.watch == agent_z) {
      const int k = (e.update_rank >= ag.update_rank) ? kn : ko;  // things['A'] is current sibling state
      if (k < L) rr = rr + e.entry_reward[a][k];
    }
    if (first_add) {
      summed = rr;
      first_add = false;
    } else {
      volatile float s2 = rr + summed;  // plot.py:211: reward + running sum
      summed = s2;
    }
  }
  // plot directives in update order: the last change_default_discount / terminate_episode call wins
  bool over = false;
  float disc = 1.0f;  // plot.py:100
  for (int i = 0; i < d->n_entities; ++i) {
    const cx_entity_desc& e = d->entities[order[i]];
    if (e.kind == CX_KIND_PICKUP) continue;
    if (e.discount_actions >> a & 1) disc = e.discount_value[a];
    if (e.terminate_actions >> a & 1) {
      over = true;
      disc = e.discount_value[a];
    }
    if (e.terminate_chars[a] && e.watch == agent_z) {
      const int k = (e.update_rank >= ag.update_rank) ? kn : ko;
      if (k < L && ((e.terminate_chars[a] >> k) & 1u)) {
        over = true;
        disc = e.terminate_value[a];
      }
    }
  }
  AgentStep out;
  out.q = q;
  out.reward = summed;
  out.over = over;
  out.discount = disc;
  return out;
}

// Static composition without the agent (painter's algorithm, engine.py:306-321) and where the agent is visible; pickup
// drapes with all their items (items_present) or none; door drapes closed but for the open ones (bit d: the d-th door
// in z-order is open).
static void compose_static(const cx_game_desc* d, int agent_z, bool items_present, std::vector<uint8_t>* basech,
                           std::vector<uint8_t>* vis, uint32_t doors_open = 0) {
  const int cells = d->rows * d->cols;
  basech->assign(cells + 1, 0);
  vis->assign(cells + 1, 0);
  for (int c = 0; c < cells; ++c) {
    (*basech)[c] = d->backdrop[c];
    (*vis)[c] = 1;
  }
  int door = 0;
  for (int z = 0; z < d->n_entities; ++z) {
    if (d->entities[z].kind == CX_KIND_DOOR && ((doors_open >> door++) & 1)) continue;
    if (z == agent_z || (d->entities[z].kind == CX_KIND_PICKUP && !items_present)) continue;
    const uint8_t* m = d->masks + (size_t)z * cells;
    for (int c = 0; c < cells; ++c)
      if (m[c]) {
        (*basech)[c] = d->entities[z].character;
        if (z > agent_z) (*vis)[c] = 0;  // painted after (in front of) the agent
      }
  }
}

// Nothing but the pickups' own reward and termination may depend on an item's presence: one Engine.play() from every
// cell under every action must not change when all items are put back (`absent` -> `present`, same doors).
static int check_items_irrelevant(const cx_game_desc* d, int agent_z, const int* order, const std::vector<uint8_t>& absent,
                                  const std::vector<uint8_t>& present, const std::vector<uint8_t>& vis) {
  const int cells = d->rows * d->cols;
  for (int p = 0; p < cells; ++p) {
    for (int a = 0; a < d->n_actions; ++a) {
      const AgentStep x = agent_step_host(d, agent_z, order, absent.data(), vis.data(), a, p);
      const AgentStep y = agent_step_host(d, agent_z, order, present.data(), vis.data(), a, p);
      if (x.q != y.q || memcmp(&x.reward, &y.reward, 4) || x.over != y.over || memcmp(&x.discount, &y.discount, 4)) {
        cx_set_error("cx_game_create: the step from cell %d under action %d depends on whether an item is present "
                     "(an item or the character under it is a blocker, an entry-reward or a terminate character of "
                     "another entity); only the pickup drape's own reward and termination may", p, a);
        return CX_ERR_UNSUPPORTED;
      }
    }
  }
  return CX_OK;
}

// The transition tables (CxAgentHeader::off_tt / off_tr / off_td layout) of the static scene `absent`, agent visible
// where `vis` says.
static void fill_step_tables(const cx_game_desc* d, int agent_z, const int* order, const CxAgentHeader& H,
                             const std::vector<uint8_t>& absent, const std::vector<uint8_t>& vis, uint32_t* tt,
                             float* tr, float* td) {
  const int cells = d->rows * d->cols, A = d->n_actions, S = cells + 1;
  for (int a = 0; a <= A; ++a) {
    if (!H.td_per_cell) td[a] = a < A ? H.act.discount[a] : 1.0f;
    for (int p = 0; p <= cells; ++p) {
      int q = p;
      float reward = 0.0f, disc = 1.0f;
      uint32_t flags = CX_FLAG_BAD_ACTION | CX_FLAG_REWARD_NONE;  // row A: env left untouched
      if (a < A) {
        const AgentStep st = agent_step_host(d, agent_z, order, absent.data(), vis.data(), a, p);
        q = st.q;
        reward = st.reward;
        disc = st.discount;
        flags = (st.over ? CX_FLAG_TERMINATED : 0) | (H.act.reward_none[a] ? CX_FLAG_REWARD_NONE : 0);
      }
      if (H.td_per_cell) td[a * S + p] = disc;
      const int shown = (q < cells && vis[q]) ? q : cells;
      // the step's performance rides in the spare top byte: no table, no load of its own (row A and the empty
      // mask: 0)
      int perf = 0;
      if (d->n_perf_regions && a < A && p < cells && q < cells)
        perf = cx_perf_step(d->perf_regions[p], d->perf_regions[q], d->n_perf_regions);
      tt[a * S + p] = (uint32_t)q | ((uint32_t)shown << 8) | (flags << 16) | ((uint32_t)(uint8_t)(int8_t)perf << 24);
      tr[a * S + p] = reward;
    }
  }
}

static int build_agent_tables(const cx_game_desc* d, int agent_z, const int* order, CxAgentHeader* H, Blob* B) {
  const int R = d->rows, C = d->cols, cells = R * C, A = d->n_actions;
  const cx_entity_desc& ag = d->entities[agent_z];
  memset(H, 0, sizeof(*H));
  H->cells = cells;
  H->n_actions = A;
  H->n_chars = d->n_chars;
  H->agent_char = ag.character;
  H->stride = cells + 1;
  int first;
  popcount_mask(d->masks + (size_t)agent_z * cells, cells, &first);
  if (ag.kind == CX_KIND_SPRITE) first = ag.init_row * C + ag.init_col;
  H->init_cell = first < 0 ? cells : first;
  H->max_steps = d->max_episode_steps;
  H->auto_reset = d->auto_reset;
  build_action_table(d, order, &H->act);

  // The step tables are lowered with every item absent, the scene (basech and what derives from it) shows every item
  // present.  Games without pickups: the two are the same.  Doors: closed (the tables of the other door states are
  // build_pick_tables').
  std::vector<uint8_t> absent, vis, basech, unused;
  compose_static(d, agent_z, false, &absent, &vis);
  compose_static(d, agent_z, true, &basech, &unused);   // (pickups in front of the agent: build_pick_tables refuses)
  int rc = check_items_irrelevant(d, agent_z, order, absent, basech, vis);
  if (rc != CX_OK) return rc;
  const int S = cells + 1;
  for (int z = 0; z < d->n_entities; ++z)
    for (int a = 0; a < A; ++a)
      if (d->entities[z].terminate_chars[a]) H->td_per_cell = 1;
  H->off_tt = B->reserve((size_t)(A + 1) * S * 4);
  H->off_tr = B->reserve((size_t)(A + 1) * S * 4);
  H->off_td = B->reserve((size_t)(A + 1) * (H->td_per_cell ? S : 1) * 4);
  fill_step_tables(d, agent_z, order, *H, absent, vis, (uint32_t*)&B->bytes[H->off_tt], (float*)&B->bytes[H->off_tr],
                   (float*)&B->bytes[H->off_td]);
  H->off_basech = B->reserve(S);
  memcpy(&B->bytes[H->off_basech], basech.data(), S);
  H->off_shown = B->reserve(S);
  for (int c = 0; c <= cells; ++c) B->bytes[H->off_shown + c] = (uint8_t)((c < cells && vis[c]) ? c : cells);
  H->off_pat = B->reserve((size_t)cells * 16);
  for (int o = 0; o < cells; ++o)
    for (int j = 0; j < 16; ++j) B->bytes[H->off_pat + o * 16 + j] = basech[(o + j) % cells];
  B->pad();
  H->blob_bytes = (int32_t)B->bytes.size();
  // extension for the observation kernel: which layered-board channel each static cell belongs to
  const int L = d->n_chars;
  H->agent_k = char_index(d, ag.character);
  H->off_basek = B->reserve(S);
  for (int c = 0; c <= cells; ++c) {
    const int k = c < cells ? char_index(d, basech[c]) : -1;
    B->bytes[H->off_basek + c] = (uint8_t)(k < 0 ? 0xFF : k);
  }
  H->off_baselay = B->reserve((size_t)L * cells);
  H->unoccluded = d->unoccluded_layers ? 1 : 0;
  if (!H->unoccluded) {
    for (int c = 0; c < cells; ++c) {
      const int k = char_index(d, basech[c]);
      if (k >= 0) B->bytes[H->off_baselay + (size_t)k * cells + c] = 1;
    }
  } else {  // rendering.py:283-286,333: the backdrop's own cells, then every static drape's whole curtain
    for (int c = 0; c < cells; ++c) {
      const int k = char_index(d, d->backdrop[c]);
      if (k >= 0) B->bytes[H->off_baselay + (size_t)k * cells + c] = 1;
    }
    for (int z = 0; z < d->n_entities; ++z) {
      if (z == agent_z) continue;
      const int k = char_index(d, d->entities[z].character);
      for (int c = 0; c < cells; ++c) B->bytes[H->off_baselay + (size_t)k * cells + c] = d->masks[(size_t)z * cells + c] ? 1 : 0;
    }
    const int ka = char_index(d, ag.character);   // the agent's plane holds the agent only
    for (int c = 0; c < cells; ++c) B->bytes[H->off_baselay + (size_t)ka * cells + c] = 0;
  }
  B->pad();
  H->blob_bytes_ext = (int32_t)B->bytes.size();
  H->off_baselay_wrap = B->reserve((size_t)L * cells + 24);
  for (int i = 0; i < L * cells + 24; ++i)
    B->bytes[H->off_baselay_wrap + i] = B->bytes[H->off_baselay + i % (L * cells)];
  B->pad();
  return CX_OK;
}

// The CX_KIND_PICKUP (and CX_KIND_DOOR) region of a single-agent game (CxPickHeader), appended to the blob behind the
// agent tables.
static int build_pick_tables(const cx_game_desc* d, int agent_z, const int* order, const CxAgentHeader& H,
                             CxPickHeader* P, Blob* B) {
  const int cells = d->rows * d->cols;
  memset(P, 0, sizeof(*P));
  int n_drapes = 0, side = -1;
  for (int z = 0; z < d->n_entities; ++z) n_drapes += d->entities[z].kind == CX_KIND_PICKUP;
  if (!n_drapes) return CX_OK;
  const cx_entity_desc& ag = d->entities[agent_z];
  if (ag.kind == CX_KIND_SPRITE) {
    cx_set_error("cx_game_create: pickup drapes need a single-agent game whose agent is a one-cell drape; this game's "
                 "agent is a sprite");
    return CX_ERR_UNSUPPORTED;
  }
  if (d->n_perf_regions) {
    cx_set_error("cx_game_create: pickup drapes together with performance regions are not supported");
    return CX_ERR_UNSUPPORTED;
  }
  if (d->unoccluded_layers) {
    cx_set_error("cx_game_create: pickup drapes need occluded layers (occlusion_in_layers=True)");
    return CX_ERR_UNSUPPORTED;
  }
  int agent_cell;
  popcount_mask(d->masks + (size_t)agent_z * cells, cells, &agent_cell);
  std::vector<uint8_t> absent, vis;
  compose_static(d, agent_z, false, &absent, &vis);
  std::vector<uint8_t> item_at(cells + 1, CX_NO_ITEM);
  std::vector<CxPickItem> items;
  std::vector<CxPickDrape> drapes;
  std::vector<int> drape_of(d->n_entities, -1);
  for (int z = 0; z < d->n_entities; ++z) {
    const cx_entity_desc& e = d->entities[z];
    if (e.kind != CX_KIND_PICKUP) continue;
    drape_of[z] = (int)drapes.size();
    const int ch = e.character;
    if (z > agent_z) {
      cx_set_error("cx_game_create: pickup drape '%c' lies in front of the agent in z-order; pickup drapes must be below "
                   "it", ch);
      return CX_ERR_UNSUPPORTED;
    }
    const int after = e.update_rank > ag.update_rank ? 1 : 0;
    if (side >= 0 && side != after) {
      cx_set_error("cx_game_create: pickup drape '%c' updates on the other side of the agent than another pickup "
                   "drape; all pickup drapes must update before it or all after it", ch);
      return CX_ERR_UNSUPPORTED;
    }
    side = after;
    for (int y = 0; y < d->n_entities; ++y) {
      const cx_entity_desc& o = d->entities[y];
      if (o.kind == CX_KIND_PICKUP || o.update_rank < e.update_rank) continue;
      bool directs = o.reward_actions || o.terminate_actions || o.discount_actions;
      for (int a = 0; a < d->n_actions; ++a) directs |= o.terminate_chars[a] != 0;
      if (directs) {   // the kernel adds the item's reward last and lets its termination win
        cx_set_error("cx_game_create: entity '%c' updates after pickup drape '%c' and calls add_reward, "
                     "terminate_episode or change_default_discount; entities after a pickup drape may not", o.character,
                     ch);
        return CX_ERR_UNSUPPORTED;
      }
    }
    if (e.watch != agent_z) {
      cx_set_error("cx_game_create: pickup drape '%c' must watch the agent", ch);
      return CX_ERR_UNSUPPORTED;
    }
    CxPickDrape pd;
    memset(&pd, 0, sizeof(pd));
    const int own = char_index(d, ch);
    for (int a = 0; a < d->n_actions; ++a) pd.reward[a] = e.entry_reward[a][own];
    pd.terminates = e.terminate_emptied ? 1 : 0;
    pd.emptied_value = e.emptied_value;
    const uint8_t* m = d->masks + (size_t)z * cells;
    for (int c = 0; c < cells; ++c) {
      if (!m[c]) continue;
      if (item_at[c] != CX_NO_ITEM) {
        cx_set_error("cx_game_create: pickup drape '%c' shares cell %d with another pickup drape", ch, c);
        return CX_ERR_UNSUPPORTED;
      }
      if (c == agent_cell) {
        cx_set_error("cx_game_create: pickup drape '%c' has an item under the agent's initial cell %d", ch, c);
        return CX_ERR_UNSUPPORTED;
      }
      if ((int)items.size() >= CX_MAX_PICKUPS) {
        cx_set_error("cx_game_create: more than %d item cells in all (pickup drape '%c')", CX_MAX_PICKUPS, ch);
        return CX_ERR_UNSUPPORTED;
      }
      CxPickItem it;
      it.cell = (uint8_t)c;
      it.under_ch = absent[c];
      const int k = char_index(d, absent[c]);
      it.under_k = (uint8_t)(k < 0 ? 0xFF : k);
      it.drape = (uint8_t)drapes.size();
      pd.items |= 1ull << items.size();
      item_at[c] = (uint8_t)items.size();
      items.push_back(it);
    }
    drapes.push_back(pd);
  }
  P->n_items = (int32_t)items.size();
  P->after = side > 0 ? 1 : 0;
  P->all = P->n_items == 64 ? ~0ull : (1ull << P->n_items) - 1;
  P->scene_all = P->all;

  // doors: their cells follow the items (CxPickHeader)
  std::vector<uint8_t> open_all, unused;
  compose_static(d, agent_z, true, &open_all, &unused, ~0u);
  for (int z = 0; z < d->n_entities; ++z) {
    const cx_entity_desc& e = d->entities[z];
    if (e.kind != CX_KIND_DOOR) continue;
    const int ch = e.character, k = e.door_key;
    if (P->n_doors >= CX_MAX_DOORS) {
      cx_set_error("cx_game_create: door drape '%c' is one more than the %d doors a game may have", ch, CX_MAX_DOORS);
      return CX_ERR_UNSUPPORTED;
    }
    if (z > agent_z) {
      cx_set_error("cx_game_create: door drape '%c' lies in front of the agent in z-order; doors must be below it", ch);
      return CX_ERR_UNSUPPORTED;
    }
    if (e.update_rank < d->entities[k].update_rank) {   // it would open one step after its key drape empties
      cx_set_error("cx_game_create: door drape '%c' updates before its key drape '%c'; a door must update after its key",
                   ch, d->entities[k].character);
      return CX_ERR_UNSUPPORTED;
    }
    bool acts = e.reward_actions || e.terminate_actions || e.discount_actions || e.watch >= 0;
    for (int a = 0; a < d->n_actions; ++a)
      acts |= e.terminate_chars[a] || e.n_zdirs[a] || e.move_dr[a] || e.move_dc[a];
    if (acts) {
      cx_set_error("cx_game_create: door drape '%c' moves, watches an entity or calls a plot directive; a door may not",
                   ch);
      return CX_ERR_UNSUPPORTED;
    }
    const uint8_t* m = d->masks + (size_t)z * cells;
    for (int c = 0; c < cells; ++c) {
      if (!m[c]) continue;
      if (item_at[c] != CX_NO_ITEM) {
        cx_set_error("cx_game_create: door drape '%c' shares cell %d with an item or another door", ch, c);
        return CX_ERR_UNSUPPORTED;
      }
      if (c == agent_cell) {
        cx_set_error("cx_game_create: door drape '%c' covers the agent's initial cell %d", ch, c);
        return CX_ERR_UNSUPPORTED;
      }
      if ((int)items.size() >= CX_MAX_PICKUPS) {
        cx_set_error("cx_game_create: more than %d item and door cells in all (door drape '%c')", CX_MAX_PICKUPS, ch);
        return CX_ERR_UNSUPPORTED;
      }
      CxPickItem it;
      it.cell = (uint8_t)c;
      it.under_ch = open_all[c];
      const int kc = char_index(d, open_all[c]);
      it.under_k = (uint8_t)(kc < 0 ? 0xFF : kc);
      it.drape = (uint8_t)P->n_doors;
      P->door_cells[P->n_doors] |= 1ull << items.size();
      item_at[c] = (uint8_t)items.size();
      items.push_back(it);
    }
    P->door_keys[P->n_doors] = drapes[drape_of[k]].items;
    drapes[drape_of[k]].opens |= 1u << P->n_doors;
    P->scene_all |= P->door_cells[P->n_doors];
    ++P->n_doors;
  }

  const int A = d->n_actions, states = 1 << P->n_doors;
  P->tt_size = (A + 1) * (cells + 1);
  P->td_size = (A + 1) * (H.td_per_cell ? cells + 1 : 1);
  P->item_at = 0;
  P->items = (cells + 1 + 15) / 16 * 16;
  P->drapes = (P->items + (int32_t)(items.size() * sizeof(CxPickItem)) + 15) / 16 * 16;
  P->door_tt = (P->drapes + (int32_t)(drapes.size() * sizeof(CxPickDrape)) + 15) / 16 * 16;
  P->door_tr = P->door_tt + (states - 1) * P->tt_size * 4;
  P->door_td = P->door_tr + (states - 1) * P->tt_size * 4;
  P->drape_cells = (P->door_td + (states - 1) * P->td_size * 4 + 15) / 16 * 16;
  P->bytes = P->drape_cells + (P->n_doors ? (int32_t)drapes.size() * 8 + 15 : 0) / 16 * 16;
  P->tt_first = (H.blob_bytes_ext + P->door_tt - H.off_tt) / 4;
  P->tr_first = (H.blob_bytes_ext + P->door_tr - H.off_tr) / 4;
  P->td_first = (H.blob_bytes_ext + P->door_td - H.off_td) / 4;
  P->off = B->reserve(P->bytes);
  memcpy(&B->bytes[P->off + P->item_at], item_at.data(), cells + 1);
  memcpy(&B->bytes[P->off + P->items], items.data(), items.size() * sizeof(CxPickItem));
  memcpy(&B->bytes[P->off + P->drapes], drapes.data(), drapes.size() * sizeof(CxPickDrape));
  for (int dr = 0; dr < (P->n_doors ? (int)drapes.size() : 0); ++dr) {
    uint64_t c = 0;
    for (int d = 0; d < P->n_doors; ++d)
      if ((drapes[dr].opens >> d) & 1) c |= P->door_cells[d];
    memcpy(&B->bytes[P->off + P->drape_cells + dr * 8], &c, 8);
  }
  for (int st = 1; st < states; ++st) {   // the step tables of every other door state, with the same item check
    std::vector<uint8_t> absent, present, vis;
    compose_static(d, agent_z, false, &absent, &vis, (uint32_t)st);
    compose_static(d, agent_z, true, &present, &unused, (uint32_t)st);
    const int rc = check_items_irrelevant(d, agent_z, order, absent, present, vis);
    if (rc != CX_OK) return rc;
    uint8_t* r = &B->bytes[P->off];
    fill_step_tables(d, agent_z, order, H, absent, vis, (uint32_t*)(r + P->door_tt) + (st - 1) * P->tt_size,
                     (float*)(r + P->door_tr) + (st - 1) * P->tt_size, (float*)(r + P->door_td) + (st - 1) * P->td_size);
  }
  B->pad();
  return CX_OK;
}

static int build_generic_tables(const cx_game_desc* d, const int* order, CxGenHeader* H, Blob* B) {
  const int R = d->rows, C = d->cols, cells = R * C, L = d->n_chars, A = d->n_actions, E = d->n_entities;
  memset(H, 0, sizeof(*H));
  H->rows = R;
  H->cols = C;
  H->cells = cells;
  H->n_actions = A;
  H->n_chars = L;
  H->n_ent = E;
  H->n_groups = d->n_groups > 0 ? d->n_groups : 1;
  H->mask_words = (cells + 31) / 32;
  H->max_steps = d->max_episode_steps;
  H->auto_reset = d->auto_reset;
  memcpy(H->chars, d->chars, CX_MAX_CHARS);
  build_action_table(d, order, &H->act);
  int first_drape = E;
  for (int z = 0; z < E; ++z)
    if (d->entities[z].kind != CX_KIND_SPRITE) {
      first_drape = z;
      break;
    }
  H->zero_backdrop = (first_drape == E);  // no drape: clear() zeroes the aliased backdrop, rendering.py:111,128
  int n_dyn = 0;
  bool any_stamp = false, needs_prev = false;
  for (int i = 0; i < E; ++i) H->update_order[i] = (uint8_t)order[i];
  for (int k = 0; k < CX_MAX_CHARS; ++k) H->z_of_char[k] = -1;
  for (int z = 0; z < E; ++z) {
    const int k = char_index(d, d->entities[z].character);
    if (k >= 0) H->z_of_char[k] = (int8_t)z;
  }
  for (int z = 0; z < E; ++z) {
    const cx_entity_desc& e = d->entities[z];
    CxGenEntity& g = H->ent[z];
    g.ch = e.character;
    g.kind = e.kind;
    g.visible = e.kind == CX_KIND_SPRITE ? (e.visible != 0) : 1;
    g.group = e.update_group;
    g.chidx = (uint8_t)char_index(d, e.character);
    g.rank = (uint8_t)e.update_rank;
    g.watch = e.watch < 0 ? 0xFF : (uint8_t)e.watch;
    g.blockers = e.blockers;
    g.reward_actions = e.reward_actions;
    memcpy(g.dr, e.move_dr, CX_MAX_ACTIONS);
    memcpy(g.dc, e.move_dc, CX_MAX_ACTIONS);
    memcpy(g.step_reward, e.step_reward, sizeof(g.step_reward));
    memcpy(g.vis_op, e.visible_op, CX_MAX_ACTIONS);
    g.terminate_actions = e.terminate_actions;
    g.discount_actions = e.discount_actions;
    memcpy(g.discount_value, e.discount_value, sizeof(g.discount_value));
    memcpy(g.term_chars, e.terminate_chars, sizeof(g.term_chars));
    memcpy(g.term_value, e.terminate_value, sizeof(g.term_value));
    for (int a = 0; a < d->n_actions; ++a)
      if (e.terminate_chars[a]) H->cond_term = 1;
    g.dyn_slot = 0xFF;
    if (e.kind != CX_KIND_STATIC) {
      if (n_dyn >= CX_MAX_DYN) {
        cx_set_error("cx_game_create: more than %d moving entities", CX_MAX_DYN);
        return CX_ERR_UNSUPPORTED;
      }
      g.dyn_slot = (uint8_t)n_dyn++;
    }
    g.stamps = (e.kind == CX_KIND_SPRITE && g.visible && z < first_drape && !H->zero_backdrop);
    any_stamp |= g.stamps != 0;
    if (((e.kind == CX_KIND_CELL || e.kind == CX_KIND_SPRITE) && e.blockers) || e.watch >= 0) needs_prev = true;
    int first;
    const uint8_t* m = d->masks + (size_t)z * cells;
    switch (e.kind) {
      case CX_KIND_CELL:
        popcount_mask(m, cells, &first);
        g.init_state = first < 0 ? (uint16_t)CX_EMPTY_CELL16 : (uint16_t)first;
        break;
      case CX_KIND_SPRITE:
        g.init_state = (uint16_t)(e.init_row * C + e.init_col);
        break;
      default:
        g.init_state = 0;
    }
  }
  // ---- render state that changes during play: extra dynamic slots behind those of the moving entities ----
  bool dyn_vis, dyn_z, dyn_bd;
  dynamic_render_needs(d, &dyn_vis, &dyn_z, &dyn_bd);
  H->dyn_render = (dyn_vis || dyn_z || dyn_bd) ? 1 : 0;
  H->slot_vis = H->slot_zperm = H->slot_bd = -1;
  for (int z = 0; z < E; ++z)
    if (H->ent[z].dyn_slot != 0xFF) H->slot_init[H->ent[z].dyn_slot] = H->ent[z].init_state;
  if (H->dyn_render) {
    const int need = (dyn_vis ? 1 : 0) + (dyn_z ? 2 : 0) + (dyn_bd ? 1 : 0);
    if (n_dyn + need > CX_MAX_DYN) {
      cx_set_error("cx_game_create: %d moving entities + %d render-state slots exceed %d state slots", n_dyn, need,
                   CX_MAX_DYN);
      return CX_ERR_UNSUPPORTED;
    }
    if (dyn_z && E > CX_ZPERM_MAX_ENT) {
      cx_set_error("cx_game_create: z-order directives are supported for games of at most %d sprites and drapes",
                   CX_ZPERM_MAX_ENT);
      return CX_ERR_UNSUPPORTED;
    }
    if (dyn_vis) {
      uint16_t bits = 0;
      for (int z = 0; z < E; ++z)
        if (H->ent[z].kind == CX_KIND_SPRITE && H->ent[z].visible) bits |= (uint16_t)(1u << z);
      H->slot_vis = n_dyn;
      H->slot_init[n_dyn++] = bits;
    }
    if (dyn_z) {
      H->slot_zperm = n_dyn;
      H->slot_init[n_dyn++] = 0x3210;
      H->slot_init[n_dyn++] = 0x7654;
    }
    if (dyn_bd) {
      H->slot_bd = n_dyn;
      H->slot_init[n_dyn++] = 0;
    }
    // With visibility or z-order changes any sprite may come to lie, visibly, behind the first drape and
    // stamp the backdrop (quirk Q1): keep a per-env plane whenever the game has both sprites and drapes.
    bool any_sprite = false;
    for (int z = 0; z < E; ++z) any_sprite |= d->entities[z].kind == CX_KIND_SPRITE;
    if ((dyn_vis || dyn_z) && any_sprite && !H->zero_backdrop) any_stamp = true;
    if (dyn_bd && any_stamp) {
      cx_set_error("cx_game_create: a rolling backdrop together with sprites that stamp the backdrop "
                   "(sprites behind the first drape, SURVEY quirk Q1) is not supported");
      return CX_ERR_UNSUPPORTED;
    }
    memcpy(H->bd_dr, d->backdrop_dr, CX_MAX_ACTIONS);
    memcpy(H->bd_dc, d->backdrop_dc, CX_MAX_ACTIONS);
    for (int a = 0; a < A; ++a) {
      int k = 0;
      for (int i = 0; i < E; ++i) {  // directives are applied in call order = update order (plot.py:157-159)
        const cx_entity_desc& e = d->entities[order[i]];
        for (int j = 0; j < e.n_zdirs[a]; ++j) {
          if (k >= CX_MAX_ZDIR_GAME) {
            cx_set_error("cx_game_create: more than %d z-order directives in one step", CX_MAX_ZDIR_GAME);
            return CX_ERR_UNSUPPORTED;
          }
          H->zdir[a][k++] = (uint8_t)((e.z_move[a][j] << 4) | (e.z_front[a][j] < 0 ? 0xF : e.z_front[a][j]));
        }
      }
      H->n_zdir[a] = (uint8_t)k;
    }
  }
  H->n_dyn = n_dyn;
  H->has_dynbd = any_stamp;
  H->needs_prev = needs_prev;
  H->off_masks = B->reserve(((size_t)E * H->mask_words + 1) * 4);  // +1: the composer's funnel shift reads one word ahead
  for (int z = 0; z < E; ++z) {
    uint32_t* w = (uint32_t*)&B->bytes[H->off_masks + (size_t)z * H->mask_words * 4];
    const uint8_t* m = d->masks + (size_t)z * cells;
    if (d->entities[z].kind == CX_KIND_STATIC || d->entities[z].kind == CX_KIND_ROLL)
      for (int c = 0; c < cells; ++c)
        if (m[c]) w[c >> 5] |= 1u << (c & 31);
  }
  H->off_backdrop = B->reserve(cells);
  memcpy(&B->bytes[H->off_backdrop], d->backdrop, cells);
  if (H->zero_backdrop) memset(&B->bytes[H->off_backdrop], 0, cells);
  H->off_entry = B->reserve((size_t)E * A * L * sizeof(float));
  float* entry = (float*)&B->bytes[H->off_entry];
  for (int z = 0; z < E; ++z)
    for (int a = 0; a < A; ++a)
      for (int k = 0; k < L; ++k) entry[(z * A + a) * L + k] = d->entities[z].entry_reward[a][k];
  H->off_rc = B->reserve((size_t)cells * 2);
  uint16_t* rc = (uint16_t*)&B->bytes[H->off_rc];
  for (int c = 0; c < cells; ++c) rc[c] = (uint16_t)(((c / C) << 8) | (c % C));
  H->off_rowbits = -1;
  if (C <= 64) {  // per-row bitsets: the fast composition path
    H->off_rowbits = B->reserve((size_t)E * R * 8);
    uint64_t* rb = (uint64_t*)&B->bytes[H->off_rowbits];
    for (int z = 0; z < E; ++z) {
      const uint8_t* m = d->masks + (size_t)z * cells;
      if (d->entities[z].kind == CX_KIND_STATIC || d->entities[z].kind == CX_KIND_ROLL)
        for (int c = 0; c < cells; ++c)
          if (m[c]) rb[z * R + c / C] |= 1ull << (c % C);
    }
  }
  // direct composer eligibility (see CxGenHeader::direct)
  bool direct_ok = cells >= 16 && E > 0 && !H->dyn_render;
  {
    size_t tab_bytes = 0;
    const int xw = (cells + 16 + 31) / 32 + 1;
    for (int z = 0; z < E; ++z) {
      const CxGenEntity& g = H->ent[z];
      if (g.kind == CX_KIND_STATIC) tab_bytes += (size_t)xw * 4;
      if (g.kind == CX_KIND_ROLL) tab_bytes += (size_t)C * xw * 4;
    }
    if (tab_bytes > 48 * 1024) direct_ok = false;
    // every visible one-cell entity must be below all masks or above all masks
    for (int z = 0; z < E && direct_ok; ++z) {
      const CxGenEntity& g = H->ent[z];
      if (g.kind == CX_KIND_STATIC || g.kind == CX_KIND_ROLL || !g.visible) continue;
      int below = 0, above = 0;
      for (int y = 0; y < E; ++y)
        if (H->ent[y].kind == CX_KIND_STATIC || H->ent[y].kind == CX_KIND_ROLL) (y < z ? below : above)++;
      if (below && above) direct_ok = false;
    }
  }
  // Mask entities (static / rolling drapes) are composed from linear bitsets.  A rolling mask, and a static
  // mask with a visible one-cell entity above it in z-order (whose cell is punched out of the mask), need a
  // per-env copy in shared memory.
  int n_lin = 0;
  bool wide_roll = false;
  for (int z = 0; z < E; ++z) {
    CxGenEntity& g = H->ent[z];
    g.lin_slot = 0xFF;
    if (g.kind != CX_KIND_STATIC && g.kind != CX_KIND_ROLL) continue;
    bool per_env = g.kind == CX_KIND_ROLL;
    if (g.kind == CX_KIND_ROLL && C > 64) wide_roll = true;
    for (int y = z + 1; y < E; ++y)
      if ((H->ent[y].kind == CX_KIND_CELL || H->ent[y].kind == CX_KIND_SPRITE) && H->ent[y].visible) per_env = true;
    if (per_env) g.lin_slot = (uint8_t)(n_lin < 255 ? n_lin : 254), ++n_lin;
  }
  H->n_lin = n_lin;
  H->fast_compose = (n_lin <= CX_MAX_LIN && !wide_roll && cells >= 16 && !H->dyn_render) ? 1 : 0;
  for (int i = 0; i < CX_MAX_LIN; ++i) H->off_colroll[i] = -1;
  if (H->fast_compose && !direct_ok) {
    // A roll by (dr, dc) is a column roll inside every board row followed by a rotation of the linear
    // bitset by dr * cols bits.  Tabulating the column rolls leaves the kernel only the rotation.
    const int lw = H->mask_words + 1;
    for (int z = 0; z < E; ++z) {
      const CxGenEntity& g = H->ent[z];
      if (g.kind != CX_KIND_ROLL || g.lin_slot >= CX_MAX_LIN || (size_t)C * lw * 4 > 16 * 1024) continue;
      const int32_t off = B->reserve((size_t)C * lw * 4);
      H->off_colroll[g.lin_slot] = off;
      const uint8_t* m = d->masks + (size_t)z * cells;
      for (int dc = 0; dc < C; ++dc) {
        uint32_t* w = (uint32_t*)&B->bytes[off + (size_t)dc * lw * 4];
        for (int r = 0; r < R; ++r)
          for (int c = 0; c < C; ++c)
            if (m[r * C + (c - dc + C) % C]) w[(r * C + c) >> 5] |= 1u << ((r * C + c) & 31);
      }
    }
  }
  H->n_masks = H->n_points = 0;
  H->n_poke = H->n_above = 0;
  for (int z = 0; z < E; ++z) {
    const CxGenEntity& g = H->ent[z];
    if (g.kind == CX_KIND_STATIC || g.kind == CX_KIND_ROLL) {
      H->mask_prog[H->n_masks++] = (uint32_t)z | ((uint32_t)g.ch << 8) | ((uint32_t)g.lin_slot << 16) | ((uint32_t)g.kind << 24);
    } else if (g.visible) {
      uint32_t holes = 0;
      for (int y = 0; y < z; ++y)
        if ((H->ent[y].kind == CX_KIND_STATIC || H->ent[y].kind == CX_KIND_ROLL) && H->ent[y].lin_slot != 0xFF &&
            H->ent[y].lin_slot < 32)
          holes |= 1u << H->ent[y].lin_slot;
      H->point_holes[H->n_points] = holes;
      H->point_prog[H->n_points++] =
          (uint32_t)z | ((uint32_t)g.ch << 8) | ((uint32_t)g.dyn_slot << 16) | ((uint32_t)(g.stamps ? 1 : 0) << 24);
    }
  }
  // ---- direct composer (see CxGenHeader::direct) --------------------------------------------------
  {
    const bool ok = direct_ok;
    const int xw = (cells + 16 + 31) / 32 + 1;
    if (ok) {
      H->direct = 1;
      H->fast_compose = 1;
      H->dtab_words = xw;
      H->n_lin = 0;
      for (int z = 0; z < E; ++z) H->ent[z].lin_slot = 0xFF;
      for (int i = 0; i < CX_MAX_LIN; ++i) H->off_colroll[i] = -1;  // (their bytes stay in the blob, unused)
      for (int i = 0; i < H->n_masks; ++i) {
        const int z = (int)(H->mask_prog[i] & 0xFF);
        const bool roll = H->ent[z].kind == CX_KIND_ROLL;
        H->mask_prog[i] |= 0xFFu << 16;
        const int rows_in_tab = roll ? C : 1;
        const int32_t off = B->reserve((size_t)rows_in_tab * xw * 4);
        H->off_dtab[i] = off;
        const uint8_t* m = d->masks + (size_t)z * cells;
        for (int dc = 0; dc < rows_in_tab; ++dc) {
          uint32_t* w = (uint32_t*)&B->bytes[off + (size_t)dc * xw * 4];
          auto bit = [&](int cell) { return m[(cell / C) * C + ((cell % C) - dc + C) % C] != 0; };
          for (int c = 0; c < cells + 16; ++c)
            if (bit(c % cells)) w[c >> 5] |= 1u << (c & 31);
        }
      }
      for (int i = 0; i < H->n_points; ++i) {
        const int z = (int)(H->point_prog[i] & 0xFF);
        int below = 0;
        for (int y = 0; y < z; ++y)
          if (H->ent[y].kind == CX_KIND_STATIC || H->ent[y].kind == CX_KIND_ROLL) ++below;
        H->point_holes[i] = 0;
        if (below) H->point_prog[i] |= 2u << 24;  // above the masks: stored over the finished board
      }
      H->n_poke = H->n_above = 0;
      for (int i = 0; i < H->n_points; ++i) {
        const uint32_t prog = H->point_prog[i];
        if (!(prog >> 24)) ++H->n_poke;
        if ((prog >> 24) & 2u) H->above_prog[H->n_above++] = (uint16_t)((prog & 0xFF00u) | ((prog >> 16) & 0xFFu));
      }
    }
  }
  // ---- table-driven step (see CxGenHeader::simple_step) ------------------------------------------------
  H->n_stampers = 0;
  for (int z = 0; z < E; ++z)
    if (H->ent[z].stamps) H->stamper[H->n_stampers++] = (uint16_t)((H->ent[z].ch << 8) | H->ent[z].dyn_slot);
  {
    const bool simple = !needs_prev && H->n_groups == 1 && !H->dyn_render;
    for (int z = 0; z < E; ++z) {
      const CxGenEntity& g = H->ent[z];
      if (g.dyn_slot == 0xFF) continue;
      H->slot_kind[g.dyn_slot] = g.kind;
      memcpy(H->slot_dr[g.dyn_slot], g.dr, CX_MAX_ACTIONS);
      memcpy(H->slot_dc[g.dyn_slot], g.dc, CX_MAX_ACTIONS);
    }
    for (int a = 0; a < A; ++a) {
      bool first_add = true;
      float summed = 0.0f;
      for (int i = 0; i < E; ++i) {
        const cx_entity_desc& e = d->entities[order[i]];
        if (!(e.reward_actions >> a & 1)) continue;
        if (first_add) {
          summed = e.step_reward[a];
          first_add = false;
        } else {
          volatile float s2 = e.step_reward[a] + summed;  // plot.py:211: reward + running sum
          summed = s2;
        }
      }
      H->simple_reward[a] = summed;
    }
    H->simple_step = simple ? 1 : 0;
    H->off_sdelta = B->reserve((size_t)CX_MAX_ACTIONS * CX_MAX_DYN * 4);
    uint32_t* sd = (uint32_t*)&B->bytes[H->off_sdelta];
    H->roll_slots = 0;
    for (int dslot = 0; dslot < n_dyn && !H->dyn_render; ++dslot) {
      if (H->slot_kind[dslot] == CX_KIND_ROLL) H->roll_slots |= 1u << dslot;
      for (int a = 0; a < A; ++a)
        sd[a * CX_MAX_DYN + dslot] =  // |dr| < rows, |dc| < cols (validated): non-negative residues
            ((uint32_t)((H->slot_dr[dslot][a] + R) % R) << 16) | (uint32_t)((H->slot_dc[dslot][a] + C) % C);
    }
    H->fast_loop = (simple && H->direct && cells <= 496 && H->n_masks <= 2) ? 1 : 0;
  }
  // envs per warp: one plane tile of at most 8 KB per warp keeps >= 20 warps per SM resident
  int tile = 32;
  while (tile > 1 && (size_t)tile * cells > 8 * 1024) tile >>= 1;
  H->tile_envs = tile;
  B->pad();
  H->blob_bytes = (int32_t)B->bytes.size();
  return CX_OK;
}

extern "C" int cx_game_create(const cx_game_desc* desc, cx_game** out) {
  if (!out) {
    cx_set_error("cx_game_create: out is NULL");
    return CX_ERR_INVALID_ARG;
  }
  *out = nullptr;
  int rc = validate(desc);
  if (rc != CX_OK) return rc;
  cx_game* g = new (std::nothrow) cx_game;
  if (!g) {
    cx_set_error("cx_game_create: out of host memory");
    return CX_ERR_NOMEM;
  }
  memset(g, 0, sizeof(*g));
  g->desc = *desc;
  g->desc.backdrop = nullptr;
  g->desc.masks = nullptr;
  g->desc.perf_regions = nullptr;
  const int cells = desc->rows * desc->cols;

  int order[CX_MAX_ENTITIES];
  for (int z = 0; z < desc->n_entities; ++z) order[desc->entities[z].update_rank] = z;

  Blob blob;
  int agent_z = -1;
  bool pickups = false;
  for (int z = 0; z < desc->n_entities; ++z) pickups |= desc->entities[z].kind == CX_KIND_PICKUP;
  if (agent_path_applies(desc, &agent_z)) {
    g->path = CX_PATH_AGENT;
    rc = build_agent_tables(desc, agent_z, order, &g->ah, &blob);
    if (rc == CX_OK) rc = build_pick_tables(desc, agent_z, order, g->ah, &g->ph, &blob);
    if (rc != CX_OK) {
      delete g;
      return rc;
    }
  } else {
    if (pickups) {
      cx_set_error("cx_game_create: pickup drapes need a single-agent game (one moving one-cell drape over a static "
                   "scene); this game runs on the generic kernels");
      delete g;
      return CX_ERR_UNSUPPORTED;
    }
    if (desc->n_perf_regions) {
      cx_set_error("cx_game_create: performance regions need a single-agent game (one moving one-cell drape over a "
                   "static scene); this game runs on the generic kernels");
      delete g;
      return CX_ERR_UNSUPPORTED;
    }
    g->path = CX_PATH_GENERIC;
    rc = build_generic_tables(desc, order, &g->gh, &blob);
    if (rc != CX_OK) {
      delete g;
      return rc;
    }
  }
  const CxActionTable& act = g->path == CX_PATH_AGENT ? g->ah.act : g->gh.act;
  bool can_term = false;
  for (int a = 0; a < desc->n_actions; ++a) {
    can_term |= act.over[a] != 0;
    for (int z = 0; z < desc->n_entities; ++z) can_term |= desc->entities[z].terminate_chars[a] != 0;
  }
  for (int z = 0; z < desc->n_entities; ++z)
    can_term |= desc->entities[z].kind == CX_KIND_PICKUP && desc->entities[z].terminate_emptied;
  const int tracks = (can_term || desc->max_episode_steps > 0 || desc->track_returns) ? 1 : 0;
  if (g->path == CX_PATH_AGENT)
    g->ah.track = tracks;
  else
    g->gh.track = tracks;

  cx_game_info& I = g->info;
  I.rows = desc->rows;
  I.cols = desc->cols;
  I.cells = cells;
  I.n_chars = desc->n_chars;
  I.n_actions = desc->n_actions;
  I.n_entities = desc->n_entities;
  I.path = g->path;
  I.can_terminate = can_term;
  I.tracks = tracks;
  I.tracks_performance = desc->n_perf_regions ? 1 : 0;
  I.has_dynamic_backdrop = g->path == CX_PATH_GENERIC ? g->gh.has_dynbd : 0;
  I.board_bytes_per_env = cells;
  I.dynamic_render = g->path == CX_PATH_GENERIC ? g->gh.dyn_render : 0;
  I.n_pickups = g->path == CX_PATH_AGENT ? g->ph.n_items : 0;
  I.state_bytes_per_env = (g->path == CX_PATH_AGENT ? 1 : 2 * g->gh.n_dyn) + (tracks ? 6 : 0) +
                          (I.has_dynamic_backdrop ? cells : 0) + (I.tracks_performance ? 4 : 0) +
                          (I.n_pickups ? 8 : 0);
  if (g->ph.n_doors && cx_agent_obs_smem_bytes(g) > 227 * 1024) {   // door games run on the lane-per-env kernel only
    cx_set_error("cx_game_create: the step tables of the %d door states (%d bytes) and the board tiles need %zu bytes of "
                 "shared memory per CTA, more than the 227 KB a CTA can have; use fewer doors, actions or cells",
                 1 << g->ph.n_doors, g->ph.bytes, cx_agent_obs_smem_bytes(g));
    delete g;
    return CX_ERR_UNSUPPORTED;
  }

  CX_CUDA_OK(cudaGetDevice(&g->device));
  CX_CUDA_OK(cudaDeviceGetAttribute(&g->sm_count, cudaDevAttrMultiProcessorCount, g->device));
  CX_CUDA_OK(cudaDeviceGetAttribute(&g->smem_per_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, g->device));
  CX_CUDA_OK(cudaMalloc((void**)&g->d_blob, blob.bytes.size()));
  CX_CUDA_OK(cudaMemcpy(g->d_blob, blob.bytes.data(), blob.bytes.size(), cudaMemcpyHostToDevice));
  CX_CUDA_OK(cudaMalloc((void**)&g->d_chars, CX_MAX_CHARS));
  CX_CUDA_OK(cudaMemcpy(g->d_chars, desc->chars, CX_MAX_CHARS, cudaMemcpyHostToDevice));
  *out = g;
  return CX_OK;
}

extern "C" int cx_game_destroy(cx_game* g) {
  if (!g) return CX_OK;
  if (g->d_blob) cudaFree(g->d_blob);
  if (g->d_chars) cudaFree(g->d_chars);
  delete g;
  return CX_OK;
}

extern "C" int cx_game_get_info(const cx_game* g, cx_game_info* out) {
  if (!g || !out) {
    cx_set_error("cx_game_get_info: NULL argument");
    return CX_ERR_INVALID_ARG;
  }
  *out = g->info;
  return CX_OK;
}

extern "C" int64_t cx_state_bytes(const cx_game* g, int64_t n) {
  if (!g || n < 1) return -1;
  return cx_layout(g, n).total;
}

static int check_common(const cx_game* g, const void* d_state, int64_t n, const char* who) {
  if (!g || !d_state) {
    cx_set_error("%s: NULL game or state", who);
    return CX_ERR_INVALID_ARG;
  }
  if (n < 1) {
    cx_set_error("%s: n_envs must be >= 1", who);
    return CX_ERR_INVALID_ARG;
  }
  if ((uintptr_t)d_state % 256) {
    cx_set_error("%s: state blob must be 256-byte aligned", who);
    return CX_ERR_INVALID_ARG;
  }
  return CX_OK;
}

extern "C" int cx_reset(const cx_game* g, void* d_state, int64_t n, const uint8_t* d_mask, void* stream) {
  int rc = check_common(g, d_state, n, "cx_reset");
  if (rc) return rc;
  return cx_launch_reset(g, d_state, n, d_mask, (cudaStream_t)stream);
}

extern "C" int cx_render(const cx_game* g, const void* d_state, int64_t n, uint8_t* d_board, void* stream) {
  int rc = check_common(g, d_state, n, "cx_render");
  if (rc) return rc;
  if (!d_board) {
    cx_set_error("cx_render: d_board is NULL");
    return CX_ERR_INVALID_ARG;
  }
  return cx_launch_render(g, d_state, n, d_board, (cudaStream_t)stream);
}

// The kernel route the environment variable CX_ROUTE forces (see CxRoute); unset or empty: automatic selection.  Read
// per call, so that one process (a test) can run the same inputs through every kernel.  An unknown name fails the call.
static int parse_route(CxRoute* route, const char* who) {
  static const struct {
    const char* name;
    CxRoute route;
  } kRoutes[] = {{"tile64", CX_ROUTE_TILE64},
                 {"tile128", CX_ROUTE_TILE128},
                 {"tile256", CX_ROUTE_TILE256},
                 {"lane", CX_ROUTE_LANE},
                 {"obs", CX_ROUTE_OBS},
                 {"no_step_composer", CX_ROUTE_NO_STEP_COMPOSER},
                 {"step_composer", CX_ROUTE_STEP_COMPOSER},
                 {"gen96", CX_ROUTE_GEN96},
                 {"gen80", CX_ROUTE_GEN80},
                 {"gen_wave", CX_ROUTE_GEN_WAVE}};
  *route = CX_ROUTE_AUTO;
  const char* e = getenv("CX_ROUTE");
  if (!e || !*e) return CX_OK;
  for (const auto& r : kRoutes)
    if (strcmp(e, r.name) == 0) {
      *route = r.route;
      return CX_OK;
    }
  cx_set_error("%s: unknown CX_ROUTE '%s' (tile64, tile128, tile256, lane, obs, no_step_composer, step_composer, "
               "gen96, gen80, gen_wave)", who, e);
  return CX_ERR_INVALID_ARG;
}

static int rollout_common(const cx_game* g, void* d_state, int64_t n, int32_t T, const uint8_t* d_actions,
                          const CxSynth& synth, float* d_reward, float* d_discount, uint8_t* d_flags,
                          uint8_t* d_board, void* stream, const char* who) {
  int rc = check_common(g, d_state, n, who);
  if (rc) return rc;
  if (T < 1) {
    cx_set_error("%s: n_steps must be >= 1", who);
    return CX_ERR_INVALID_ARG;
  }
  if ((!synth.on && !d_actions) || !d_reward || !d_flags || !d_board) {
    cx_set_error("%s: actions/reward/flags/board must not be NULL", who);
    return CX_ERR_INVALID_ARG;
  }
  if (synth.on && (synth.env_offset & 3)) {
    cx_set_error("%s: env_offset must be a multiple of 4", who);
    return CX_ERR_INVALID_ARG;
  }
  CxRoute route;
  rc = parse_route(&route, who);
  if (rc) return rc;
  // one step of a small batch: the stateless composer (cx_agent_step_kernels.cu) -- 2.5 against 3.1 us at 4,096 envs,
  // equal at 65,536; large batches amortise the tile staging over enough envs (2^20: 11 us against 28 us)
  if (g->path == CX_PATH_AGENT && T == 1 && !synth.on && (n < 65536 || route == CX_ROUTE_STEP_COMPOSER) &&
      route != CX_ROUTE_NO_STEP_COMPOSER && cx_agent_step_applies(g, d_board, nullptr))
    return cx_launch_agent_step(g, d_state, n, d_actions, d_reward, d_discount, d_flags, d_board, nullptr, CX_DTYPE_U8,
                                (cudaStream_t)stream);
  if (g->path == CX_PATH_AGENT) {
    const bool tile = route == CX_ROUTE_TILE64 || route == CX_ROUTE_TILE128 || route == CX_ROUTE_TILE256;
    // Batches below 32,768 envs that k_agent_rollout_lane (next) does not take -- rows that are not 16-byte aligned, i.e.
    // n not a multiple of 16 -- run on the lane-per-env TMA kernel, which handles ragged warps and unaligned buffers and
    // is a little faster there than the scalar path of k_agent_rollout (Demo 1, 32 steps: 4,096 envs 16.6 against 17.9 us).
    // The tile routes send them to k_agent_rollout as well, the obs route sends every batch here.
    int64_t small_n = 32768;
    if (tile) small_n = 0;
    if (route == CX_ROUTE_OBS) small_n = INT64_MAX;
    // Batches of a multiple of 16 envs up to ~1,800 envs per SM (2^18 on 148 SMs): k_agent_rollout_lane (lane = env, STG.128 tile
    // copies; cx_agent_lane_kernels.cu).  Demo 1, 32-step launches, % of the copy peak against the best tile build:
    // 4,096 envs 7.1 / 3.5, 65,536 56.5 / 49.7, 2^17 80.0 / 77.5, 2^18 90.3 / 90.6, 2^19 89.6 / 91.5, 2^20 86 / 95.
    // The lane route sends every batch it takes here, the tile and obs routes none.
    // Boards above 96 cells: only tiny batches (its tile copy is 2 * cells / 32 LDS.128 + STG.128 pairs per lane and
    // step, one bulk store in the TMA kernels: random 15x16 maze, 65,536 envs 64 against 88 %, 16,384 envs 18 against 36 us).
    int64_t lane_n = (int64_t)g->sm_count * (g->ah.cells <= CX_AGENT_TILE_MAX_CELLS ? 1800 : 200);
    if (tile || route == CX_ROUTE_OBS) lane_n = 0;
    if (route == CX_ROUTE_LANE) lane_n = INT64_MAX;
    if (n <= lane_n && T > 1 &&
        cx_agent_lane_applies(g, n, d_actions, synth.actions_out, d_reward, d_discount, d_flags, d_board))
      return cx_launch_agent_rollout_lane(g, d_state, n, T, d_actions, synth, d_reward, d_discount, d_flags, d_board,
                                          (cudaStream_t)stream);
    // games with pickups: always here (the PICK build), whatever the route
    if (g->ah.cells > CX_AGENT_TILE_MAX_CELLS || n < small_n || g->info.n_pickups)  // large boards, small batches: lane-per-env kernel, board only
      return cx_launch_agent_rollout_obs(g, d_state, n, T, d_actions, synth, d_reward, d_discount, d_flags, d_board,
                                         nullptr, (cudaStream_t)stream);
    return cx_launch_agent_rollout(g, d_state, n, T, d_actions, synth, d_reward, d_discount, d_flags, d_board, route,
                                   (cudaStream_t)stream);
  }
  return cx_launch_generic_rollout(g, d_state, n, T, d_actions, synth, d_reward, d_discount, d_flags, d_board, route,
                                   (cudaStream_t)stream);
}

extern "C" int cx_rollout(const cx_game* g, void* d_state, int64_t n, int32_t T, const uint8_t* d_actions,
                          float* d_reward, float* d_discount, uint8_t* d_flags, uint8_t* d_board, void* stream) {
  CxSynth none;
  memset(&none, 0, sizeof(none));
  return rollout_common(g, d_state, n, T, d_actions, none, d_reward, d_discount, d_flags, d_board, stream,
                        "cx_rollout");
}

extern "C" int cx_rollout_synth(const cx_game* g, void* d_state, int64_t n, int32_t T, uint64_t seed,
                                uint64_t env_offset, uint64_t t0, uint8_t* d_actions_out, float* d_reward,
                                float* d_discount, uint8_t* d_flags, uint8_t* d_board, void* stream) {
  CxSynth sy;
  sy.on = 1;
  sy.seed = seed;
  sy.env_offset = env_offset;
  sy.t0 = t0;
  sy.actions_out = d_actions_out;
  return rollout_common(g, d_state, n, T, nullptr, sy, d_reward, d_discount, d_flags, d_board, stream,
                        "cx_rollout_synth");
}

extern "C" int cx_rollout_observations(const cx_game* g, void* d_state, int64_t n, int32_t T, const uint8_t* d_actions,
                                       float* d_reward, float* d_discount, uint8_t* d_flags, uint8_t* d_board,
                                       uint8_t* d_layered, void* stream) {
  if (!d_layered) {
    cx_set_error("cx_rollout_observations: layered must not be NULL");
    return CX_ERR_INVALID_ARG;
  }
  CxRoute route;
  int rc = parse_route(&route, "cx_rollout_observations");
  if (rc) return rc;
  if (g && d_actions && d_reward && d_flags && d_board && T == 1 && route != CX_ROUTE_NO_STEP_COMPOSER &&
      cx_agent_step_applies(g, d_board, d_layered)) {
    rc = check_common(g, d_state, n, "cx_rollout_observations");
    if (rc) return rc;
    return cx_launch_agent_step(g, d_state, n, d_actions, d_reward, d_discount, d_flags, d_board, d_layered,
                                CX_DTYPE_U8, (cudaStream_t)stream);
  }
  if (g && d_actions && d_reward && d_flags && d_board && T >= 1 && cx_agent_obs_applies(g, true)) {
    rc = check_common(g, d_state, n, "cx_rollout_observations");
    if (rc) return rc;
    CxSynth none;
    memset(&none, 0, sizeof(none));
    return cx_launch_agent_rollout_obs(g, d_state, n, T, d_actions, none, d_reward, d_discount, d_flags, d_board,
                                       d_layered, (cudaStream_t)stream);
  }
  if (g && g->desc.unoccluded_layers) {
    if (g->path == CX_PATH_GENERIC && d_actions && d_reward && d_flags && d_board && T >= 1) {
      // generic games: the kernel reads the unoccluded layers off its entity state at every step
      rc = check_common(g, d_state, n, "cx_rollout_observations");
      if (rc) return rc;
      CxSynth none;
      memset(&none, 0, sizeof(none));
      return cx_launch_generic_rollout(g, d_state, n, T, d_actions, none, d_reward, d_discount, d_flags, d_board,
                                       route, (cudaStream_t)stream, d_layered);
    }
    cx_set_error("cx_rollout_observations: unoccluded layers need the fused kernels (16-byte aligned buffers, "
                 "boards that fit the lane-per-env kernel)");
    return CX_ERR_UNSUPPORTED;
  }
  // any other game or geometry: the step kernel, then the layers from the finished boards
  rc = cx_rollout(g, d_state, n, T, d_actions, d_reward, d_discount, d_flags, d_board, stream);
  if (rc) return rc;
  return cx_layers_from_board(g, d_board, (int64_t)T * n, d_layered, stream);
}

extern "C" int cx_rollout_policy(const cx_game* g, void* d_state, int64_t n, int32_t T, const float* d_w1t,
                                 const float* d_b1, int32_t n_hidden, const float* d_w2, const float* d_b2, uint64_t seed,
                                 uint64_t env_offset, const uint64_t* d_step, uint64_t step_offset, float* d_states,
                                 uint8_t* d_actions, float* d_reward, uint8_t* d_flags, float* d_logp, void* stream) {
  int rc = check_common(g, d_state, n, "cx_rollout_policy");
  if (rc) return rc;
  if (g->info.n_pickups) {
    cx_set_error("cx_rollout_policy: games with pickup drapes are not supported; use cx_policy_sample_board and "
                 "cx_step");
    return CX_ERR_UNSUPPORTED;
  }
  if (T < 1 || !d_w1t || !d_b1 || !d_w2 || !d_b2 || !d_states || !d_actions || !d_reward || !d_flags || n_hidden < 1 ||
      n_hidden > 32) {
    cx_set_error("cx_rollout_policy: bad argument (n_steps >= 1, n_hidden in 1..32, no NULL buffers)");
    return CX_ERR_INVALID_ARG;
  }
  return cx_launch_agent_policy_rollout(g, d_state, n, T, d_w1t, d_b1, n_hidden, d_w2, d_b2, seed, env_offset, d_step,
                                        step_offset, d_states, d_actions, d_reward, d_flags, d_logp, (cudaStream_t)stream);
}

extern "C" int cx_step(const cx_game* g, void* d_state, int64_t n, const uint8_t* d_actions, float* d_reward,
                       float* d_discount, uint8_t* d_flags, uint8_t* d_board, void* stream) {
  return cx_rollout(g, d_state, n, 1, d_actions, d_reward, d_discount, d_flags, d_board, stream);
}

extern "C" int cx_step_observations(const cx_game* g, void* d_state, int64_t n, const uint8_t* d_actions,
                                    float* d_reward, float* d_discount, uint8_t* d_flags, uint8_t* d_board,
                                    void* d_layered, int32_t dtype, void* stream) {
  int rc = check_common(g, d_state, n, "cx_step_observations");
  if (rc) return rc;
  if (!d_actions || !d_reward || !d_flags || !d_board || !d_layered) {
    cx_set_error("cx_step_observations: actions/reward/flags/board/layered must not be NULL");
    return CX_ERR_INVALID_ARG;
  }
  if (dtype != CX_DTYPE_U8 && dtype != CX_DTYPE_F32 && dtype != CX_DTYPE_BF16) {
    cx_set_error("cx_step_observations: unknown layered_dtype %d", dtype);
    return CX_ERR_INVALID_ARG;
  }
  CxRoute route;
  rc = parse_route(&route, "cx_step_observations");
  if (rc) return rc;
  if (route != CX_ROUTE_NO_STEP_COMPOSER && cx_agent_step_applies(g, d_board, d_layered))
    return cx_launch_agent_step(g, d_state, n, d_actions, d_reward, d_discount, d_flags, d_board, d_layered, dtype,
                                (cudaStream_t)stream);
  if (dtype == CX_DTYPE_U8)
    return cx_rollout_observations(g, d_state, n, 1, d_actions, d_reward, d_discount, d_flags, d_board,
                                   static_cast<uint8_t*>(d_layered), stream);
  if (g->desc.unoccluded_layers) {
    cx_set_error("cx_step_observations: unoccluded float planes need 16-byte aligned buffers");
    return CX_ERR_UNSUPPORTED;
  }
  if (dtype == CX_DTYPE_BF16) {
    cx_set_error("cx_step_observations: bfloat16 planes are emitted by the single-agent step kernel only "
                 "(16-byte aligned buffers); use CX_DTYPE_F32 for this game");
    return CX_ERR_UNSUPPORTED;
  }
  rc = cx_rollout(g, d_state, n, 1, d_actions, d_reward, d_discount, d_flags, d_board, stream);
  if (rc) return rc;
  return cx_layers_from_board_f32(g, d_board, n, static_cast<float*>(d_layered), stream);
}

extern "C" int cx_render_observations(const cx_game* g, const void* d_state, int64_t n, uint8_t* d_board,
                                      void* d_layered, int32_t dtype, void* stream) {
  int rc = check_common(g, d_state, n, "cx_render_observations");
  if (rc) return rc;
  if (!d_board || !d_layered || (dtype != CX_DTYPE_U8 && dtype != CX_DTYPE_F32 && dtype != CX_DTYPE_BF16)) {
    cx_set_error("cx_render_observations: board/layered must not be NULL, layered_dtype must be a cx_dtype");
    return CX_ERR_INVALID_ARG;
  }
  if (cx_agent_step_applies(g, d_board, d_layered))   // the composer with nothing to step
    return cx_launch_agent_step(g, const_cast<void*>(d_state), n, nullptr, nullptr, nullptr, nullptr, d_board, d_layered,
                                dtype, (cudaStream_t)stream);
  if (g->desc.unoccluded_layers && g->path == CX_PATH_GENERIC && dtype == CX_DTYPE_U8)
    return cx_launch_generic_render(g, d_state, n, d_board, (cudaStream_t)stream, static_cast<uint8_t*>(d_layered));
  if (g->desc.unoccluded_layers || dtype == CX_DTYPE_BF16) {
    cx_set_error("cx_render_observations: this game / element type needs the single-agent composer (16-byte aligned "
                 "buffers)");
    return CX_ERR_UNSUPPORTED;
  }
  rc = cx_launch_render(g, d_state, n, d_board, (cudaStream_t)stream);
  if (rc) return rc;
  return dtype == CX_DTYPE_U8 ? cx_layers_from_board(g, d_board, n, static_cast<uint8_t*>(d_layered), stream)
                              : cx_layers_from_board_f32(g, d_board, n, static_cast<float*>(d_layered), stream);
}

extern "C" int cx_get_entity_state(const cx_game* g, const void* d_state, int64_t n, int32_t z, int32_t* d_cells,
                                   void* stream) {
  int rc = check_common(g, d_state, n, "cx_get_entity_state");
  if (rc) return rc;
  if (z < 0 || z >= g->info.n_entities || !d_cells) {
    cx_set_error("cx_get_entity_state: bad z_index %d or NULL output", z);
    return CX_ERR_INVALID_ARG;
  }
  if (g->desc.entities[z].kind == CX_KIND_PICKUP || g->desc.entities[z].kind == CX_KIND_DOOR) {
    cx_set_error("cx_get_entity_state: entity %d is a pickup or door drape (its items, and with them the doors: "
                 "cx_get_pickups)", z);
    return CX_ERR_INVALID_ARG;
  }
  return cx_launch_get_entity(g, d_state, n, z, d_cells, (cudaStream_t)stream);
}

extern "C" int cx_set_entity_state(const cx_game* g, void* d_state, int64_t n, int32_t z, const int32_t* d_cells,
                                   void* stream) {
  int rc = check_common(g, d_state, n, "cx_set_entity_state");
  if (rc) return rc;
  if (z < 0 || z >= g->info.n_entities || !d_cells) {
    cx_set_error("cx_set_entity_state: bad z_index %d or NULL input", z);
    return CX_ERR_INVALID_ARG;
  }
  if (g->desc.entities[z].kind == CX_KIND_STATIC || g->desc.entities[z].kind == CX_KIND_PICKUP ||
      g->desc.entities[z].kind == CX_KIND_DOOR) {
    cx_set_error("cx_set_entity_state: entity %d is static, a pickup or a door drape", z);
    return CX_ERR_INVALID_ARG;
  }
  return cx_launch_set_entity(g, d_state, n, z, d_cells, (cudaStream_t)stream);
}

extern "C" int cx_get_episode_state(const cx_game* g, const void* d_state, int64_t n, int32_t* d_steps,
                                    float* d_returns, void* stream) {
  int rc = check_common(g, d_state, n, "cx_get_episode_state");
  if (rc) return rc;
  if (!g->info.tracks) {
    cx_set_error("cx_get_episode_state: this game keeps no per-env episode counters "
                 "(set max_episode_steps or track_returns)");
    return CX_ERR_INVALID_ARG;
  }
  return cx_launch_get_episode(g, d_state, n, d_steps, d_returns, (cudaStream_t)stream);
}

extern "C" int cx_get_episode_performance(const cx_game* g, const void* d_state, int64_t n, float* d_perf,
                                          void* stream) {
  int rc = check_common(g, d_state, n, "cx_get_episode_performance");
  if (rc) return rc;
  if (!g->info.tracks_performance) {
    cx_set_error("cx_get_episode_performance: this game tracks no performance (create it with perf_regions)");
    return CX_ERR_INVALID_ARG;
  }
  if (!d_perf) {
    cx_set_error("cx_get_episode_performance: d_perf is NULL");
    return CX_ERR_INVALID_ARG;
  }
  const CxStateLayout L = cx_layout(g, n);
  CX_CUDA_OK(cudaMemcpyAsync(d_perf, static_cast<const uint8_t*>(d_state) + L.off_perf, (size_t)n * sizeof(float),
                             cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return CX_OK;
}

extern "C" int cx_get_pickups(const cx_game* g, const void* d_state, int64_t n, uint64_t* d_bits, void* stream) {
  int rc = check_common(g, d_state, n, "cx_get_pickups");
  if (rc) return rc;
  if (!g->info.n_pickups || !d_bits) {
    cx_set_error("cx_get_pickups: the game has no pickup drapes, or d_bits is NULL");
    return CX_ERR_INVALID_ARG;
  }
  const CxStateLayout L = cx_layout(g, n);
  CX_CUDA_OK(cudaMemcpyAsync(d_bits, static_cast<const uint8_t*>(d_state) + L.off_pick, (size_t)n * sizeof(uint64_t),
                             cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return CX_OK;
}

extern "C" int cx_get_render_state(const cx_game* g, const void* d_state, int64_t n, uint32_t* d_zorder,
                                   uint32_t* d_visible, int32_t* d_backdrop_off, void* stream) {
  int rc = check_common(g, d_state, n, "cx_get_render_state");
  if (rc) return rc;
  return cx_launch_get_render_state(g, d_state, n, d_zorder, d_visible, d_backdrop_off, (cudaStream_t)stream);
}

extern "C" int cx_stats_fold(const cx_game* g, void* d_state, void* stream) {
  if (!g || !d_state) {
    cx_set_error("cx_stats_fold: NULL argument");
    return CX_ERR_INVALID_ARG;
  }
  return cx_launch_stats_fold(d_state, (cudaStream_t)stream);
}

extern "C" int cx_stats_read(const cx_game* g, const void* d_state, double* h_out, void* stream) {
  if (!g || !d_state || !h_out) {
    cx_set_error("cx_stats_read: NULL argument");
    return CX_ERR_INVALID_ARG;
  }
  cudaStream_t s = (cudaStream_t)stream;
  int rc = cx_launch_stats_fold(const_cast<void*>(d_state), s);   // the partial blocks are part of the statistics
  if (rc) return rc;
  CX_CUDA_OK(cudaMemcpyAsync(h_out, d_state, CX_STATS_DOUBLES * sizeof(double), cudaMemcpyDeviceToHost, s));
  CX_CUDA_OK(cudaStreamSynchronize(s));
  return CX_OK;
}
