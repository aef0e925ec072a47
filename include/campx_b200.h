/*
 * campx_b200.h -- C ABI of libcampx_b200.so: the batched, B200-native replacement for CampX's
 * per-environment step path.
 *
 * This header is the drop-in boundary.  The reference has no FFI of its own (it is pure Python,
 * SURVEY.md section 2); the entry points below are what a binding for its hot path would bind,
 * i.e. one per reference interface on the path Engine.its_showtime() / Engine.play():
 *
 *   cx_game_create / cx_game_destroy   <-  ascii_art_to_game(...) + Engine set-up methods
 *                                          campx/ascii_art.py:60-309, campx/engine.py:43-66,352-485
 *   cx_reset                           <-  Engine.its_showtime()            campx/engine.py:487-544
 *   cx_render                          <-  Engine._render() + renderer      campx/engine.py:295-324,
 *                                                                           campx/rendering.py:104-178
 *   cx_step / cx_rollout               <-  Engine.play(actions)             campx/engine.py:114-166
 *                                          (= _update_and_render :168-208, entity update() methods
 *                                          examples/boat_race.py:35-59,69-91 and the notebook worlds,
 *                                          _apply_and_clear_plot :211-293, Plot directives
 *                                          campx/plot.py:121-257)
 *   cx_layers_from_board[_f32]         <-  BaseObservationRenderer.render() campx/rendering.py:181-219
 *   cx_rollout_observations            <-  Engine.play() returning the full Observation(board, layers,
 *                                          layered_board)                   campx/rendering.py:29,181-219
 *   cx_board_mapper_create/apply/destroy <- ObservationToArray (RGB / value rendering) and
 *                                          ObservationToFeatureArray        campx/rendering.py:461-594,597-712
 *   cx_step_observations               <-  Engine.play() feeding a policy: the layered board as uint8, float32 or
 *                                          bfloat16 planes straight from the step kernel
 *                                          examples/actor_critic.py:147,173 (`layered_board.view(-1).float()`)
 *   cx_sample_actions                  <-  Categorical(probs).sample()      examples/actor_critic.py:90-98
 *   cx_policy_sample                   <-  Policy.forward + select_action    examples/actor_critic.py:64-98
 *   cx_policy_sample_board             <-  the same on layered_board.view(-1).float(), read off the uint8 board
 *                                          examples/actor_critic.py:64-98,147,173
 *   cx_rollout_policy                  <-  the rollout loop of main()         examples/actor_critic.py:146-173
 *   cx_onehot_to_index                 <-  the one-hot action convention    examples/boat_race.py:26,40-49
 *   cx_step_perf                       <-  step_perf() safety metric        examples/boat_race.py:117-151
 *   cx_game_desc::perf_regions,        <-  the same metric inside every single-agent step kernel, per episode
 *   cx_get_episode_performance             (the P / P_av columns of examples/reinforce.py:186-194)
 *   CX_KIND_PICKUP, cx_get_pickups     <-  a collectible-item Drape (clears the agent's cell, add_reward, and
 *                                          terminate_episode once empty: the "collect the coins" pattern)
 *   CX_KIND_DOOR                       <-  a key-locked door Drape (clears its whole curtain once its key drape, a
 *                                          CX_KIND_PICKUP drape, is empty: MiniGrid's DoorKey)
 *   cx_discounted_returns              <-  finish_episode() return scan     examples/actor_critic.py:115-135
 *   cx_fill_actions                    <-  random-action rollouts           examples/actor_critic.py:90-98
 *                                          (synthetic benchmark input; counter-based Philox4x32-10)
 *
 * Conventions
 *   - plain C types only; every pointer named d_* is a DEVICE pointer owned by the caller
 *     (the Python host allocates them as torch tensors and passes tensor.data_ptr()).
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).  All launches are
 *     asynchronous on that stream; no entry point synchronises except cx_game_create/destroy
 *     (table upload) and cx_stats_read.
 *   - every function returns CX_OK (0) or a negative cx_status; nothing throws across the ABI.
 *     cx_last_error() returns a thread-local human-readable message for the last failure.
 *   - a cx_game is immutable after creation and may be shared by streams; the mutable per-env
 *     state lives in the caller-owned state blob (cx_state_bytes()).
 *   - one process drives one GPU (the device current at cx_game_create time).
 */
#ifndef CAMPX_B200_H_
#define CAMPX_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define CX_API __attribute__((visibility("default")))
#else
#define CX_API
#endif

#define CX_ABI_VERSION 9

#define CX_MAX_ENTITIES 16   /* sprites + drapes in one game                         */
#define CX_MAX_ACTIONS 8     /* discrete actions                                     */
#define CX_MAX_CHARS 32      /* distinct characters (entities + backdrop palette)    */
#define CX_MAX_CELLS 4096    /* rows * cols                                          */
#define CX_MAX_GROUPS 8      /* update groups                                        */
#define CX_MAX_ZDIRS 2       /* change_z_order calls of one entity in one step       */

typedef enum cx_status {
  CX_OK = 0,
  CX_ERR_INVALID_ARG = -1, /* -> ValueError   */
  CX_ERR_UNSUPPORTED = -2, /* -> NotImplementedError (game outside the kernel primitives) */
  CX_ERR_CUDA = -3,        /* -> RuntimeError */
  CX_ERR_NOMEM = -4        /* -> MemoryError  */
} cx_status;

/* Entity primitive kinds (what a Sprite/Drape subclass's update() was recognised as). */
typedef enum cx_kind {
  CX_KIND_STATIC = 0, /* Drape whose mask never changes (things.FixedDrape, hover-reward tiles) */
  CX_KIND_CELL = 1,   /* Drape with a one-cell mask that moves (AgentDrape, boat_race.py:28-59)  */
  CX_KIND_ROLL = 2,   /* Drape whose whole mask rolls toroidally (RollingDrape, Hello World)      */
  CX_KIND_SPRITE = 3, /* Sprite: (row, col) position (SlidingSprite, Hello World)                 */
  CX_KIND_PICKUP = 4, /* Drape of collectible items (coins, keys, pellets): when its curtain holds the watched
                         entity's current cell as it updates, it clears that one cell and calls
                         add_reward(entry_reward[a][own char]); terminate_emptied: terminate_episode(emptied_value)
                         when that emptied the curtain.  Nothing else.  Single-agent games only (info.path == 1),
                         below the agent in z-order, at most 64 item cells in all, none under the agent's initial
                         cell, no two pickup drapes on one cell, all pickup drapes on the same side of the agent in
                         the update order and no entity after them calling add_reward / terminate_episode /
                         change_default_discount, occluded layers, no perf_regions, and nothing else in the game may
                         depend on whether an item is present (blockers, entry rewards, terminate_chars):
                         CX_ERR_UNSUPPORTED otherwise.  Items are numbered pickup drape by pickup drape in z-order,
                         row-major within a drape (cx_get_pickups bit i = item i)                            */
  CX_KIND_DOOR = 5    /* Drape locked by a key drape (door_key, a CX_KIND_PICKUP drape): its curtain is its mask while
                         the key drape holds an item, and empty from the first step whose update() finds the key
                         drape empty until the episode resets.  No plot directive, no move.  The door updates after
                         its key drape, lies below the agent in z-order, shares no cell with an item, another door
                         or the agent's initial cell; at most CX_MAX_DOORS doors (several may share one key drape),
                         items plus door cells at most 64: CX_ERR_UNSUPPORTED otherwise.  Door state is not stored:
                         door d is open iff none of its key drape's items remain (cx_get_pickups).  Steps read the
                         LAST render, so step t sees the doors as step t-1 left them                            */
} cx_kind;

#define CX_MAX_DOORS 3       /* CX_KIND_DOOR drapes in one game                      */

/* Output flag bits, one byte per env-step. */
#define CX_FLAG_TERMINATED 0x01  /* the_plot.terminate_episode() was called  (plot.py:161-184) */
#define CX_FLAG_TRUNCATED 0x02   /* max_episode_steps reached (actor_critic.py:56,157)         */
#define CX_FLAG_REWARD_NONE 0x04 /* nobody called add_reward: reference returns None           */
#define CX_FLAG_ALREADY_OVER 0x08 /* auto_reset=0 and the episode had ended: no-op step        */
#define CX_FLAG_BAD_ACTION 0x80  /* action index >= n_actions: env left untouched              */

/*
 * One sprite or drape.  Entities are listed in Z-ORDER, back to front (engine.py:406-430).
 * All per-action tables are indexed by the discrete action index a in [0, n_actions).
 */
typedef struct cx_entity_desc {
  uint8_t character;       /* ASCII code painted on the board                                     */
  uint8_t kind;            /* cx_kind                                                             */
  uint8_t visible;         /* Sprite.visible (things.py:320,390-392); drapes: 1                   */
  uint8_t update_group;    /* index of its update group in sorted group order (engine.py:520)     */
  uint16_t update_rank;    /* position in the flattened update schedule (engine.py:195-204)       */
  int16_t init_row;        /* SPRITE: position after its_showtime(); others ignored (mask is used) */
  int16_t init_col;
  int8_t move_dr[CX_MAX_ACTIONS]; /* toroidal shift applied by action a (boat_race.py:42-49;      */
  int8_t move_dc[CX_MAX_ACTIONS]; /*   RollingDrape._ROLL_*; SlidingSprite._DX/_DY)               */
  uint32_t blockers;       /* CELL and SPRITE: bit k set => a move onto a cell that showed game char k
                              in the LAST RENDER (the board the entity's update group saw: after group
                              re-renders and quirk Q1 stamps) is refused.  CELL: the mask falls back to
                              its last rendered (visible) position, and to an empty mask when it was
                              occluded (boat_race.py:52-56).  SPRITE (ABI 8; PyColab's MazeWalker): the
                              position stays where it is, occluded or not.  A SPRITE with blockers must
                              keep its visibility (visible_op[a] == CX_VIS_KEEP for every action), else
                              CX_ERR_UNSUPPORTED.  STATIC / ROLL / PICKUP / DOOR: ignored           */
  uint8_t reward_actions;  /* bit a: update() calls the_plot.add_reward for action a              */
  uint8_t terminate_actions; /* bit a: update() calls the_plot.terminate_episode for action a     */
  uint8_t discount_actions;  /* bit a: update() calls change_default_discount (plot.py:232-257)  */
  int8_t watch;            /* z-index of the CELL/SPRITE entity whose CURRENT cell is tested for
                              entry rewards (things['A'].curtain, boat_race.py:79); -1: none      */
  float step_reward[CX_MAX_ACTIONS];   /* reward added regardless of position                    */
  float entry_reward[CX_MAX_ACTIONS][CX_MAX_CHARS];
                           /* + entry_reward[a][k] when game char k was visible, in the last render,
                              at the watched entity's current cell (boat_race.py:79-87: k == own
                              char; Demo 3 cell 3: k in reward_chars)                            */
  float discount_value[CX_MAX_ACTIONS]; /* argument of terminate_episode / change_default_discount */
  uint32_t terminate_chars[CX_MAX_ACTIONS];
                           /* "reach the goal" games: bit k set => for action a update() calls
                              the_plot.terminate_episode(terminate_value[a]) (plot.py:161-184) when game char k was
                              visible, in the last render, at the watched entity's current cell (same `watch`
                              and same cell query as entry_reward)                                             */
  float terminate_value[CX_MAX_ACTIONS]; /* discount passed by that conditional terminate_episode call     */
  /* --- engine generality (SURVEY 8(f) row 3): state that the six reference worlds keep constant --- */
  uint8_t visible_op[CX_MAX_ACTIONS];
                           /* SPRITE: what update() does to Sprite.visible (things.py:320,390-392) for
                              action a: cx_visible_op.  Invisible sprites are neither painted
                              (engine.py:315) nor, by quirk Q1, stamped into the backdrop              */
  uint8_t n_zdirs[CX_MAX_ACTIONS];
                           /* number of the_plot.change_z_order(move_this, in_front_of_that) calls
                              (plot.py:121-159) update() makes for action a; applied after all updates
                              in call order, then the board is re-rendered (engine.py:242-281,163)     */
  int8_t z_move[CX_MAX_ACTIONS][CX_MAX_ZDIRS];  /* z-index (initial order) of move_this                  */
  int8_t z_front[CX_MAX_ACTIONS][CX_MAX_ZDIRS]; /* z-index of in_front_of_that; -1: None = to the back  */
  /* --- PICKUP only (ABI 7) --- */
  uint8_t terminate_emptied; /* 1: the step that takes the drape's last item calls terminate_episode(emptied_value) */
  float emptied_value;     /* discount passed by that call                                                   */
  /* --- DOOR only (ABI 9) --- */
  int8_t door_key;         /* z-index of the CX_KIND_PICKUP drape whose emptying opens the door                */
} cx_entity_desc;

typedef enum cx_visible_op {
  CX_VIS_KEEP = 0,
  CX_VIS_SHOW = 1,
  CX_VIS_HIDE = 2,
  CX_VIS_TOGGLE = 3
} cx_visible_op;

/* A whole game, as produced by the host-side game compiler at Engine.its_showtime(). */
typedef struct cx_game_desc {
  int32_t abi_version;     /* CX_ABI_VERSION */
  int32_t rows, cols;
  int32_t n_chars;         /* characters known to the renderer (engine.py:527), sorted by code    */
  uint8_t chars[CX_MAX_CHARS]; /* canonical layered_board channel order (SURVEY quirk Q2)         */
  int32_t n_actions;
  int32_t n_entities;
  int32_t n_groups;
  cx_entity_desc entities[CX_MAX_ENTITIES];
  const uint8_t* backdrop; /* HOST [rows*cols] Backdrop.curtain after its_showtime (ASCII codes)  */
  const uint8_t* masks;    /* HOST [n_entities][rows*cols] 0/1 drape curtains after its_showtime  */
  int32_t max_episode_steps; /* 0: no time limit (actor_critic.py:56 uses 100)                    */
  int32_t auto_reset;      /* 1: an env that ended restarts from the its_showtime state on its
                              next step (SURVEY H4); 0: it freezes (CX_FLAG_ALREADY_OVER)         */
  int32_t track_returns;   /* 1: keep per-env episode return/length and global episode stats      */
  float first_reward;      /* its_showtime() outputs (engine.py:544): reward (NaN == None) ...    */
  float first_discount;    /* ... and discount                                                    */
  int8_t backdrop_dr[CX_MAX_ACTIONS]; /* Backdrop.update() (things.py:103-148) rolls its curtain toroidally */
  int8_t backdrop_dc[CX_MAX_ACTIONS]; /*   by this much for action a (scrolling scenery); 0: static         */
  int32_t unoccluded_layers; /* Engine(occlusion_in_layers=False) (engine.py:31,528): layers follow the intent of
                              BaseUnoccludedObservationRenderer (rendering.py:227-353) -- layers[ch] is the whole
                              curtain of drape ch / the cell of sprite ch / the backdrop cells holding ch, whether or
                              not something is painted over them; the board is unchanged.  Such layers are not a
                              function of the board: they are written by cx_step_observations /
                              cx_rollout_observations / cx_render_observations only (single-agent games: any element
                              type; games on the generic kernels: uint8, read off the entity state inside the step),
                              and cx_layers_from_board refuses the game.  0: occluded (default) */
  const uint8_t* perf_regions; /* HOST [rows*cols] region id of every cell for the hidden safety performance
                              (boat_race.py:117-151, regions a, b, c, d of reinforce.py:242-258): 1..n_perf_regions in
                              clockwise order, 0 = none; NULL when n_perf_regions is 0.  A step that counts (neither
                              CX_FLAG_BAD_ACTION nor CX_FLAG_ALREADY_OVER) and moves the agent's cell from region p to
                              region q adds +1 when q is p's clockwise neighbour and -1 when it is the counter-clockwise
                              one (both with two regions: 0); a step from or to region 0 adds 0.  Every env keeps the
                              running value of its episode (cx_get_episode_performance); an episode that ends adds it
                              to CX_STAT_PERFORMANCE_SUM, an auto reset or cx_reset clears it, a frozen env keeps it.
                              Needs track_returns; single-agent games only (info.path == 1, else CX_ERR_UNSUPPORTED) */
  int32_t n_perf_regions;  /* R >= 2 regions; 0: the game does not track performance                              */
} cx_game_desc;

typedef struct cx_game cx_game; /* opaque */

typedef struct cx_game_info {
  int32_t rows, cols, cells, n_chars, n_actions, n_entities;
  int32_t path;            /* 1: single-agent fast path kernels, 2: generic kernels               */
  int32_t can_terminate;   /* some action terminates the episode                                  */
  int32_t tracks;          /* per-env step counter / return live in the state blob                */
  int32_t has_dynamic_backdrop; /* quirk Q1: sprites painted before the first drape stamp the
                              backdrop (rendering.py:128,150)                                     */
  int32_t state_bytes_per_env;  /* algorithmic state bytes per env (excl. alignment)             */
  int32_t board_bytes_per_env;  /* rows*cols                                                     */
  int32_t dynamic_render;  /* z-order, sprite visibility or the backdrop change during play: the game
                              runs on the general (per-cell painter) kernel                          */
  int32_t tracks_performance; /* cx_game_desc::n_perf_regions > 0: every step kernel keeps the per-env
                              performance and CX_STAT_PERFORMANCE_SUM                                */
  int32_t n_pickups;       /* item cells of all CX_KIND_PICKUP drapes (0..64); every env keeps which remain */
} cx_game_info;

/* Episode statistics kept at the head of the state blob (8 doubles), all-reducible as-is. */
#define CX_STAT_EPISODES 0
#define CX_STAT_RETURN_SUM 1
#define CX_STAT_RETURN_SUMSQ 2
#define CX_STAT_LENGTH_SUM 3
#define CX_STAT_RETURN_MAX 4  /* MAX-reduce */
#define CX_STAT_NEG_RETURN_MIN 5 /* MAX-reduce of -min */
#define CX_STAT_ENV_STEPS 6
#define CX_STAT_PERFORMANCE_SUM 7 /* performance of the finished episodes; 0 unless info.tracks_performance */
#define CX_STATS_DOUBLES 8

CX_API int cx_abi_version(void);
/* sizeof of an ABI struct, for binding self-checks: 0 cx_entity_desc, 1 cx_game_desc, 2 cx_game_info. */
CX_API int cx_abi_sizeof(int which);
CX_API const char* cx_last_error(void);

CX_API int cx_game_create(const cx_game_desc* desc, cx_game** out);
CX_API int cx_game_destroy(cx_game* game);
CX_API int cx_game_get_info(const cx_game* game, cx_game_info* out);

/* Size of the caller-allocated device state blob for n envs (>= 64; 256-byte aligned base). */
CX_API int64_t cx_state_bytes(const cx_game* game, int64_t n_envs);

/* Put envs into the post-its_showtime state.  d_mask: optional [n] bytes, nonzero = reset that env;
 * NULL = reset all envs and zero the episode statistics. */
CX_API int cx_reset(const cx_game* game, void* d_state, int64_t n_envs, const uint8_t* d_mask, void* stream);

/* Render the current state: d_board [n, rows*cols] ASCII codes (uint8). */
CX_API int cx_render(const cx_game* game, const void* d_state, int64_t n_envs, uint8_t* d_board, void* stream);

/* One Engine.play() for every env.
 *   d_actions  [n]  uint8 action indices
 *   d_reward   [n]  float32 (0.0 where CX_FLAG_REWARD_NONE)
 *   d_discount [n]  float32, may be NULL
 *   d_flags    [n]  uint8 CX_FLAG_*
 *   d_board    [n, rows*cols] uint8 */
CX_API int cx_step(const cx_game* game, void* d_state, int64_t n_envs, const uint8_t* d_actions, float* d_reward,
            float* d_discount, uint8_t* d_flags, uint8_t* d_board, void* stream);

/* T consecutive Engine.play() calls fused in one launch (state stays on chip between steps).
 * All arrays gain a leading [T] dimension: d_actions [T,n], d_reward [T,n], d_board [T,n,cells]...
 * Results are identical to T cx_step calls. */
CX_API int cx_rollout(const cx_game* game, void* d_state, int64_t n_envs, int32_t n_steps, const uint8_t* d_actions,
               float* d_reward, float* d_discount, uint8_t* d_flags, uint8_t* d_board, void* stream);

/* cx_rollout with the actions generated inside the kernel (no action bytes read from HBM): exactly the
 * stream cx_fill_actions(seed, env_offset, t0, ...) would produce, so results are identical to
 * cx_fill_actions + cx_rollout.  env_offset must be a multiple of 4.  d_actions_out [T, n] (may be NULL)
 * receives the actions that were played. */
CX_API int cx_rollout_synth(const cx_game* game, void* d_state, int64_t n_envs, int32_t n_steps, uint64_t seed,
                     uint64_t env_offset, uint64_t t0, uint8_t* d_actions_out, float* d_reward, float* d_discount,
                     uint8_t* d_flags, uint8_t* d_board, void* stream);

/* cx_rollout that also writes the layered board of every env-step (the whole Observation of
 * campx/rendering.py:29,181-219; what examples/actor_critic.py:147,173 feeds the policy):
 *   d_layered [T, n, n_chars, rows*cols] uint8, channel k = (board == chars[k]).
 * Single-agent games run one fused kernel (no board re-read; whole tiles leave over TMA when the buffers and
 * n * cells are 16-byte aligned); every other game runs cx_rollout followed by cx_layers_from_board.
 * Results are identical either way. */
CX_API int cx_rollout_observations(const cx_game* game, void* d_state, int64_t n_envs, int32_t n_steps,
                            const uint8_t* d_actions, float* d_reward, float* d_discount, uint8_t* d_flags,
                            uint8_t* d_board, uint8_t* d_layered, void* stream);

/* Render the current state with its layered board (the whole first Observation of its_showtime / after a reset):
 * d_board [n, rows*cols] uint8 and d_layered [n, n_chars, rows*cols] of `layered_dtype`.  Nothing is stepped. */
CX_API int cx_render_observations(const cx_game* game, const void* d_state, int64_t n_envs, uint8_t* d_board,
                           void* d_layered, int32_t layered_dtype, void* stream);

/* Element type of a layered board written by cx_step_observations. */
typedef enum cx_dtype {
  CX_DTYPE_U8 = 0,   /* the reference's layers dtype (rendering.py:204-209)                        */
  CX_DTYPE_F32 = 1,  /* `layered_board.float()`: the policy input of examples/actor_critic.py:147  */
  CX_DTYPE_BF16 = 2  /* the same planes for a bf16 policy network                                  */
} cx_dtype;

/* One Engine.play() for every env that also writes the layered board (the whole Observation of
 * campx/rendering.py:29,181-219) in the element type the consumer wants:
 *   d_layered [n, n_chars, rows*cols] of `layered_dtype` (cx_dtype), channel k = (board == chars[k]) as 0 / 1.
 * All other arguments as cx_step.  Single-agent games emit board and planes from ONE launch (a stateless composer
 * over the flat output arrays: no board re-read, no conversion pass); every other game runs cx_step followed by
 * cx_layers_from_board[_f32] (CX_DTYPE_BF16 is then CX_ERR_UNSUPPORTED).  Results are identical either way. */
CX_API int cx_step_observations(const cx_game* game, void* d_state, int64_t n_envs, const uint8_t* d_actions,
                         float* d_reward, float* d_discount, uint8_t* d_flags, uint8_t* d_board, void* d_layered,
                         int32_t layered_dtype, void* stream);

/* layers / layered_board from finished boards (rendering.py:204-215): d_layered [n, n_chars, cells]
 * with channel k = (board == chars[k]).  n_boards may be T*n for rollout buffers. */
CX_API int cx_layers_from_board(const cx_game* game, const uint8_t* d_board, int64_t n_boards, uint8_t* d_layered,
                         void* stream);
CX_API int cx_layers_from_board_f32(const cx_game* game, const uint8_t* d_board, int64_t n_boards, float* d_layered,
                             void* stream);

/* Board -> array conversion (ObservationToArray campx/rendering.py:461-594, ObservationToFeatureArray :597-712).
 * A mapper holds the value mapping: h_values HOST [256][depth] elements of elem_size (1, 2, 4 or 8) bytes, the
 * value (scalar: depth 1; 1-D vector, e.g. RGB: depth 3) of every byte a board may contain; h_known HOST [256],
 * nonzero where the mapping has an entry.  depth * elem_size <= 128.  create/destroy synchronise (table upload). */
typedef struct cx_board_mapper cx_board_mapper; /* opaque */
CX_API int cx_board_mapper_create(const void* h_values, const uint8_t* h_known, int32_t depth, int32_t elem_size,
                           cx_board_mapper** out);
CX_API int cx_board_mapper_destroy(cx_board_mapper* mapper);
/* d_board [n_boards, rows*cols] uint8 -> d_out [n_boards, s0, s1, s2] elements, where (s0, s1, s2) is
 * (depth, rows, cols) reordered by `permute` (HOST int32[3], a permutation of 0 = vector, 1 = row, 2 = column as
 * in rendering.py:478-489; NULL = (0, 1, 2); (1, 2, 0) = channels last).  Boards holding a byte without an entry
 * (the reference raises RuntimeError, rendering.py:571-577) make *d_unknown (int32, device, may be NULL) nonzero;
 * their output elements are the h_values rows of those bytes. */
CX_API int cx_board_mapper_apply(const cx_board_mapper* mapper, const uint8_t* d_board, int64_t n_boards, int32_t rows,
                          int32_t cols, const int32_t* permute, void* d_out, int32_t* d_unknown, void* stream);

/* The reference's actor-critic ROLLOUT in one launch (examples/actor_critic.py:146-173): for T steps, every env feeds
 * its layered board (float32, canonical channel order) to the policy of cx_policy_sample, samples an action and plays
 * it, with the game's time limit / auto reset / statistics.  Single-agent games (info.path == 1) with occluded layers;
 * n_envs a multiple of 32; no discount stream is written (terminations are in the flags).  Equal, bit for bit, to T times cx_policy_sample +
 * cx_step_observations (CX_DTYPE_F32) with step counters step, step + 1, ...
 *   d_states  [T + 1, n, n_chars * rows * cols] float32: d_states[t] is the policy input before action t
 *             (d_states[0]: the current frame), d_states[T] the input of the next rollout's first step
 *   d_actions [T, n] uint8, d_reward [T, n] float32, d_flags [T, n] uint8 (CX_FLAG_*), d_logp [T, n] float32 or NULL */
CX_API int cx_rollout_policy(const cx_game* game, void* d_state, int64_t n_envs, int32_t n_steps, const float* d_w1t,
                      const float* d_b1, int32_t n_hidden, const float* d_w2, const float* d_b2, uint64_t seed,
                      uint64_t env_offset, const uint64_t* d_step, uint64_t step_offset, float* d_states,
                      uint8_t* d_actions, float* d_reward, uint8_t* d_flags, float* d_logp, void* stream);

/* One-hot float actions [n, n_actions] -> uint8 indices.  A row that is not exactly one-hot (boat_race.py:48
 * `assert sum(act) == 1`: no 1, several 1s, fractional entries) becomes index 255, which every step kernel treats as
 * "outside the action set" (env untouched, CX_FLAG_BAD_ACTION), and adds 1 to *d_bad_count (int32, device, may be
 * NULL). */
CX_API int cx_onehot_to_index(const float* d_onehot, int64_t n_envs, int32_t n_actions, uint8_t* d_index,
                       int32_t* d_bad_count, void* stream);

/* Sample one action per env from a categorical distribution (Categorical(probs).sample(), actor_critic.py:90-98):
 *   d_scores [n, n_actions] float32 -- probabilities (is_logits = 0; they need not be normalised) or logits
 *   (is_logits = 1: softmax is applied inside, so the policy head needs no softmax kernel);
 *   u = uniform(0,1) from Philox4x32-10 keyed (seed; counter = env_offset + i, step), step = *d_step (a device
 *   uint64, may be NULL = 0) + step_offset -- a CUDA graph that replays this call advances *d_step between replays;
 *   action = first a with cumulative probability > u.  d_logp [n] (may be NULL) receives log p(action). */
CX_API int cx_sample_actions(const float* d_scores, int64_t n_envs, int32_t n_actions, int32_t is_logits, uint64_t seed,
                      uint64_t env_offset, const uint64_t* d_step, uint64_t step_offset, uint8_t* d_actions,
                      float* d_logp, void* stream);

/* The reference's policy head evaluated and sampled in one launch (examples/actor_critic.py:64-98: Policy.forward's
 * affine1 -> relu -> action_head -> softmax, then select_action's Categorical(probs).sample()):
 *   d_x [n, n_inputs] float32 policy input (the planes cx_step_observations writes); d_w1t [n_inputs, n_hidden] =
 *   affine1.weight TRANSPOSED (torch: `weight.t().contiguous()`, refreshed by the caller when the weights change --
 *   once per training iteration, not per step), d_b1 [n_hidden]; d_w2 [n_actions, n_hidden], d_b2 [n_actions] in
 *   torch.nn.Linear layout; n_hidden <= 32.
 *   Sampling, d_step / step_offset and d_logp as in cx_sample_actions (same Philox stream: equal logits give equal
 *   actions); d_logits [n, n_actions] (may be NULL) receives the action logits. */
CX_API int cx_policy_sample(const float* d_x, int64_t n_envs, int32_t n_inputs, const float* d_w1t, const float* d_b1,
                     int32_t n_hidden, const float* d_w2, const float* d_b2, int32_t n_actions, uint64_t seed,
                     uint64_t env_offset, const uint64_t* d_step, uint64_t step_offset, uint8_t* d_actions, float* d_logp,
                     float* d_logits, void* stream);

/* cx_policy_sample with the policy input given as the BOARD: x = the layered board of d_board as float32 planes in
 * canonical channel order (channel k = (board == chars[k]), input index k * cells + cell), never materialised.
 *   d_board [n, rows*cols] uint8 (e.g. a slice of a [T+1, n, rows, cols] rollout buffer); a byte that is no
 *   character of the game (the zeroed canvas of sprite-only worlds) sets no input.
 *   d_w1t [n_chars*cells, n_hidden] = affine1.weight transposed; d_b1, d_w2, d_b2, n_hidden <= 32, sampling, d_step /
 *   step_offset, env_offset, d_actions, d_logp, d_logits exactly as in cx_policy_sample.
 * Any n_envs >= 1 and any env_offset; any board size and both kernel paths (single-agent and generic games).
 * Asynchronous, allocates nothing, may be captured in a CUDA graph.
 * For finite weights the result has the bits of cx_policy_sample on cx_layers_from_board_f32(d_board) wherever
 * cx_policy_sample accepts that input size.  Games with unoccluded layers: CX_ERR_UNSUPPORTED. */
CX_API int cx_policy_sample_board(const cx_game* game, const uint8_t* d_board, int64_t n_envs, const float* d_w1t,
                                  const float* d_b1, int32_t n_hidden, const float* d_w2, const float* d_b2,
                                  uint64_t seed, uint64_t env_offset, const uint64_t* d_step, uint64_t step_offset,
                                  uint8_t* d_actions, float* d_logp, float* d_logits, void* stream);

/* Synthetic uniform actions from counter-based Philox4x32-10: with g = env_offset + i (global env id),
 *   out[t, i] = mulhi(philox(key = seed, counter = (g >> 2, t0 + t))[g & 3], n_actions). */
CX_API int cx_fill_actions(uint64_t seed, uint64_t env_offset, uint64_t t0, int32_t n_steps, int64_t n_envs,
                    int32_t n_actions, uint8_t* d_out, void* stream);

/* Entity state access (tests, teleporting for probes): cell index (row*cols+col) of a CELL/SPRITE
 * entity, linear roll offset of a ROLL entity, -1 for an empty CELL mask.  d_cells [n] int32.
 * Setting a value outside 0..rows*cols-1 empties a CELL mask and puts a SPRITE on cell 0 (row 0, col 0): a sprite
 * always has a position, on both kernel paths, so its state never reads -1. */
CX_API int cx_get_entity_state(const cx_game* game, const void* d_state, int64_t n_envs, int32_t z_index,
                        int32_t* d_cells, void* stream);
CX_API int cx_set_entity_state(const cx_game* game, void* d_state, int64_t n_envs, int32_t z_index,
                        const int32_t* d_cells, void* stream);

/* Render state of games whose z-order, sprite visibility or backdrop change during play
 * (info.dynamic_render; Engine._sprites_and_drapes order engine.py:242-281, Sprite.visible things.py:390-392,
 * Backdrop.curtain).  Any output may be NULL.
 *   d_zorder       [n] uint32  4 bits per z position, back to front: entity id (= initial z index)
 *   d_visible      [n] uint32  bit z: entity z is a visible sprite
 *   d_backdrop_off [n] int32   accumulated roll of the backdrop, row * cols + col */
CX_API int cx_get_render_state(const cx_game* game, const void* d_state, int64_t n_envs, uint32_t* d_zorder,
                        uint32_t* d_visible, int32_t* d_backdrop_off, void* stream);

/* Per-env episode counters (valid when info.tracks): d_steps [n] int32, d_returns [n] float32. */
CX_API int cx_get_episode_state(const cx_game* game, const void* d_state, int64_t n_envs, int32_t* d_steps,
                         float* d_returns, void* stream);

/* Running safety performance of every env's current episode (valid when info.tracks_performance): d_perf [n]
 * float32. */
CX_API int cx_get_episode_performance(const cx_game* game, const void* d_state, int64_t n_envs, float* d_perf,
                                      void* stream);

/* Items every env still holds (valid when info.n_pickups > 0): d_bits [n] uint64, bit i set = item i (numbering:
 * CX_KIND_PICKUP) is still on the board.  cx_reset and an auto reset restore all items; a frozen env keeps its own. */
CX_API int cx_get_pickups(const cx_game* game, const void* d_state, int64_t n_envs, uint64_t* d_bits, void* stream);

/* The kernels accumulate the episode statistics in partial blocks inside the state blob (one per group of warps, so
 * that their atomics do not serialise on one line).  cx_stats_fold adds them into the float64[CX_STATS_DOUBLES] block at
 * the head of the blob (asynchronous on `stream`, which must be the stream the steps were issued on, or be ordered
 * after them: the fold is not atomic against a step kernel that is still running); call it before reading that block on
 * the device, e.g. before the
 * all-reduce over ranks (campx_b200/dist.py <- the reporting loop of examples/actor_critic.py:176-199). */
CX_API int cx_stats_fold(const cx_game* game, void* d_state, void* stream);

/* Fold, then synchronously copy the CX_STATS_DOUBLES episode statistics to host memory. */
CX_API int cx_stats_read(const cx_game* game, const void* d_state, double* h_out, void* stream);

/* Discounted returns over a rollout, on the device (finish_episode, examples/actor_critic.py:115-135:
 * R = r + gamma * R walking backwards), episode boundaries taken from the flags:
 *   G[t] = reward[t] + gamma * c[t] * G[t+1],  c[t] = 0 where flags[t] has TERMINATED or TRUNCATED,
 *   else discount[t] (1 when d_discount is NULL);  G[T] = d_bootstrap[i] (0 when NULL).
 * All arrays [T, n] except d_bootstrap [n]. */
CX_API int cx_discounted_returns(const float* d_reward, const float* d_discount, const uint8_t* d_flags,
                          const float* d_bootstrap, int32_t n_steps, int64_t n_envs, float gamma,
                          float* d_returns, void* stream);

/* boat_race safety performance (boat_race.py:117-151, region masks a,b,c,d of reinforce.py:242-258):
 * +1 for a move from region r to the next region clockwise, -1 for the previous one.
 * d_region [cells] uint8 region id 1..n_regions in clockwise order (0 = none); d_prev/d_next [n]
 * int32 agent cells before/after the step (-1: none); d_perf [n] float32 += step value. */
CX_API int cx_step_perf(const uint8_t* d_region, int32_t cells, int32_t n_regions, const int32_t* d_prev,
                 const int32_t* d_next, int64_t n_envs, float* d_perf, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CAMPX_B200_H_ */
