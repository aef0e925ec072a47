"""ctypes binding of libcampx_b200.so (the C ABI declared in include/campx_b200.h).

There is NO CPU fallback: if the shared library is missing, or no CUDA device is present when a
compute entry point is needed, this module raises.  The library is built in-tree by
`__graft_entry__.build()` / `make -C campx_b200/csrc` into `campx_b200/lib/`.
"""
import ctypes
import os

CX_ABI_VERSION = 9
CX_MAX_ENTITIES = 16
CX_MAX_ACTIONS = 8
CX_MAX_CHARS = 32
CX_MAX_CELLS = 4096
CX_MAX_GROUPS = 8
CX_MAX_ZDIRS = 2

CX_OK = 0
CX_ERR_INVALID_ARG = -1
CX_ERR_UNSUPPORTED = -2
CX_ERR_CUDA = -3
CX_ERR_NOMEM = -4

CX_KIND_STATIC, CX_KIND_CELL, CX_KIND_ROLL, CX_KIND_SPRITE, CX_KIND_PICKUP, CX_KIND_DOOR = 0, 1, 2, 3, 4, 5
CX_MAX_PICKUPS = 64          # item cells of all pickup drapes of one game (door games: items plus door cells)
CX_MAX_DOORS = 3             # door drapes of one game
CX_VIS_KEEP, CX_VIS_SHOW, CX_VIS_HIDE, CX_VIS_TOGGLE = 0, 1, 2, 3

CX_FLAG_TERMINATED = 0x01
CX_FLAG_TRUNCATED = 0x02
CX_FLAG_REWARD_NONE = 0x04
CX_FLAG_ALREADY_OVER = 0x08
CX_FLAG_BAD_ACTION = 0x80

CX_DTYPE_U8, CX_DTYPE_F32, CX_DTYPE_BF16 = 0, 1, 2

CX_STATS_DOUBLES = 8
STAT_NAMES = ("episodes", "return_sum", "return_sumsq", "length_sum", "return_max", "neg_return_min",
              "env_steps", "reserved")
CX_STAT_PERFORMANCE_SUM = 7   # slot 7: "performance_sum" for games that track performance, else "reserved" (always 0)
STAT_NAMES_PERFORMANCE = STAT_NAMES[:CX_STAT_PERFORMANCE_SUM] + ("performance_sum",)

CX_PATH_AGENT, CX_PATH_GENERIC = 1, 2

LIB_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib")
LIB_PATH = os.environ.get("CAMPX_B200_LIB") or os.path.join(LIB_DIR, "libcampx_b200.so")   # env: development knob


class NativeLibraryError(RuntimeError):
    """The CUDA library is not built / not loadable.  There is deliberately no fallback path."""


class EntityDesc(ctypes.Structure):
    _fields_ = [
        ("character", ctypes.c_uint8),
        ("kind", ctypes.c_uint8),
        ("visible", ctypes.c_uint8),
        ("update_group", ctypes.c_uint8),
        ("update_rank", ctypes.c_uint16),
        ("init_row", ctypes.c_int16),
        ("init_col", ctypes.c_int16),
        ("move_dr", ctypes.c_int8 * CX_MAX_ACTIONS),
        ("move_dc", ctypes.c_int8 * CX_MAX_ACTIONS),
        ("blockers", ctypes.c_uint32),
        ("reward_actions", ctypes.c_uint8),
        ("terminate_actions", ctypes.c_uint8),
        ("discount_actions", ctypes.c_uint8),
        ("watch", ctypes.c_int8),
        ("step_reward", ctypes.c_float * CX_MAX_ACTIONS),
        ("entry_reward", (ctypes.c_float * CX_MAX_CHARS) * CX_MAX_ACTIONS),
        ("discount_value", ctypes.c_float * CX_MAX_ACTIONS),
        ("terminate_chars", ctypes.c_uint32 * CX_MAX_ACTIONS),
        ("terminate_value", ctypes.c_float * CX_MAX_ACTIONS),
        ("visible_op", ctypes.c_uint8 * CX_MAX_ACTIONS),
        ("n_zdirs", ctypes.c_uint8 * CX_MAX_ACTIONS),
        ("z_move", (ctypes.c_int8 * CX_MAX_ZDIRS) * CX_MAX_ACTIONS),
        ("z_front", (ctypes.c_int8 * CX_MAX_ZDIRS) * CX_MAX_ACTIONS),
        ("terminate_emptied", ctypes.c_uint8),
        ("emptied_value", ctypes.c_float),
        ("door_key", ctypes.c_int8),
    ]


class GameDesc(ctypes.Structure):
    _fields_ = [
        ("abi_version", ctypes.c_int32),
        ("rows", ctypes.c_int32),
        ("cols", ctypes.c_int32),
        ("n_chars", ctypes.c_int32),
        ("chars", ctypes.c_uint8 * CX_MAX_CHARS),
        ("n_actions", ctypes.c_int32),
        ("n_entities", ctypes.c_int32),
        ("n_groups", ctypes.c_int32),
        ("entities", EntityDesc * CX_MAX_ENTITIES),
        ("backdrop", ctypes.POINTER(ctypes.c_uint8)),
        ("masks", ctypes.POINTER(ctypes.c_uint8)),
        ("max_episode_steps", ctypes.c_int32),
        ("auto_reset", ctypes.c_int32),
        ("track_returns", ctypes.c_int32),
        ("first_reward", ctypes.c_float),
        ("first_discount", ctypes.c_float),
        ("backdrop_dr", ctypes.c_int8 * CX_MAX_ACTIONS),
        ("backdrop_dc", ctypes.c_int8 * CX_MAX_ACTIONS),
        ("unoccluded_layers", ctypes.c_int32),
        ("perf_regions", ctypes.POINTER(ctypes.c_uint8)),
        ("n_perf_regions", ctypes.c_int32),
    ]


class GameInfo(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in (
        "rows", "cols", "cells", "n_chars", "n_actions", "n_entities", "path", "can_terminate", "tracks",
        "has_dynamic_backdrop", "state_bytes_per_env", "board_bytes_per_env", "dynamic_render",
        "tracks_performance", "n_pickups")]


_P = ctypes.c_void_p
_I64 = ctypes.c_int64
_I32 = ctypes.c_int32
_U64 = ctypes.c_uint64

# name -> (restype, argtypes); must list every prototype of include/campx_b200.h
PROTOTYPES = {
    "cx_abi_version": (ctypes.c_int, []),
    "cx_abi_sizeof": (ctypes.c_int, [ctypes.c_int]),
    "cx_last_error": (ctypes.c_char_p, []),
    "cx_game_create": (ctypes.c_int, [ctypes.POINTER(GameDesc), ctypes.POINTER(_P)]),
    "cx_game_destroy": (ctypes.c_int, [_P]),
    "cx_game_get_info": (ctypes.c_int, [_P, ctypes.POINTER(GameInfo)]),
    "cx_state_bytes": (_I64, [_P, _I64]),
    "cx_reset": (ctypes.c_int, [_P, _P, _I64, _P, _P]),
    "cx_render": (ctypes.c_int, [_P, _P, _I64, _P, _P]),
    "cx_step": (ctypes.c_int, [_P, _P, _I64, _P, _P, _P, _P, _P, _P]),
    "cx_rollout": (ctypes.c_int, [_P, _P, _I64, _I32, _P, _P, _P, _P, _P, _P]),
    "cx_rollout_synth": (ctypes.c_int, [_P, _P, _I64, _I32, _U64, _U64, _U64, _P, _P, _P, _P, _P, _P]),
    "cx_rollout_observations": (ctypes.c_int, [_P, _P, _I64, _I32, _P, _P, _P, _P, _P, _P, _P]),
    "cx_render_observations": (ctypes.c_int, [_P, _P, _I64, _P, _P, _I32, _P]),
    "cx_step_observations": (ctypes.c_int, [_P, _P, _I64, _P, _P, _P, _P, _P, _P, _I32, _P]),
    "cx_sample_actions": (ctypes.c_int, [_P, _I64, _I32, _I32, _U64, _U64, _P, _U64, _P, _P, _P]),
    "cx_policy_sample": (ctypes.c_int, [_P, _I64, _I32, _P, _P, _I32, _P, _P, _I32, _U64, _U64, _P, _U64, _P, _P, _P, _P]),
    "cx_policy_sample_board": (ctypes.c_int, [_P, _P, _I64, _P, _P, _I32, _P, _P, _U64, _U64, _P, _U64, _P, _P, _P, _P]),
    "cx_rollout_policy": (ctypes.c_int, [_P, _P, _I64, _I32, _P, _P, _I32, _P, _P, _U64, _U64, _P, _U64, _P, _P, _P, _P, _P, _P]),
    "cx_layers_from_board": (ctypes.c_int, [_P, _P, _I64, _P, _P]),
    "cx_layers_from_board_f32": (ctypes.c_int, [_P, _P, _I64, _P, _P]),
    "cx_board_mapper_create": (ctypes.c_int, [_P, _P, _I32, _I32, ctypes.POINTER(_P)]),
    "cx_board_mapper_destroy": (ctypes.c_int, [_P]),
    "cx_board_mapper_apply": (ctypes.c_int, [_P, _P, _I64, _I32, _I32, ctypes.POINTER(_I32), _P, _P, _P]),
    "cx_onehot_to_index": (ctypes.c_int, [_P, _I64, _I32, _P, _P, _P]),
    "cx_fill_actions": (ctypes.c_int, [_U64, _U64, _U64, _I32, _I64, _I32, _P, _P]),
    "cx_get_entity_state": (ctypes.c_int, [_P, _P, _I64, _I32, _P, _P]),
    "cx_set_entity_state": (ctypes.c_int, [_P, _P, _I64, _I32, _P, _P]),
    "cx_get_render_state": (ctypes.c_int, [_P, _P, _I64, _P, _P, _P, _P]),
    "cx_get_episode_state": (ctypes.c_int, [_P, _P, _I64, _P, _P, _P]),
    "cx_get_episode_performance": (ctypes.c_int, [_P, _P, _I64, _P, _P]),
    "cx_get_pickups": (ctypes.c_int, [_P, _P, _I64, _P, _P]),
    "cx_stats_fold": (ctypes.c_int, [_P, _P, _P]),
    "cx_stats_read": (ctypes.c_int, [_P, _P, ctypes.POINTER(ctypes.c_double), _P]),
    "cx_step_perf": (ctypes.c_int, [_P, _I32, _I32, _P, _P, _I64, _P, _P]),
    "cx_discounted_returns": (ctypes.c_int, [_P, _P, _P, _P, _I32, _I64, ctypes.c_float, _P, _P]),
}

_lib = None


def load():
    """Load (once) and return the shared library with typed prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryError(
            "campx_b200: %s is missing. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C campx_b200/csrc`. campx_b200 has no CPU fallback." % LIB_PATH)
    try:
        lib = ctypes.CDLL(LIB_PATH)
    except OSError as e:
        raise NativeLibraryError("campx_b200: cannot load %s: %s" % (LIB_PATH, e))
    for name, (res, args) in PROTOTYPES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            raise NativeLibraryError("campx_b200: %s does not export %s (stale build?)" % (LIB_PATH, name))
        fn.restype = res
        fn.argtypes = args
    if lib.cx_abi_version() != CX_ABI_VERSION:
        raise NativeLibraryError("campx_b200: library ABI %d != binding ABI %d (rebuild)"
                                 % (lib.cx_abi_version(), CX_ABI_VERSION))
    for which, struct in ((0, EntityDesc), (1, GameDesc), (2, GameInfo)):
        if lib.cx_abi_sizeof(which) != ctypes.sizeof(struct):
            raise NativeLibraryError("campx_b200: struct layout mismatch for %s: C %d vs ctypes %d"
                                     % (struct.__name__, lib.cx_abi_sizeof(which), ctypes.sizeof(struct)))
    _lib = lib
    return lib


_EXC = {CX_ERR_INVALID_ARG: ValueError, CX_ERR_UNSUPPORTED: NotImplementedError,
        CX_ERR_CUDA: RuntimeError, CX_ERR_NOMEM: MemoryError}


def check(rc):
    """Map a cx_status to the exception class the reference would raise for that failure."""
    if rc == CX_OK:
        return
    msg = load().cx_last_error().decode("utf-8", "replace")
    raise _EXC.get(rc, RuntimeError)(msg)


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise NativeLibraryError("campx_b200 needs a CUDA device (B200, sm_100a); there is no CPU path")
