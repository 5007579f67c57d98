"""ctypes binding of libsprl_b200.so (include/sprl_b200.h).

The library is the product: CUDA kernels + a C ABI.  This module only declares
the prototypes and converts errors to exceptions; there is no Python or CPU
implementation behind it.  Importing works without a GPU (symbols resolve);
any compute call without a device raises SprlError(SPRL_E_NOGPU).
"""
import ctypes as C
import os

from . import build as _build

SPRL_OK = 0
SPRL_E_INVALID, SPRL_E_CUDA, SPRL_E_CAPACITY, SPRL_E_STATE, SPRL_E_IO, SPRL_E_NOGPU = -1, -2, -3, -4, -5, -6
GAME_OTHELLO, GAME_C4, GAME_GO7, GAME_GO9 = 0, 1, 2, 3
EVAL_UNIFORM, EVAL_HASHNET, EVAL_EXTERNAL, EVAL_OTHELLO_HEURISTIC = 0, 1, 2, 3
INITQ_ZERO, INITQ_PARENT, INITQ_DROP_PARENT = 0, 1, 2
EVALNET_PATH_AUTO, EVALNET_PATH_STREAMING, EVALNET_PATH_RESIDENT = 0, 1, 2
EVALNET_PRECISION_FP32_SPLIT, EVALNET_PRECISION_FP16 = 0, 1

EXPORTS = [
    "sprl_last_error", "sprl_device_count", "sprl_game_info_get", "sprl_env_step", "sprl_env_line", "sprl_env_rollout",
    "sprl_env_perft", "sprl_default_config", "sprl_create", "sprl_destroy", "sprl_set_stream",
    "sprl_bind_eval_buffers", "sprl_eval_batch", "sprl_eval_rows", "sprl_set_game_stride", "sprl_set_openings", "sprl_begin_iteration", "sprl_round", "sprl_poll",
    "sprl_run_iteration", "sprl_iteration_counts", "sprl_collect_samples", "sprl_collect_samples_device", "sprl_stream_samples", "sprl_stream_info",
    "sprl_match_begin", "sprl_run_match", "sprl_match_results", "sprl_begin_trees", "sprl_search", "sprl_search_batch",
    "sprl_apply_evaluations", "sprl_root_stats", "sprl_advance", "sprl_move_stats", "sprl_debug_check_guards", "sprl_get_stats", "sprl_reset_stats", "sprl_write_npy_f32",
    "sprl_evalnet_create", "sprl_evalnet_update", "sprl_evalnet_forward", "sprl_evalnet_forward_counted", "sprl_evalnet_status", "sprl_evalnet_info", "sprl_evalnet_set_path", "sprl_evalnet_set_precision", "sprl_evalnet_phases", "sprl_evalnet_destroy",
]


class SprlError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"libsprl_b200 error {code}: {message}")
        self.code = code


class GameInfo(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("rows", "cols", "cells", "actions", "history", "nsym", "max_plies")]


class Config(C.Structure):
    _fields_ = [("device", C.c_int), ("game", C.c_int), ("evaluator", C.c_int), ("seed", C.c_uint64),
                ("num_slots", C.c_int), ("sims", C.c_int), ("max_batch", C.c_int), ("max_queue", C.c_int),
                ("dir_eps", C.c_float), ("dir_alpha", C.c_float), ("u_weight", C.c_float),
                ("add_noise", C.c_int), ("use_sym", C.c_int), ("init_q", C.c_int),
                ("units_per_tree", C.c_int64), ("max_games", C.c_int64), ("record_stats", C.c_int),
                ("rounds_per_launch", C.c_int), ("fix_symmetry_mask", C.c_int)]


class Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("sims", "evals", "moves", "games", "depth_sum", "legal_sum", "nodes_visited",
                                          "leaves_terminal", "leaves_gray", "leaves_empty", "units_high_water",
                                          "units_per_tree", "launches", "device_bytes", "leaves_duplicate")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class AgentConfig(C.Structure):
    _fields_ = [("evaluator", C.c_int), ("use_sym", C.c_int), ("init_q", C.c_int), ("hash_salt", C.c_uint64)]


class ConvBnParams(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("weight", "bias", "bn_weight", "bn_bias", "bn_mean", "bn_var")]


class NetworkParams(C.Structure):
    _fields_ = ([(n, C.c_int) for n in ("rows", "cols", "in_planes", "channels", "blocks", "actions", "policy_channels",
                                         "value_channels", "value_hidden")] +
                [("bn_eps", C.c_float), ("stem", ConvBnParams), ("tower", C.POINTER(ConvBnParams))] +
                [(n, C.c_void_p) for n in ("policy_conv_w", "policy_conv_b", "policy_fc_w", "policy_fc_b", "value_conv_w",
                                           "value_conv_b", "value_fc1_w", "value_fc1_b", "value_fc2_w", "value_fc2_b")])


FORWARD_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p)

_lib = None


def lib_path():
    return _build.LIB_PATH


def load():
    """Loads the shared library (building it in-tree first when it is missing or stale)."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("SPRL_B200_LIB") or _build.LIB_PATH      # SPRL_B200_LIB: another build of the library, e.g. a parent commit's for A/B runs
    if path == _build.LIB_PATH and (not os.path.exists(path) or os.environ.get("SPRL_B200_REBUILD")):
        _build.build_library()
    lib = C.CDLL(path)
    lib.sprl_last_error.restype = C.c_char_p
    lib.sprl_eval_batch.restype = C.c_int64
    lib.sprl_eval_batch.argtypes = [C.c_void_p]
    lib.sprl_destroy.restype = None
    lib.sprl_destroy.argtypes = [C.c_void_p]
    lib.sprl_create.argtypes = [C.POINTER(Config), C.POINTER(C.c_void_p)]
    lib.sprl_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    lib.sprl_bind_eval_buffers.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.sprl_eval_rows.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    lib.sprl_set_game_stride.argtypes = [C.c_void_p, C.c_uint64]
    lib.sprl_set_openings.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    lib.sprl_begin_iteration.argtypes = [C.c_void_p, C.c_uint64, C.c_int64]
    lib.sprl_round.argtypes = [C.c_void_p]
    lib.sprl_poll.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    lib.sprl_run_iteration.argtypes = [C.c_void_p, C.c_uint64, C.c_int64, C.c_void_p, C.c_void_p]
    lib.sprl_iteration_counts.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    lib.sprl_collect_samples.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)]
    lib.sprl_collect_samples_device.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                                C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]
    lib.sprl_stream_samples.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    lib.sprl_stream_info.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_uint64)]
    lib.sprl_match_begin.argtypes = [C.c_void_p, C.POINTER(AgentConfig), C.c_uint64, C.c_int64]
    lib.sprl_run_match.argtypes = [C.c_void_p, C.POINTER(AgentConfig), C.c_uint64, C.c_int64, C.c_void_p, C.c_void_p]
    lib.sprl_match_results.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64),
                                       C.POINTER(C.c_int64)]
    lib.sprl_begin_trees.argtypes = [C.c_void_p, C.c_uint64, C.c_int64]
    lib.sprl_search.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    lib.sprl_search_batch.argtypes = [C.c_void_p]
    lib.sprl_apply_evaluations.argtypes = [C.c_void_p]
    lib.sprl_root_stats.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 11
    lib.sprl_advance.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
    lib.sprl_move_stats.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 10 + [C.POINTER(C.c_int64)]
    lib.sprl_debug_check_guards.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    lib.sprl_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
    lib.sprl_reset_stats.argtypes = [C.c_void_p]
    lib.sprl_env_step.argtypes = [C.c_int, C.c_int, C.c_int64] + [C.c_void_p] * 8
    lib.sprl_env_line.argtypes = [C.c_int, C.c_int, C.c_int32] + [C.c_void_p] * 6
    lib.sprl_env_rollout.argtypes = [C.c_int, C.c_int, C.c_uint64, C.c_uint64, C.c_int64, C.c_void_p, C.c_void_p,
                                     C.c_int64] + [C.c_void_p] * 6 + [C.POINTER(C.c_int64), C.POINTER(C.c_float)]
    lib.sprl_env_perft.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_float)]
    lib.sprl_write_npy_f32.argtypes = [C.c_char_p, C.c_void_p, C.POINTER(C.c_uint64), C.c_int]
    lib.sprl_evalnet_create.argtypes = [C.c_int, C.POINTER(NetworkParams), C.POINTER(C.c_void_p)]
    lib.sprl_evalnet_update.argtypes = [C.c_void_p, C.POINTER(NetworkParams)]
    lib.sprl_evalnet_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.sprl_evalnet_forward_counted.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.sprl_evalnet_status.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
    lib.sprl_evalnet_info.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    lib.sprl_evalnet_set_path.argtypes = [C.c_void_p, C.c_int]
    lib.sprl_evalnet_set_precision.argtypes = [C.c_void_p, C.c_int]
    lib.sprl_evalnet_phases.argtypes = [C.c_void_p]
    lib.sprl_evalnet_destroy.restype = None
    lib.sprl_evalnet_destroy.argtypes = [C.c_void_p]
    lib.sprl_default_config.argtypes = [C.c_int, C.POINTER(Config)]
    lib.sprl_game_info_get.argtypes = [C.c_int, C.POINTER(GameInfo)]
    _lib = lib
    return lib


def check(rc):
    if rc != SPRL_OK:
        raise SprlError(rc, load().sprl_last_error().decode(errors="replace"))


def game_info(game):
    gi = GameInfo()
    check(load().sprl_game_info_get(game, C.byref(gi)))
    return gi


def default_config(game):
    cfg = Config()
    check(load().sprl_default_config(game, C.byref(cfg)))
    return cfg
