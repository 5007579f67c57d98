"""ctypes binding of the CPU oracle (oracle/liboracle.so) and reader for the
trace files written by oracle/_ref/ref_trace.  TEST INFRASTRUCTURE: imported
only from tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs."""
import ctypes as C
import os
import struct
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
LIB_PATH = os.path.join(ORACLE_DIR, "liboracle.so")
REF_TRACE = os.path.join(ORACLE_DIR, "_ref", "ref_trace")

OG_OTHELLO, OG_C4, OG_GO7, OG_GO9 = 0, 1, 2, 3
OE_UNIFORM, OE_HASHNET, OE_CALLBACK, OE_HEURISTIC = 0, 1, 2, 3
OQ_ZERO, OQ_PARENT, OQ_DROP_PARENT = 0, 1, 2
GAME_NAMES = {OG_OTHELLO: "othello", OG_C4: "c4", OG_GO7: "go", OG_GO9: "go9"}

_DT = {"b": np.int8, "i": np.int32, "f": np.float32, "Q": np.uint64}


def read_trace(path):
    """Parse a ref_trace file: a sequence of named raw arrays."""
    out = {}
    with open(path, "rb") as f:
        data = f.read()
    p = 0
    while p < len(data):
        (nl,) = struct.unpack_from("<I", data, p); p += 4
        name = data[p:p + nl].decode(); p += nl
        dt = chr(data[p]); p += 1
        (nd,) = struct.unpack_from("<I", data, p); p += 4
        dims = struct.unpack_from("<%dQ" % nd, data, p); p += 8 * nd
        dtype = np.dtype(_DT[dt])
        n = int(np.prod(dims)) if nd else 1
        out[name] = np.frombuffer(data, dtype=dtype, count=n, offset=p).reshape(dims).copy()
        p += n * dtype.itemsize
    return out


def have_ref():
    return os.path.exists(REF_TRACE)


def run_ref(*args, tool="ref_trace"):
    """Run the verbatim-reference trace tool (only where oracle/_ref was built).  tool: ref_trace, ref_trace9 (the
    two-constant Go 9x9 build, game name "go") or ref_trace_torch (with the reference's LibTorch GridNetwork)."""
    return subprocess.run([os.path.join(ORACLE_DIR, "_ref", tool), *map(str, args)], check=True, capture_output=True, text=True).stdout


class GameInfo(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("rows", "cols", "cells", "actions", "history", "nsym", "max_plies")] + [("komi", C.c_float)]


EVAL_CB = C.CFUNCTYPE(None, C.c_void_p, C.POINTER(C.c_float), C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float))


class SelfplayCfg(C.Structure):
    _fields_ = [("game", C.c_int), ("evaluator", C.c_int), ("seed", C.c_uint64), ("sims", C.c_int),
                ("max_batch", C.c_int), ("max_queue", C.c_int), ("dir_eps", C.c_float), ("dir_alpha", C.c_float),
                ("add_noise", C.c_int), ("use_sym", C.c_int), ("init_q", C.c_int), ("u_weight", C.c_float),
                ("eval_cb", EVAL_CB), ("eval_user", C.c_void_p), ("hash_salt", C.c_uint64), ("fix_symmetry_mask", C.c_int),
                ("caller_moves", C.c_int)]


DEPTH_BINS = 128


class SearchStats(C.Structure):
    """oracle_search_stats: totals and shape of the searches (descent depths, deep descents by ending, duplicates)."""
    _fields_ = [("total_traversals", C.c_int64), ("total_evals", C.c_int64), ("leaves_terminal", C.c_int64),
                ("leaves_gray", C.c_int64), ("leaves_empty", C.c_int64), ("select_depth_sum", C.c_double),
                ("select_legal_sum", C.c_double), ("select_depth_max", C.c_int32), ("depth_hist", C.c_int64 * DEPTH_BINS),
                ("deep_terminal", C.c_int64), ("deep_gray", C.c_int64), ("deep_queued", C.c_int64),
                ("queue_max", C.c_int32), ("dup_total", C.c_int64), ("dup_first32", C.c_int64)]

    def as_dict(self):
        d = {n: getattr(self, n) for n, _ in self._fields_}
        d["depth_hist"] = np.array(self.depth_hist[:], np.int64)
        return d


class MatchOut(C.Structure):
    _fields_ = [("cap_moves", C.c_int64), ("game_moves", C.c_void_p), ("game_winner", C.c_void_p),
                ("game_rng_draws", C.c_void_p), ("move_N", C.c_void_p), ("move_W", C.c_void_p), ("move_P", C.c_void_p),
                ("move_root_N", C.c_void_p), ("move_root_W", C.c_void_p), ("move_action", C.c_void_p),
                ("move_traversals", C.c_void_p), ("move_agent", C.c_void_p), ("move_player", C.c_void_p),
                ("n_moves", C.c_int64), ("wins", C.c_int64 * 2), ("draws", C.c_int64)]


class SelfplayOut(C.Structure):
    _fields_ = [("cap_moves", C.c_int64), ("cap_samples", C.c_int64),
                ("game_moves", C.c_void_p), ("game_samples", C.c_void_p), ("game_rng_draws", C.c_void_p),
                ("move_N", C.c_void_p), ("move_W", C.c_void_p), ("move_P", C.c_void_p),
                ("move_root_N", C.c_void_p), ("move_root_W", C.c_void_p), ("move_action", C.c_void_p),
                ("move_traversals", C.c_void_p), ("move_evals", C.c_void_p), ("move_player", C.c_void_p),
                ("move_board", C.c_void_p), ("states", C.c_void_p), ("distributions", C.c_void_p),
                ("outcomes", C.c_void_p), ("n_moves", C.c_int64), ("n_samples", C.c_int64),
                ("total_traversals", C.c_int64), ("total_evals", C.c_int64),
                ("select_depth_sum", C.c_double), ("select_legal_sum", C.c_double), ("select_nodes", C.c_int64),
                ("leaves_terminal", C.c_int64), ("leaves_gray", C.c_int64), ("leaves_empty", C.c_int64)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            subprocess.run(["make", "-C", ORACLE_DIR, "oracle"], check=True, capture_output=True)
        _lib = C.CDLL(LIB_PATH)
        _lib.oracle_rollout.restype = C.c_int64
        _lib.oracle_det_powf.restype = C.c_float
        _lib.oracle_det_powf.argtypes = [C.c_float, C.c_float]
        _lib.oracle_det_expf.restype = C.c_float
        _lib.oracle_det_expf.argtypes = [C.c_float]
        _lib.oracle_philox.restype = C.c_uint32
        _lib.oracle_philox.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64]
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def game_info(game):
    gi = GameInfo()
    assert lib().oracle_game_info(C.c_int(game), C.byref(gi)) == 0
    return gi


def perft(game, depth):
    out = C.c_uint64(0)
    assert lib().oracle_perft(C.c_int(game), C.c_int(depth), C.byref(out)) == 0
    return out.value


def rollout(game, seed, first_game, ngames):
    gi = game_info(game)
    cap = ngames * 200
    r = dict(game_steps=np.zeros(ngames, np.int32), cells=np.zeros((cap, gi.cells), np.int8),
             player=np.zeros(cap, np.int8), terminal=np.zeros(cap, np.int8), winner=np.zeros(cap, np.int8),
             mask=np.zeros((cap, gi.actions), np.int8), action=np.zeros(cap, np.int32))
    n = lib().oracle_rollout(C.c_int(game), C.c_uint64(seed), C.c_uint64(first_game), C.c_int(ngames), C.c_int64(cap),
                             _p(r["game_steps"]), _p(r["cells"]), _p(r["player"]), _p(r["terminal"]),
                             _p(r["winner"]), _p(r["mask"]), _p(r["action"]))
    assert n >= 0
    for k in list(r):
        if k != "game_steps":
            r[k] = r[k][:n]
    return r


def replay(game, actions):
    gi = game_info(game)
    a = np.asarray(actions, np.int32)
    cells = np.zeros(gi.cells, np.int8)
    mask = np.zeros(gi.actions, np.int8)
    player, terminal, winner = C.c_int8(), C.c_int8(), C.c_int8()
    rewards = np.zeros(2, np.float32)
    rc = lib().oracle_replay(C.c_int(game), _p(a), C.c_int(len(a)), _p(cells), C.byref(player), C.byref(terminal),
                             C.byref(winner), _p(mask), _p(rewards))
    return dict(rc=rc, cells=cells, player=player.value, terminal=terminal.value, winner=winner.value,
                mask=mask, rewards=rewards)


def selfplay(game, evaluator, seed, first_game, ngames, sims, max_batch, max_queue, eps=0.25, alpha=0.3,
             add_noise=True, use_sym=True, init_q=OQ_PARENT, u_weight=1.1, eval_fn=None, max_moves_per_game=200,
             fix_symmetry_mask=False, caller_moves=False, search_stats=False):
    """Run the oracle's selfPlay for `ngames` games; returns a dict shaped like a ref_trace selfplay trace, plus
    "stats": the totals of oracle_selfplay_out and, with search_stats, the fields of oracle_search_stats."""
    gi = game_info(game)
    S = gi.nsym if use_sym else 1
    cap_m = ngames * max_moves_per_game
    cap_s = cap_m * S
    A, B = gi.actions, gi.cells
    arr = dict(game_moves=np.zeros(ngames, np.int32), game_samples=np.zeros(ngames, np.int32),
               game_rng_draws=np.zeros(ngames, np.uint64),
               move_N=np.zeros((cap_m, A), np.float32), move_W=np.zeros((cap_m, A), np.float32),
               move_P=np.zeros((cap_m, A), np.float32), move_root_N=np.zeros(cap_m, np.float32),
               move_root_W=np.zeros(cap_m, np.float32), move_action=np.zeros(cap_m, np.int32),
               move_traversals=np.zeros(cap_m, np.int32), move_evals=np.zeros(cap_m, np.int32),
               move_player=np.zeros(cap_m, np.int8), move_board=np.zeros((cap_m, B), np.int8),
               states=np.zeros((cap_s, 2 * gi.history + 1, gi.rows, gi.cols), np.float32),
               distributions=np.zeros((cap_s, A), np.float32), outcomes=np.zeros(cap_s, np.float32))
    cfg = SelfplayCfg(game=game, evaluator=evaluator, seed=seed, sims=sims, max_batch=max_batch, max_queue=max_queue,
                      dir_eps=eps, dir_alpha=alpha, add_noise=int(add_noise), use_sym=int(use_sym), init_q=init_q,
                      u_weight=u_weight, fix_symmetry_mask=int(fix_symmetry_mask), caller_moves=int(caller_moves))
    keep = None
    if evaluator == OE_CALLBACK:
        planes_per = (2 * gi.history + 1) * B

        def _cb(_user, planes, n, logits, values):
            x = np.ctypeslib.as_array(planes, shape=(n, 2 * gi.history + 1, gi.rows, gi.cols))
            lg, v = eval_fn(x)
            np.ctypeslib.as_array(logits, shape=(n, A))[:] = np.asarray(lg, np.float32).reshape(n, A)
            np.ctypeslib.as_array(values, shape=(n,))[:] = np.asarray(v, np.float32).reshape(n)
        keep = EVAL_CB(_cb)
        cfg.eval_cb = keep
        del planes_per
    out = SelfplayOut(cap_moves=cap_m, cap_samples=cap_s)
    for k, v in arr.items():
        setattr(out, k, v.ctypes.data)
    search = SearchStats()
    if search_stats:
        rc = lib().oracle_selfplay_ex(C.byref(cfg), C.c_uint64(first_game), C.c_int(ngames), C.byref(out), C.byref(search))
    else:
        rc = lib().oracle_selfplay(C.byref(cfg), C.c_uint64(first_game), C.c_int(ngames), C.byref(out))
    assert rc == 0, rc
    M, N = out.n_moves, out.n_samples
    res = {}
    for k, v in arr.items():
        if k.startswith("move_"):
            res[k] = v[:M]
        elif k in ("states", "distributions", "outcomes"):
            res[k] = v[:N]
        else:
            res[k] = v
    res["stats"] = dict(total_traversals=out.total_traversals, total_evals=out.total_evals,
                        select_depth_sum=out.select_depth_sum, select_legal_sum=out.select_legal_sum,
                        select_nodes=out.select_nodes, leaves_terminal=out.leaves_terminal,
                        leaves_gray=out.leaves_gray, leaves_empty=out.leaves_empty)
    if search_stats:
        res["stats"] = dict(search.as_dict(), **res["stats"])
    return res


def _make_eval_cb(gi, eval_fn):
    A = gi.actions

    def _cb(_user, planes, n, logits, values):
        x = np.ctypeslib.as_array(planes, shape=(n, 2 * gi.history + 1, gi.rows, gi.cols))
        lg, v = eval_fn(x)
        np.ctypeslib.as_array(logits, shape=(n, A))[:] = np.asarray(lg, np.float32).reshape(n, A)
        np.ctypeslib.as_array(values, shape=(n,))[:] = np.asarray(v, np.float32).reshape(n)
    return EVAL_CB(_cb)


def match(game, agents, seed, first_game, ngames, sims, max_batch, max_queue, max_moves_per_game=200, search_stats=False):
    """Run the oracle's match play.  agents = two dicts with keys evaluator, use_sym, init_q and optionally
    hash_salt / eval_fn.  Returns a dict shaped like a ref_trace match trace (+ wins, draws, and with search_stats
    "stats": the fields of oracle_search_stats over both agents' searches)."""
    gi = game_info(game)
    A = gi.actions
    cap_m = ngames * max_moves_per_game
    arr = dict(game_moves=np.zeros(ngames, np.int32), game_winner=np.zeros(ngames, np.int32),
               game_rng_draws=np.zeros(ngames, np.uint64),
               move_N=np.zeros((cap_m, A), np.float32), move_W=np.zeros((cap_m, A), np.float32),
               move_P=np.zeros((cap_m, A), np.float32), move_root_N=np.zeros(cap_m, np.float32),
               move_root_W=np.zeros(cap_m, np.float32), move_action=np.zeros(cap_m, np.int32),
               move_traversals=np.zeros(cap_m, np.int32), move_agent=np.zeros(cap_m, np.int32),
               move_player=np.zeros(cap_m, np.int8))
    cfgs = (SelfplayCfg * 2)()
    keep = []
    for k, ag in enumerate(agents):
        cfgs[k] = SelfplayCfg(game=game, evaluator=ag["evaluator"], seed=seed, sims=sims, max_batch=max_batch,
                              max_queue=max_queue, use_sym=int(ag.get("use_sym", 1)), init_q=ag.get("init_q", OQ_PARENT),
                              hash_salt=ag.get("hash_salt", 0))
        if ag["evaluator"] == OE_CALLBACK:
            keep.append(_make_eval_cb(gi, ag["eval_fn"]))
            cfgs[k].eval_cb = keep[-1]
    out = MatchOut(cap_moves=cap_m)
    for k, v in arr.items():
        setattr(out, k, v.ctypes.data)
    search = SearchStats()
    if search_stats:
        rc = lib().oracle_match_ex(cfgs, C.c_uint64(first_game), C.c_int(ngames), C.byref(out), C.byref(search))
    else:
        rc = lib().oracle_match(cfgs, C.c_uint64(first_game), C.c_int(ngames), C.byref(out))
    assert rc == 0, rc
    res = {k: (v[:out.n_moves] if k.startswith("move_") else v) for k, v in arr.items()}
    res["wins"] = (out.wins[0], out.wins[1])
    res["draws"] = out.draws
    if search_stats:
        res["stats"] = search.as_dict()
    return res


def write_npy(path, arr):
    a = np.ascontiguousarray(arr, np.float32)
    shape = (C.c_uint64 * a.ndim)(*a.shape)
    assert lib().oracle_write_npy_f32(path.encode(), _p(a), shape, C.c_int(a.ndim)) == 0
