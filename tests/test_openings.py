"""Games, matches and step-wise trees that start from opening lines (sprl_set_openings / Engine.set_openings).

A game that starts from line L is the game whose tree is built at the start position and advanced through L before any
search: the line draws no random number, its positions are the game's history, and only searched moves are sampled,
recorded and counted.  The reference is the oracle's own self-play and match play with the opening added (tests/oracle_open.c:
oracle_selfplay_open / oracle_match_open); it is pinned here to the existing golden traces (no lines) and to oracle_replay
(the history), and the engine is compared with it bit for bit.
Lines are prefixes of recorded random play-outs: lengths 0, 1, 2, an odd and an even mid-game length, mixed in one table;
for Go, lines that hold passes and captures."""
import atexit
import ctypes as C
import functools
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import golden_util as G
import oracle_py as O
from sprl_b200 import capi
from sprl_b200 import selfplay as SP
from test_gpu_parity import EXACT_KEYS, MATCH_KEYS, compare_selfplay

GAMES = {"othello": (capi.GAME_OTHELLO, O.OG_OTHELLO), "c4": (capi.GAME_C4, O.OG_C4), "go": (capi.GAME_GO7, O.OG_GO7),
         "go9": (capi.GAME_GO9, O.OG_GO9)}
EVALS = {"hash": (capi.EVAL_HASHNET, O.OE_HASHNET), "hash1": (capi.EVAL_HASHNET, O.OE_HASHNET),
         "uniform": (capi.EVAL_UNIFORM, O.OE_UNIFORM), "heuristic": (capi.EVAL_OTHELLO_HEURISTIC, O.OE_HEURISTIC)}
INITQ = {"parent": capi.INITQ_PARENT, "zero": capi.INITQ_ZERO, "drop": capi.INITQ_DROP_PARENT}
MID = {"othello": (7, 12), "c4": (5, 8), "go": (11, 20), "go9": (15, 24)}     # an odd and an even mid-game length


# ---------------------------------------------------------------------------------------------- opening lines
def rollout_games(og, seed, n):
    """(actions, cells) of each of n recorded random play-outs of the oracle (the engine's env_rollout is pinned to it)."""
    r = O.rollout(og, seed, 0, n)
    out, at = [], 0
    for s in r["game_steps"]:
        out.append((r["action"][at:at + s - 1].copy(), r["cells"][at:at + s].copy()))
        at += s
    return out


def capture_pass_line(og, games):
    """The shortest prefix of a play-out that holds a pass and a capture and ends before the game does (Go)."""
    gi = O.game_info(og)
    best = None
    for actions, cells in games:
        stones = (cells != -1).sum(1)
        passed = captured = False
        for k, a in enumerate(actions[:-1]):
            passed |= a == gi.cells
            captured |= a != gi.cells and stones[k + 1] < stones[k] + 1
            if passed and captured:
                if best is None or k + 1 < len(best):
                    best = actions[:k + 1]
                break
    assert best is not None
    return [int(a) for a in best]


def opening_lines(name, seed=5):
    """Prefixes of play-outs of lengths 0, 1, 2 and the two mid-game lengths, each from a different play-out; for Go
    also a line with a pass and a capture.  Every line ends before its play-out does (a game has a move left)."""
    og = GAMES[name][1]
    games = [g for g in rollout_games(og, seed, 24) if len(g[0]) > max(MID[name]) + 1]
    lines = [[int(a) for a in games[k % len(games)][0][:n]] for k, n in enumerate((0, 1, 2) + MID[name])]
    if name in ("go", "go9"):
        lines.append(capture_pass_line(og, rollout_games(og, seed + 1, 64)))
    return lines


def table(lines):
    offsets = np.zeros(len(lines) + 1, np.int64)
    offsets[1:] = np.cumsum([len(line) for line in lines])
    actions = np.array([a for line in lines for a in line] or [0], np.int32)
    return offsets, actions


# ---------------------------------------------------------------------------------------------- the oracle with lines
@functools.lru_cache(maxsize=None)
def open_lib():
    """tests/oracle_open.c (which includes oracle/oracle_search.c) with oracle/oracle_games.c, built like the oracle
    (oracle/Makefile's flags) into a temporary directory."""
    here = os.path.dirname(os.path.abspath(__file__))
    out = tempfile.mkdtemp(prefix="oracle_open_")
    atexit.register(shutil.rmtree, out, True)
    path = os.path.join(out, "liboracle_open.so")
    subprocess.run([os.environ.get("CC") or "cc", "-std=c11", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-o", path,
                    os.path.join(here, "oracle_open.c"), os.path.join(O.ORACLE_DIR, "oracle_games.c")], check=True, capture_output=True)
    return C.CDLL(path)


class _OpenLib:
    """liboracle whose _ex entry points are the _open ones of tests/oracle_open.c with a table of lines: lets
    oracle_py.selfplay / match shape the traces of games that start from lines."""

    def __init__(self, lines):
        self.offsets, self.actions = table(lines)
        self.n = len(lines)
        self.lib = O.lib()

    def __getattr__(self, name):
        return getattr(self.lib, name)

    def oracle_selfplay_ex(self, cfg, first, n, out, search):
        return open_lib().oracle_selfplay_open(cfg, first, n, out, search, C.c_int64(self.n), O._p(self.offsets), O._p(self.actions))

    def oracle_match_ex(self, cfgs, first, n, out, search):
        return open_lib().oracle_match_open(cfgs, first, n, out, search, C.c_int64(self.n), O._p(self.offsets), O._p(self.actions))


def _with_lines(fn, lines, *args, **kw):
    O.lib()
    plain = O._lib
    O._lib = _OpenLib(lines)
    try:
        return fn(*args, search_stats=True, **kw)
    finally:
        O._lib = plain


def oracle_selfplay(lines, *args, **kw):
    return _with_lines(O.selfplay, lines, *args, **kw)


def oracle_match(lines, *args, **kw):
    ref = _with_lines(O.match, lines, *args, **kw)
    ref["game_winner"] = ref["game_winner"].astype(np.int8)
    return ref


def open_rc(og, lines, match=False):
    """Return code of the oracle's _open entry point for one game from the first line (HashNet, 8 descents)."""
    offsets, actions = table(lines)
    cfg = O.SelfplayCfg(game=og, evaluator=O.OE_HASHNET, seed=0, sims=8, max_batch=8, max_queue=4, dir_eps=0.25,
                        dir_alpha=0.3, add_noise=1, use_sym=1, init_q=O.OQ_PARENT, u_weight=1.1)
    if match:
        return open_lib().oracle_match_open((O.SelfplayCfg * 2)(cfg, cfg), C.c_uint64(0), C.c_int(1), C.byref(O.MatchOut(cap_moves=1000)),
                                         None, C.c_int64(len(lines)), O._p(offsets), O._p(actions))
    return open_lib().oracle_selfplay_open(C.byref(cfg), C.c_uint64(0), C.c_int(1), C.byref(O.SelfplayOut(cap_moves=1000, cap_samples=8000)),
                                        None, C.c_int64(len(lines)), O._p(offsets), O._p(actions))


# ---------------------------------------------------------------------------------------------- CPU: the oracle
@pytest.mark.parametrize("name", G.SELFPLAY_FIXTURES)
def test_oracle_selfplay_without_lines_is_the_golden(name):
    cmd, ref = G.load("selfplay_" + name)
    got = oracle_selfplay([], G.GAME_ID[cmd["game"]], G.EVAL_ID[cmd["evaluator"]], cmd["seed"], cmd["first_game"], cmd["ngames"],
                          cmd["sims"], cmd["max_batch"], cmd["max_queue"], cmd["eps"], cmd["alpha"], bool(cmd["noise"]),
                          bool(cmd["sym"]), G.INITQ_ID[cmd["initq"]])
    G.assert_trace_equal(ref, got, EXACT_KEYS + ["game_samples", "move_evals", "move_board"])
    G.assert_trace_equal(ref, got, ["distributions"], exact=False)


@pytest.mark.parametrize("name", G.MATCH_FIXTURES)
def test_oracle_match_without_lines_is_the_golden(name):
    cmd, ref = G.load("match_" + name)
    got = oracle_match([], G.GAME_ID[cmd["game"]], G.match_agents(cmd), cmd["seed"], cmd["first_game"], cmd["ngames"],
                       cmd["sims"], cmd["max_batch"], cmd["max_queue"])
    G.assert_trace_equal(ref, got, ["game_moves", "game_winner", "game_rng_draws", "move_N", "move_W", "move_P", "move_root_N",
                                    "move_root_W", "move_action", "move_traversals", "move_agent", "move_player"])


@pytest.mark.parametrize("name", ["othello", "c4", "go"])
def test_oracle_game_from_a_line_samples_searched_moves_over_the_line_history(name):
    """Game t plays line t % n_lines; it records searched moves only, its first sample's history planes are the boards of
    the line's last positions (oracle_replay), and the whole game (line + searched moves) replays to its outcome."""
    og = GAMES[name][1]
    gi = O.game_info(og)
    lines = opening_lines(name)
    ref = oracle_selfplay(lines, og, O.OE_HASHNET, 3, 0, len(lines), 24, 8, 4, 0.25, 0.3)
    S, P = gi.nsym, 2 * gi.history + 1
    assert len(ref["states"]) == S * ref["game_moves"].sum() == S * len(ref["move_action"])
    first = np.concatenate([[0], np.cumsum(ref["game_moves"])[:-1]])
    for t, line in enumerate(lines):
        end = O.replay(og, line)
        assert end["rc"] == 0 and end["terminal"] == 0
        m0 = first[t]
        assert ref["move_player"][m0] == end["player"]
        assert np.array_equal(ref["move_board"][m0], end["cells"])
        planes = ref["states"][m0 * S].reshape(P, -1)         # symmetry 0 = identity
        for h in range(gi.history):
            if h <= len(line):
                cells = O.replay(og, line[:len(line) - h])["cells"]
                want_own, want_opp = cells == end["player"], cells == 1 - end["player"]
            else:
                want_own = want_opp = np.zeros(gi.cells, bool)
            assert np.array_equal(planes[2 * h], want_own.astype(np.float32)), (t, h)
            assert np.array_equal(planes[2 * h + 1], want_opp.astype(np.float32)), (t, h)
        whole = O.replay(og, line + [int(a) for a in ref["move_action"][m0:m0 + ref["game_moves"][t]]])
        assert whole["rc"] == 0 and whole["terminal"] == 1
        outcome = ref["outcomes"][m0 * S]
        assert outcome == whole["rewards"][ref["move_player"][m0]]


def test_oracle_refuses_illegal_lines():
    for og in (O.OG_OTHELLO, O.OG_C4, O.OG_GO7):
        gi = O.game_info(og)
        mask = O.replay(og, [])["mask"]
        illegal = int(np.nonzero(mask == 0)[0][0]) if (mask == 0).any() else gi.actions
        for match in (False, True):
            assert open_rc(og, [[illegal]], match) == -3
            assert open_rc(og, [[gi.actions]], match) == -3
            assert open_rc(og, [[-1]], match) == -3
            assert open_rc(og, [[]], match) == 0
    # a line that reaches a terminal position (tests/test_c4.cpp's known answer: ZERO wins) leaves nothing to search
    for match in (False, True):
        assert open_rc(O.OG_C4, [[3, 3, 4, 4, 2, 3, 1]], match) == -3
        assert open_rc(O.OG_C4, [[3, 3, 4, 4, 2, 3]], match) == 0


# ---------------------------------------------------------------------------------------------- GPU: the engine
def engine(game, ev, seed, sims, b, q, ngames, slots, **kw):
    return SP.Engine(game, ev, seed=seed, sims=sims, max_batch=b, max_queue=q, num_slots=slots, max_games=ngames,
                     record_stats=1, **kw)


def finish(eng, ngames, samples):
    states, dists, outcomes = samples
    got = eng.move_stats(ngames)
    got.update(states=states, distributions=dists, outcomes=outcomes, stats=eng.stats())
    pools, damaged = eng.check_guards()
    assert pools > 20 and damaged == 0
    return got


def check_stats(st, ref):
    rs = ref["stats"]
    assert st["sims"] == rs["total_traversals"] and st["evals"] == rs["total_evals"]
    assert st["leaves_terminal"] == rs["leaves_terminal"] and st["leaves_gray"] == rs["leaves_gray"]
    assert st["moves"] == len(ref["move_action"]) and st["games"] == len(ref["game_moves"])


@pytest.mark.gpu
@pytest.mark.parametrize("name,sims,b,q,alpha,ngames,slots", [
    ("othello", 100, 8, 4, 0.3, 14, 5),
    ("c4", 200, 8, 4, 0.5, 14, 4),
    ("go", 60, 16, 8, 0.2, 8, 3),
    ("go9", 40, 16, 8, 0.2, 6, 2),
])
def test_selfplay_from_lines_vs_oracle(name, sims, b, q, alpha, ngames, slots):
    """HashNet self-play from a mixed table, more games than slots: slots start later games from the table inside the
    search kernel.  Samples, move statistics, draws and winners bit for bit."""
    game, og = GAMES[name]
    lines = opening_lines(name)
    seed, first = 77, 300
    ref = oracle_selfplay(lines, og, O.OE_HASHNET, seed, first, ngames, sims, b, q, 0.25, alpha, max_moves_per_game=170)
    with engine(game, capi.EVAL_HASHNET, seed, sims, b, q, ngames, slots, dir_eps=0.25, dir_alpha=alpha) as eng:
        eng.set_openings(lines)
        got = finish(eng, ngames, eng.run_iteration(ngames, first_game=first))
        assert eng.iteration_counts() == (len(ref["move_action"]), len(ref["states"]))
    compare_selfplay(ref, got)
    check_stats(got["stats"], ref)


@pytest.mark.gpu
def test_selfplay_from_lines_through_evalnet_and_a_captured_graph_vs_oracle():
    """The library evaluator on the external-evaluator path, the round captured as one CUDA graph; fewer slots than games."""
    import test_evalnet_selfplay as E
    c = E.cfg("othello", "othello", 120, 8, 4, 0.3, 7, slots=3, first=40)
    lines = opening_lines("othello")
    ev = E.oracle_evaluator(c["ev"], on_gpu=True)
    ref = oracle_selfplay(lines, O.OG_OTHELLO, O.OE_CALLBACK, E.SEED, c["first"], c["ngames"], c["sims"], c["b"], c["q"], 0.25,
                          c["alpha"], eval_fn=ev, max_moves_per_game=130)
    ev.close()
    net = E.setting_evalnet(c["ev"])
    with E.selfplay_engine(c, c["slots"], c["ngames"]) as eng:
        eng.set_openings(lines)
        eng.attach_evalnet(net, use_cuda_graph=True)
        got = finish(eng, c["ngames"], eng.run_iteration(c["ngames"], first_game=c["first"]))
        assert eng._nn["graph"] is not None
    net.status()
    net.close()
    compare_selfplay(ref, got)
    check_stats(got["stats"], ref)


@pytest.mark.gpu
@pytest.mark.parametrize("name,evs,sims,b,q,ngames,pairs", [
    ("othello", ("hash", "hash1"), 80, 8, 4, 12, 3),
    ("c4", ("hash", "uniform"), 96, 8, 4, 12, 4),
    ("go", ("hash", "hash1"), 40, 16, 8, 6, 2),
])
def test_match_from_lines_vs_oracle(name, evs, sims, b, q, ngames, pairs):
    """Ids 2k and 2k+1 play one line with the colours swapped; odd- and even-length lines (an odd one makes Player ONE
    the first side to search).  Bit for bit, wins and draws included."""
    game, og = GAMES[name]
    lines = opening_lines(name)
    seed, first = 7, 10
    o_agents = [dict(evaluator=EVALS[e][1], hash_salt=G.HASH_SALT.get(e, 0), use_sym=1, init_q=O.OQ_PARENT) for e in evs]
    g_agents = [dict(evaluator=EVALS[e][0], hash_salt=G.HASH_SALT.get(e, 0), use_sym=1, init_q=capi.INITQ_PARENT) for e in evs]
    ref = oracle_match(lines, og, o_agents, seed, first, ngames, sims, b, q, max_moves_per_game=170)
    # both colour assignments of each line: the first searched move of games 2k and 2k+1 is made by the same Player from
    # the same position, by different agents
    at = np.concatenate([[0], np.cumsum(ref["game_moves"])[:-1]])
    for g in range(0, ngames, 2):
        line = lines[((first + g) // 2) % len(lines)]
        assert ref["move_player"][at[g]] == ref["move_player"][at[g + 1]] == len(line) % 2
        assert ref["move_agent"][at[g]] != ref["move_agent"][at[g + 1]]
    assert {len(lines[((first + g) // 2) % len(lines)]) % 2 for g in range(ngames)} == {0, 1}
    with SP.Engine(game, capi.EVAL_UNIFORM, seed=seed, sims=sims, max_batch=b, max_queue=q, dir_eps=0.25, dir_alpha=0.1,
                   u_weight=1.0, add_noise=1, num_slots=2 * pairs, max_games=ngames, record_stats=1) as eng:
        eng.set_openings(lines)
        got = eng.run_match(g_agents, ngames, first_game=first)
        got.update(eng.move_stats(ngames))
        assert eng.check_guards()[1] == 0
    G.assert_trace_equal(ref, got, MATCH_KEYS)
    assert got["wins"] == ref["wins"] and got["draws"] == ref["draws"]
    assert got["wins"][0] + got["wins"][1] + got["draws"] == ngames


def walk(eng, n, sims, lines=None, steps=3):
    """Step-wise trees: with `lines`, advance tree i through its line first (sprl_advance, -1 once it ends).  Then
    `steps` times: search, read the decision nodes, advance every tree by its most-visited action."""
    if lines is not None:
        for k in range(max(len(line) for line in lines)):
            eng.advance([line[k] if k < len(line) else -1 for line in lines])
    rows = []
    for _ in range(steps):
        eng.search(sims)
        st = eng.root_stats()
        rows.append(st)
        eng.advance(np.where(st["terminal"] == 0, st["N"].argmax(1), -1))
    return rows


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["othello", "c4", "go", "go9"])
def test_stepwise_trees_from_lines_equal_trees_advanced_through_them(name):
    """begin_trees under a table, then search, equals begin_trees at the start, sprl_advance through each tree's line
    (stream id t: line t % n_lines), then the same search: every decision node's statistics, and after the games are
    played out the move records of the searched moves."""
    game, _ = GAMES[name]
    lines = opening_lines(name)
    n, first, sims = 2 * len(lines) + 1, 3, 48
    mine = [lines[(first + t) % len(lines)] for t in range(n)]
    kw = dict(seed=5, sims=sims, max_batch=8, max_queue=4, dir_eps=0.25, dir_alpha=0.3, num_slots=n, max_games=n, record_stats=1)
    with SP.Engine(game, capi.EVAL_HASHNET, **kw) as a, SP.Engine(game, capi.EVAL_HASHNET, **kw) as b:
        a.set_openings(lines)
        a.begin_trees(n, first_game=first)
        b.begin_trees(n, first_game=first)
        ra, rb = walk(a, n, sims), walk(b, n, sims, mine)
        for sa, sb in zip(ra, rb):
            for k in sa:
                assert np.array_equal(sa[k], sb[k]), k
        while (a.root_stats()["terminal"] == 0).any():          # play the games out, the same way on both
            ra, rb = walk(a, n, sims, steps=1), walk(b, n, sims, steps=1)
            for k in ra[0]:
                assert np.array_equal(ra[0][k], rb[0][k]), k
        ma, mb = a.move_stats(n), b.move_stats(n)
        for eng in (a, b):
            assert eng.poll() == (0, 0) and eng.check_guards()[1] == 0
    # b's records include the caller's advances through the lines: they are a's records after them
    assert np.array_equal(ma["game_moves"], mb["game_moves"] - np.array([len(line) for line in mine]))
    keep = np.concatenate([np.arange(s + len(line), s + m) for s, m, line in
                           zip(np.concatenate([[0], np.cumsum(mb["game_moves"])[:-1]]), mb["game_moves"], mine)])
    for k in ("move_N", "move_W", "move_P", "move_root_N", "move_root_W", "move_action", "move_traversals", "move_player"):
        assert np.array_equal(ma[k], mb[k][keep]), k
    assert np.array_equal(ma["game_rng_draws"], mb["game_rng_draws"])


@pytest.mark.gpu
def test_one_captured_graph_serves_changing_tables():
    """The same engine and the same captured round: an iteration under table A, one under table B, one with openings off;
    one slot for several games, so the later games start from the table inside the graph.  Each run equals the oracle's,
    and the last one the golden trace of the reference."""
    import torch
    name = "othello_hash_400_8_4"
    cmd, golden = G.load("selfplay_" + name)
    c = dict(seed=cmd["seed"], sims=cmd["sims"], b=cmd["max_batch"], q=cmd["max_queue"], eps=cmd["eps"], alpha=cmd["alpha"])
    lines = opening_lines("othello")
    tables = [lines[:3], lines[2:][::-1], []]
    ngames = 4
    dev = torch.device("cuda", 0)
    with engine(capi.GAME_OTHELLO, capi.EVAL_HASHNET, c["seed"], c["sims"], c["b"], c["q"], ngames, 1, dir_eps=c["eps"],
                dir_alpha=c["alpha"]) as eng, torch.cuda.device(dev):
        graph = None
        for k, tab in enumerate(tables):
            first, n = (cmd["first_game"], cmd["ngames"]) if not tab else (60 + k, ngames)
            eng.set_openings(tab)
            eng.set_stream(torch.cuda.current_stream(dev).cuda_stream)
            eng.begin_iteration(first, n)
            if graph is None:
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    eng.set_stream(torch.cuda.current_stream(dev).cuda_stream)
                    eng.round()
                eng.set_stream(torch.cuda.current_stream(dev).cuda_stream)
            while True:
                for _ in range(16):
                    graph.replay()
                playing, failed = eng.poll()
                assert failed == 0
                if playing == 0:
                    break
            got = finish(eng, n, eng.collect_samples())
            ref = oracle_selfplay(tab, O.OG_OTHELLO, O.OE_HASHNET, c["seed"], first, n, c["sims"], c["b"], c["q"], c["eps"], c["alpha"])
            compare_selfplay(ref, got)
    compare_selfplay(golden, got)


@pytest.mark.gpu
def test_sharded_streamed_and_refused_openings():
    """Under openings: two engines playing the shards of world size 2 reproduce the unsharded run (a game's line follows
    its stream id); streamed samples equal the collected ones; sprl_set_openings refuses illegal and finished lines and a
    change while games are playing, and the previous table then stays in force."""
    from sprl_b200 import shard
    lines = opening_lines("othello")
    n, world = 10, 2
    kw = dict(seed=4, sims=48, max_batch=8, max_queue=4, dir_eps=0.25, dir_alpha=0.3, record_stats=1)
    with SP.Engine(capi.GAME_OTHELLO, capi.EVAL_HASHNET, num_slots=4, max_games=n, **kw) as eng:
        eng.set_openings(lines)
        samples = eng.run_iteration(n)
        whole = eng.move_stats(n)
    per_rank = []
    for r in range(world):
        first, stride, count = shard.shard_plan(n, r, world)
        with SP.Engine(capi.GAME_OTHELLO, capi.EVAL_HASHNET, num_slots=count, max_games=count, **kw) as eng:
            eng.set_openings(lines)
            eng.set_game_stride(stride)
            eng.run_iteration(count, first_game=first)
            ms = eng.move_stats(count)
            assert eng.check_guards()[1] == 0
        bounds = np.concatenate([[0], np.cumsum(ms["game_moves"])])
        per_rank.append([(ms["move_N"][bounds[k]:bounds[k + 1]], ms["move_action"][bounds[k]:bounds[k + 1]]) for k in range(count)])
    merged = shard.merge_shards(per_rank, world)
    bounds = np.concatenate([[0], np.cumsum(whole["game_moves"])])
    for g in range(n):
        assert np.array_equal(merged[g][0], whole["move_N"][bounds[g]:bounds[g + 1]]), g
        assert np.array_equal(merged[g][1], whole["move_action"][bounds[g]:bounds[g + 1]]), g

    with SP.Engine(capi.GAME_OTHELLO, capi.EVAL_HASHNET, num_slots=4, max_games=n, **kw) as eng:
        eng.set_openings(lines)
        eng.stream_samples(n * 8 * 70)
        eng.begin_iteration(0, n)
        eng.round()
        with pytest.raises(capi.SprlError) as ei:          # games are playing
            eng.set_openings([])
        assert ei.value.code == capi.SPRL_E_STATE
        while eng.poll()[0]:
            for _ in range(8):
                eng.round()
        got = eng.collect_samples()
        for a, b in zip(got, samples):
            assert np.array_equal(a, b)
        eng.stream_samples(0)
        mask = SP.env_line(capi.GAME_OTHELLO, [])["mask"][0]
        for bad in ([[int(np.nonzero(mask == 0)[0][0])]], [[19], [-1]], [[65]]):
            with pytest.raises(capi.SprlError) as ei:
                eng.set_openings(bad)
            assert ei.value.code == capi.SPRL_E_INVALID and "line" in str(ei.value) and "ply" in str(ei.value)
        with pytest.raises(capi.SprlError) as ei:          # Connect Four: a line that ends the game
            with SP.Engine(capi.GAME_C4, capi.EVAL_HASHNET, num_slots=2, max_games=2, sims=16) as c4:
                c4.set_openings([[3, 3], [3, 3, 4, 4, 2, 3, 1]])
        assert ei.value.code == capi.SPRL_E_INVALID and "line 1" in str(ei.value) and "terminal" in str(ei.value)
        assert np.array_equal(eng.run_iteration(n)[0], samples[0])      # the refused tables left the lines in force
        assert eng.check_guards()[1] == 0
