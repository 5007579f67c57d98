"""GPU parity tests (run on the B200 box): the CUDA path, called through the C ABI,
against the CPU oracle on the same seeded inputs and against the golden fixtures
produced by the unmodified reference.  Integer / index work is compared bit-exact;
fp32 search statistics are compared bit-exact too (the kernels keep the reference's
operand order, no FMA); sampled distributions within 1e-6 (pow)."""
import os

import numpy as np
import pytest

import golden_util as G
import oracle_py as O
from sprl_b200 import capi
from sprl_b200 import selfplay as SP

pytestmark = pytest.mark.gpu

GAMES = {"othello": capi.GAME_OTHELLO, "c4": capi.GAME_C4, "go": capi.GAME_GO7, "go9": capi.GAME_GO9}
EVALS = {"hash": capi.EVAL_HASHNET, "hash1": capi.EVAL_HASHNET, "uniform": capi.EVAL_UNIFORM,
         "heuristic": capi.EVAL_OTHELLO_HEURISTIC}
INITQ = {"parent": capi.INITQ_PARENT, "zero": capi.INITQ_ZERO, "drop": capi.INITQ_DROP_PARENT}
O_EVALS = {capi.EVAL_HASHNET: O.OE_HASHNET, capi.EVAL_UNIFORM: O.OE_UNIFORM, capi.EVAL_OTHELLO_HEURISTIC: O.OE_HEURISTIC}
MATCH_KEYS = ["game_moves", "game_winner", "game_rng_draws", "move_N", "move_W", "move_P", "move_root_N", "move_root_W",
              "move_action", "move_traversals", "move_player"]

EXACT_KEYS = ["game_moves", "game_rng_draws", "move_N", "move_W", "move_P", "move_root_N", "move_root_W",
              "move_action", "move_traversals", "move_player", "states", "outcomes"]


def test_device_present():
    assert capi.load().sprl_device_count() > 0, "no CUDA device: the GPU tests must not pass on a fallback"


# ------------------------------------------------------------------ environment
def test_perft_bit_exact():
    table = G.perft_table()
    for name, counts in table.items():
        for d, want in enumerate(counts, start=1):
            got, _ = SP.env_perft(GAMES[name], d)
            assert got == want, (name, d, got, want)
    # Othello perft(10): confirmed against the verbatim reference during the survey (SURVEY.md 8c)
    assert SP.env_perft(capi.GAME_OTHELLO, 10)[0] == 24571284
    # Othello perft(11): published value
    assert SP.env_perft(capi.GAME_OTHELLO, 11)[0] == 212258800
    # (Go 9x9 = the reference with the two constants of games/GoNode.hpp:16,20 edited, oracle/Makefile: ref9; Go 7x7
    # depth 4 = 5,536,331 from the verbatim reference)
    assert SP.env_perft(capi.GAME_OTHELLO, 0)[0] == 1


@pytest.mark.parametrize("name", G.ROLLOUT_FIXTURES)
def test_rollout_golden(name):
    cmd, ref = G.load("rollout_" + name)
    got = SP.env_rollout(GAMES[cmd["game"]], cmd["seed"], cmd["first_game"], cmd["ngames"], record=True)
    G.assert_trace_equal(ref, got)


@pytest.mark.parametrize("game,n", [(capi.GAME_OTHELLO, 2000), (capi.GAME_C4, 3000), (capi.GAME_GO7, 500), (capi.GAME_GO9, 120)])
def test_rollout_vs_oracle_state_by_state(game, n):
    got = SP.env_rollout(game, 77, 1000, n, record=True)
    ref = O.rollout(game, 77, 1000, n)
    G.assert_trace_equal(ref, got)
    assert got["total_positions"] == len(ref["player"])


def test_rollout_sweep_65536_games_state_by_state():
    """BASELINE.json config 2: 2^16 Othello rollouts compared state by state -- with the verbatim reference through the
    committed SHA-256 digests of its arrays (16 chunks of 4,096 games), and with the oracle on the first chunk."""
    fx = G.load_json("rollout_othello_65536.json")
    c = fx["cmd"]
    positions = 0
    for i, want in enumerate(fx["chunks"]):
        got = SP.env_rollout(GAMES[c["game"]], c["seed"], c["first_game"] + i * c["chunk"], c["chunk"], record=True)
        assert G.rollout_digests(got, c["chunk"])[0] == want, f"chunk {i}"
        positions += got["total_positions"]
        if i == 0:
            G.assert_trace_equal(O.rollout(G.GAME_ID[c["game"]], c["seed"], c["first_game"], c["chunk"]), got)
    assert positions == fx["positions"]


def test_rollout_large_sweep_properties():
    n = 1 << 18
    r = SP.env_rollout(capi.GAME_OTHELLO, 0, 0, n)
    assert r["game_steps"].min() >= 10 and r["game_steps"].max() <= 129
    assert r["total_positions"] == int(r["game_steps"].astype(np.int64).sum())
    # the first games of the sweep are the games of a small, recorded run
    small = SP.env_rollout(capi.GAME_OTHELLO, 0, 0, 64, record=True)
    assert np.array_equal(small["game_steps"], r["game_steps"][:64])
    assert np.array_equal(small["final_winner"], r["final_winner"][:64])
    assert set(np.unique(r["final_winner"])) <= {-1, 0, 1}


@pytest.mark.parametrize("game,ngames", [(capi.GAME_OTHELLO, 40), (capi.GAME_C4, 60), (capi.GAME_GO7, 12), (capi.GAME_GO9, 4)])
def test_env_line_replays_rollouts_position_by_position(game, ngames):
    """sprl_env_line (a chain of GameNode::getAddChild calls from the start position) against the roll-out traces, which the
    tests above pin to the oracle state by state: every position of every game -- cells, player, legal mask, terminal flag,
    winner -- for all four games (Go: the line is the superko history); an illegal action is refused."""
    r = SP.env_rollout(game, 5, 100, ngames, record=True)
    at = 0
    for g in range(ngames):
        n = int(r["game_steps"][g])
        sl = slice(at, at + n)
        line = SP.env_line(game, r["action"][sl][:-1])
        for k in ("cells", "player", "mask", "terminal", "winner"):
            assert np.array_equal(line[k], r[k][sl]), (g, k)
        at += n
    gi = capi.game_info(game)
    first = SP.env_line(game, [])
    illegal = [a for a in range(gi.actions) if not first["mask"][0][a]]
    if illegal:
        with pytest.raises(capi.SprlError):
            SP.env_line(game, [illegal[0]])
    with pytest.raises(capi.SprlError):
        SP.env_line(game, [gi.actions])


def test_env_step_matches_oracle_positions():
    for game in (O.OG_OTHELLO, O.OG_C4):
        ref = O.rollout(game, 3, 0, 200)
        idx = np.nonzero(ref["action"] >= 0)[0]
        out = SP.env_step(game, ref["cells"][idx], ref["player"][idx], ref["action"][idx])
        nxt = idx + 1
        assert np.array_equal(out["cells"], ref["cells"][nxt])
        assert np.array_equal(out["player"], ref["player"][nxt])
        assert np.array_equal(out["terminal"], ref["terminal"][nxt])
        assert np.array_equal(out["winner"], ref["winner"][nxt])
        assert np.array_equal(out["mask"], ref["mask"][nxt])
    assert SP.env_step(capi.GAME_OTHELLO, np.zeros((0, 64), np.int8), np.zeros(0, np.int8), np.zeros(0, np.int32))["cells"].shape == (0, 64)


# -------------------------------------------------------------------- self-play
def run_engine(game, evaluator, seed, first_game, ngames, sims, b, q, eps, alpha, noise, sym, initq, num_slots=None, **kw):
    with SP.Engine(game, evaluator, seed=seed, sims=sims, max_batch=b, max_queue=q, dir_eps=eps, dir_alpha=alpha,
                   add_noise=int(noise), use_sym=int(sym), init_q=initq, num_slots=num_slots or ngames,
                   max_games=ngames, record_stats=1, **kw) as eng:
        states, dists, outcomes = eng.run_iteration(ngames, first_game=first_game)
        got = eng.move_stats(ngames)
        pools, damaged = eng.check_guards()            # no kernel wrote outside its pools (every parity run checks)
        assert pools > 20 and damaged == 0
        got.update(states=states, distributions=dists, outcomes=outcomes, stats=eng.stats())
    return got


def compare_selfplay(ref, got):
    G.assert_trace_equal(ref, got, EXACT_KEYS)
    G.assert_trace_equal(ref, got, ["distributions"], exact=False)


@pytest.mark.parametrize("name", G.SELFPLAY_FIXTURES)
def test_selfplay_golden(name):
    cmd, ref = G.load("selfplay_" + name)
    got = run_engine(GAMES[cmd["game"]], EVALS[cmd["evaluator"]], cmd["seed"], cmd["first_game"], cmd["ngames"],
                     cmd["sims"], cmd["max_batch"], cmd["max_queue"], cmd["eps"], cmd["alpha"], cmd["noise"],
                     cmd["sym"], INITQ[cmd["initq"]])
    compare_selfplay(ref, got)


@pytest.mark.parametrize("game,ev,sims,b,q,alpha,ngames,slots", [
    (capi.GAME_OTHELLO, "hash", 400, 8, 4, 0.3, 24, 24),
    (capi.GAME_OTHELLO, "hash", 100, 8, 4, 0.3, 40, 7),       # slots reused by several games
    (capi.GAME_OTHELLO, "uniform", 64, 1, 1, 0.3, 16, 16),
    (capi.GAME_OTHELLO, "hash", 150, 32, 32, 0.3, 8, 8),      # wide queue
    (capi.GAME_C4, "hash", 512, 8, 4, 0.5, 24, 5),
    (capi.GAME_C4, "uniform", 200, 8, 4, 0.5, 16, 16),
    (capi.GAME_GO7, "hash", 100, 16, 8, 0.2, 6, 6),
    (capi.GAME_GO9, "hash", 60, 16, 8, 0.2, 3, 3),
])
def test_selfplay_vs_oracle(game, ev, sims, b, q, alpha, ngames, slots):
    seed, first = 1234, 500
    ref = O.selfplay(game, O.OE_HASHNET if ev == "hash" else O.OE_UNIFORM, seed, first, ngames, sims, b, q, 0.25, alpha,
                     max_moves_per_game=170)
    got = run_engine(game, EVALS[ev], seed, first, ngames, sims, b, q, 0.25, alpha, 1, 1, capi.INITQ_PARENT, num_slots=slots)
    compare_selfplay(ref, got)
    st, rs = got["stats"], ref["stats"]
    assert st["sims"] == rs["total_traversals"] and st["evals"] == rs["total_evals"]
    assert st["leaves_terminal"] == rs["leaves_terminal"] and st["leaves_gray"] == rs["leaves_gray"]
    assert st["depth_sum"] == int(rs["select_depth_sum"]) and st["legal_sum"] == int(rs["select_legal_sum"])


def test_selfplay_variants_vs_oracle():
    # no symmetrizer, no noise, InitQ::ZERO
    for noise, sym, initq, oq in [(0, 0, capi.INITQ_ZERO, O.OQ_ZERO), (1, 0, capi.INITQ_PARENT, O.OQ_PARENT), (0, 1, capi.INITQ_ZERO, O.OQ_ZERO)]:
        ref = O.selfplay(O.OG_OTHELLO, O.OE_HASHNET, 9, 0, 4, 80, 8, 4, 0.25, 0.3, add_noise=bool(noise), use_sym=bool(sym), init_q=oq)
        got = run_engine(capi.GAME_OTHELLO, capi.EVAL_HASHNET, 9, 0, 4, 80, 8, 4, 0.25, 0.3, noise, sym, initq)
        compare_selfplay(ref, got)


def test_results_do_not_depend_on_slot_count():
    a = run_engine(capi.GAME_OTHELLO, capi.EVAL_HASHNET, 5, 0, 12, 60, 8, 4, 0.25, 0.3, 1, 1, capi.INITQ_PARENT, num_slots=12)
    b = run_engine(capi.GAME_OTHELLO, capi.EVAL_HASHNET, 5, 0, 12, 60, 8, 4, 0.25, 0.3, 1, 1, capi.INITQ_PARENT, num_slots=5,
                   rounds_per_launch=3)
    for k in EXACT_KEYS + ["distributions"]:
        assert np.array_equal(a[k], b[k]), k


def test_capacity_overflow_is_reported():
    with pytest.raises(capi.SprlError) as ei:
        run_engine(capi.GAME_OTHELLO, capi.EVAL_HASHNET, 5, 0, 2, 400, 8, 4, 0.25, 0.3, 1, 1, capi.INITQ_PARENT, units_per_tree=600)
    assert ei.value.code == capi.SPRL_E_CAPACITY


def test_sample_round_trip_properties():
    """Size-independent properties at a larger scale: every sample block of 8 is the D4 orbit
    of its first element; distributions sum to 1; outcomes are in {-1,0,1} and flip with the mover."""
    with SP.Engine(capi.GAME_OTHELLO, capi.EVAL_UNIFORM, seed=3, sims=50, max_batch=8, max_queue=4, num_slots=256, max_games=512) as eng:
        states, dists, outcomes = eng.run_iteration(512)
        st = eng.stats()
    assert st["games"] == 512 and states.shape[0] == 8 * st["moves"]
    assert np.allclose(dists.sum(1), 1.0, atol=1e-5)
    assert set(np.unique(outcomes)) <= {-1.0, 0.0, 1.0}
    s = states.reshape(-1, 8, 3, 8, 8)
    assert np.array_equal(s[:, 4], s[:, 0][..., ::-1])                      # symmetry 4 = column flip
    assert np.array_equal(s[:, 2], s[:, 0][..., ::-1, ::-1])                # symmetry 2 = rotation by 180
    assert np.array_equal(s[:, 7], np.swapaxes(s[:, 0], -1, -2))            # symmetry 7 = transpose
    d = dists.reshape(-1, 8, 65)
    assert np.array_equal(d[:, 4, :64].reshape(-1, 8, 8), d[:, 0, :64].reshape(-1, 8, 8)[..., ::-1])
    assert np.array_equal(d[:, :, 64], np.repeat(d[:, :1, 64], 8, 1))
    o = outcomes.reshape(-1, 8)
    assert (o == o[:, :1]).all()
    colour = s[:, 0, 2, 0, 0]                                                # 1.0 when player ZERO moved
    assert set(np.unique(colour)) <= {0.0, 1.0}


def test_headline_configuration_at_scale():
    """BASELINE.json's configuration (Othello, 400 sims/move, 8/4 leaf batching, D4 symmetry, Dirichlet 0.25 / 0.3,
    InitQ::PARENT) over 1,024 concurrent games: the first games are bit-identical to the oracle's (a game's result does
    not depend on how many other games share the GPU), and the whole iteration satisfies the reference's invariants."""
    n, head = 1024, 3
    with SP.Engine(capi.GAME_OTHELLO, capi.EVAL_HASHNET, seed=0, sims=400, max_batch=8, max_queue=4, dir_eps=0.25, dir_alpha=0.3,
                   num_slots=n, max_games=n, record_stats=1) as eng:
        states, dists, outcomes = eng.run_iteration(n)
        got = eng.move_stats(n)
        st = eng.stats()
    ref = O.selfplay(O.OG_OTHELLO, O.OE_HASHNET, 0, 0, head, 400, 8, 4, 0.25, 0.3)
    m = int(ref["game_moves"].sum())
    assert np.array_equal(got["game_moves"][:head], ref["game_moves"]) and np.array_equal(got["game_rng_draws"][:head], ref["game_rng_draws"])
    for k in ("move_N", "move_W", "move_P", "move_root_N", "move_root_W", "move_action", "move_traversals", "move_player"):
        assert np.array_equal(got[k][:m], ref[k]), k
    assert np.array_equal(states[:8 * m], ref["states"]) and np.array_equal(outcomes[:8 * m], ref["outcomes"])
    # invariants over all games (SURVEY 8a: Q7 whole batches, Q2/Q4 root visit bookkeeping, A17 sample layout)
    assert st["games"] == n and states.shape[0] == dists.shape[0] == outcomes.shape[0] == 8 * st["moves"]
    assert (got["move_traversals"] >= 400).all() and (got["move_traversals"] < 408).all()
    assert np.array_equal(got["move_N"].sum(1) <= got["move_traversals"], np.ones(len(got["move_traversals"]), bool))
    first = np.concatenate([[0], np.cumsum(got["game_moves"])[:-1]])
    assert np.array_equal(got["move_root_N"][first], got["move_traversals"][first].astype(np.float32))      # fresh root: N() = its own descents
    assert np.array_equal(got["move_N"][first].sum(1), got["move_traversals"][first] - 4)                   # Q4: queued 4 times before it expands
    assert np.allclose(dists.sum(1), 1.0, atol=1e-5) and (dists >= 0).all()
    assert set(np.unique(outcomes)) <= {-1.0, 0.0, 1.0}
    assert 50 <= got["game_moves"].mean() <= 64 and got["game_moves"].max() <= 128
    assert st["sims"] == int(got["move_traversals"].astype(np.int64).sum())


# ------------------------------------------------- external evaluator (the traced-network path)
from integer_net import IntegerNet  # noqa: E402  (exact in fp32 on any device)


@pytest.mark.parametrize("game,sims,b,q,alpha,ngames,graph", [
    (capi.GAME_OTHELLO, 120, 8, 4, 0.3, 12, False),
    (capi.GAME_OTHELLO, 64, 8, 4, 0.3, 6, True),           # search launch + forward replayed as one CUDA graph
    (capi.GAME_C4, 100, 8, 4, 0.5, 8, False),
    (capi.GAME_GO7, 48, 16, 8, 0.2, 3, False),             # 8 history boards: 17 input planes
])
def test_external_evaluator_bit_exact(game, sims, b, q, alpha, ngames, graph):
    import torch
    gi = capi.game_info(game)
    net = IntegerNet(2 * gi.history + 1, gi.cells, gi.actions, seed=game)
    ref = O.selfplay(game, O.OE_CALLBACK, 21, 0, ngames, sims, b, q, 0.25, alpha, eval_fn=net.numpy, max_moves_per_game=170)
    with SP.Engine(game, capi.EVAL_EXTERNAL, seed=21, sims=sims, max_batch=b, max_queue=q, dir_eps=0.25, dir_alpha=alpha,
                   num_slots=ngames, max_games=ngames, record_stats=1) as eng:
        eng.attach_network(net.torch_fn(torch.device("cuda", 0)), use_cuda_graph=graph)
        states, dists, outcomes = eng.run_iteration(ngames)
        got = eng.move_stats(ngames)
        got.update(states=states, distributions=dists, outcomes=outcomes)
        st = eng.stats()
        assert eng.check_guards()[1] == 0
    assert net.calls > 0
    compare_selfplay(ref, got)
    assert st["sims"] == ref["stats"]["total_traversals"] and st["evals"] == ref["stats"]["total_evals"]
    # quirk Q4: the fresh root alone is queued max_queue times in the first batch of a game; the copies are counted like the
    # reference's getNumEvals but share one evaluator row.  The bound holds for q <= 32: only the first 32 entries of a
    # batch are compared (tests/test_search_edges.py checks the exact count for wider queues)
    assert (q - 1) * ngames <= st["leaves_duplicate"] < st["evals"] // 2


def test_reused_engine_and_captured_graph_follow_the_new_iteration():
    """One Engine, one captured CUDA graph, two iterations with different first_game / num_games and fewer slots than
    games: slots start later games on the device, so the stream ids and the game count must come from the iteration
    that is running, not from the one the graph was captured in (per-iteration values live in device memory)."""
    import torch
    game, sims, b, q = capi.GAME_OTHELLO, 48, 8, 4
    gi = capi.game_info(game)
    net = IntegerNet(2 * gi.history + 1, gi.cells, gi.actions, seed=3)
    with SP.Engine(game, capi.EVAL_EXTERNAL, seed=9, sims=sims, max_batch=b, max_queue=q, dir_eps=0.25, dir_alpha=0.3,
                   num_slots=3, max_games=16, record_stats=1) as eng:
        eng.attach_network(net.torch_fn(torch.device("cuda", 0)), use_cuda_graph=True)
        for first, ngames in ((0, 7), (1000, 10), (40, 4)):
            ref = O.selfplay(game, O.OE_CALLBACK, 9, first, ngames, sims, b, q, 0.25, 0.3, eval_fn=net.numpy, max_moves_per_game=170)
            states, dists, outcomes = eng.run_iteration(ngames, first_game=first)
            got = eng.move_stats(ngames)
            got.update(states=states, distributions=dists, outcomes=outcomes)
            compare_selfplay(ref, got)


# ------------------------------------------------- step-wise trees: UCTTree's own surface through the C ABI
def walk_trees(eng, ngames, sims, first_game):
    """A caller of the step-wise ABI that does what ref_trace `treewalk` does with the reference's UCTTree: search,
    read the decision node, play the FIRST most-visited action, advance -- all trees in lock step."""
    A = eng.gi.actions
    rows = [[] for _ in range(ngames)]
    eng.begin_trees(ngames, first_game=first_game)
    live = np.ones(ngames, bool)
    while live.any():
        eng.search(sims)
        st = eng.root_stats()
        assert (st["terminal"][live] == 0).all()
        assert ((st["N"] > 0) <= (st["mask"] > 0)).all()            # visits only on legal actions
        actions = np.where(live, st["N"].argmax(1), -1).astype(np.int32)
        for g in np.nonzero(live)[0]:
            rows[g].append({k: st[k][g].copy() for k in ("N", "W", "P", "root_N", "root_W", "traversals", "player")} | {"action": actions[g]})
        eng.advance(actions)
        live &= eng.root_stats()["terminal"] == 0
    flat = [r for g in range(ngames) for r in rows[g]]
    got = dict(game_moves=np.array([len(r) for r in rows], np.int32),
               move_N=np.stack([r["N"] for r in flat]), move_W=np.stack([r["W"] for r in flat]), move_P=np.stack([r["P"] for r in flat]),
               move_root_N=np.array([r["root_N"] for r in flat], np.float32), move_root_W=np.array([r["root_W"] for r in flat], np.float32),
               move_action=np.array([r["action"] for r in flat], np.int32), move_traversals=np.array([r["traversals"] for r in flat], np.int32),
               move_player=np.array([r["player"] for r in flat], np.int8), game_winner=eng.root_stats()["winner"].astype(np.int32))
    assert got["move_N"].shape[1] == A
    return got


STEP_KEYS = ["game_moves", "game_winner", "move_N", "move_W", "move_P", "move_root_N", "move_root_W", "move_action", "move_traversals", "move_player"]


@pytest.mark.parametrize("name", G.TREEWALK_FIXTURES)
def test_stepwise_trees_golden(name):
    """sprl_begin_trees / sprl_search / sprl_root_stats / sprl_advance against the verbatim reference driven through
    its public UCTTree API (uct/UCTTree.hpp:62-210) by a caller that plays the first most-visited action: every
    decision node of every game, N / W / P bit for bit (Dirichlet noise and symmetries on)."""
    cmd, ref = G.load("treewalk_" + name)
    with SP.Engine(GAMES[cmd["game"]], EVALS[cmd["evaluator"]], seed=cmd["seed"], sims=cmd["sims"], max_batch=cmd["max_batch"],
                   max_queue=cmd["max_queue"], dir_eps=cmd["eps"], dir_alpha=cmd["alpha"], add_noise=cmd["noise"], use_sym=cmd["sym"],
                   init_q=INITQ[cmd["initq"]], num_slots=cmd["ngames"], max_games=cmd["ngames"]) as eng:
        got = walk_trees(eng, cmd["ngames"], cmd["sims"], cmd["first_game"])
        playing, failed = eng.poll()
    assert playing == 0 and failed == 0
    G.assert_trace_equal(ref, got, STEP_KEYS)


def test_stepwise_trees_vs_oracle_with_a_network_and_fewer_trees_than_slots():
    """The same walk with the external evaluator (planes -> network -> logits between the two halves of every loop
    trip) against the oracle; then illegal actions are refused."""
    import torch
    game, sims, b, q, ngames = capi.GAME_OTHELLO, 40, 8, 4, 5
    gi = capi.game_info(game)
    net = IntegerNet(2 * gi.history + 1, gi.cells, gi.actions, seed=8)
    ref = O.selfplay(game, O.OE_CALLBACK, 13, 200, ngames, sims, b, q, 0.25, 0.3, eval_fn=net.numpy, caller_moves=True, max_moves_per_game=170)
    with SP.Engine(game, capi.EVAL_EXTERNAL, seed=13, sims=sims, max_batch=b, max_queue=q, dir_eps=0.25, dir_alpha=0.3,
                   num_slots=8, max_games=8) as eng:
        eng.attach_network(net.torch_fn(torch.device("cuda", 0)), use_cuda_graph=False)
        got = walk_trees(eng, ngames, sims, 200)
        G.assert_trace_equal(ref, got, [k for k in STEP_KEYS if k != "game_winner"])
        eng.begin_trees(2)
        with pytest.raises(capi.SprlError) as err:
            eng.advance(np.array([0, 19], np.int32))          # a1 is not a legal first move (d3 is)
        assert "not legal" in str(err.value)
    with SP.Engine(game, capi.EVAL_UNIFORM, num_slots=2, max_games=2, sims=16) as eng:
        with pytest.raises(capi.SprlError):
            eng.search(8)                                     # no trees begun


def test_external_evaluator_needs_a_network():
    with SP.Engine(capi.GAME_OTHELLO, capi.EVAL_EXTERNAL, num_slots=2, max_games=2, sims=16) as eng:
        with pytest.raises(capi.SprlError):
            eng.run_iteration(2)


def test_traced_network_matches_cpu_forward():
    """The LibTorch boundary (SURVEY.md 8c: parity unpinned by the reference): the same traced
    module in fp32 on the GPU (TF32 off) against its CPU forward, |dlogit| <= 1e-4."""
    import torch
    from sprl_b200.network import make_network, trace_network
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    net = make_network("othello", 0)
    x = (torch.rand(512, 3, 8, 8) > 0.5).float()
    with torch.no_grad():
        lg_cpu, v_cpu = net(x)
        lg_gpu, v_gpu = trace_network(make_network("othello", 0), torch.device("cuda", 0))(x.cuda())
    assert (lg_gpu.cpu() - lg_cpu).abs().max().item() <= 1e-4
    assert (v_gpu.cpu() - v_cpu).abs().max().item() <= 1e-4


# ---------------------------------------------------------------------- sharding across ranks
def test_sharded_generation_equals_unsharded():
    """Games are keyed by their id, not by the rank that plays them: two engines playing the
    shards of world_size 2 (game_id % 2, as bench.py does per GPU) reproduce the unsharded run."""
    from sprl_b200 import shard
    n, world = 10, 2
    kw = dict(seed=4, sims=60, max_batch=8, max_queue=4, dir_eps=0.25, dir_alpha=0.3, record_stats=1)
    with SP.Engine(capi.GAME_OTHELLO, capi.EVAL_HASHNET, num_slots=n, max_games=n, **kw) as eng:
        eng.run_iteration(n)
        whole = eng.move_stats(n)
    per_rank = []
    for r in range(world):
        first, stride, count = shard.shard_plan(n, r, world)
        with SP.Engine(capi.GAME_OTHELLO, capi.EVAL_HASHNET, num_slots=count, max_games=count, **kw) as eng:
            eng.set_game_stride(stride)
            eng.run_iteration(count, first_game=first)
            ms = eng.move_stats(count)
        bounds = np.concatenate([[0], np.cumsum(ms["game_moves"])])
        per_rank.append([(ms["move_N"][bounds[k]:bounds[k + 1]], ms["move_action"][bounds[k]:bounds[k + 1]]) for k in range(count)])
    merged = shard.merge_shards(per_rank, world)
    bounds = np.concatenate([[0], np.cumsum(whole["game_moves"])])
    for g in range(n):
        assert np.array_equal(merged[g][0], whole["move_N"][bounds[g]:bounds[g + 1]]), g
        assert np.array_equal(merged[g][1], whole["move_action"][bounds[g]:bounds[g + 1]]), g


def test_streamed_samples_equal_the_collected_ones():
    """sprl_stream_samples: finished games leave for the (page-locked) host arrays while the others still play -- more
    games than slots, so most of them finish early; the result is the array collect_samples() builds at the end, bit for
    bit, for a second iteration on the same registration too, and a too small capacity is reported."""
    kw = dict(seed=4, sims=32, max_batch=8, max_queue=4, num_slots=24, max_games=400)
    with SP.Engine(capi.GAME_OTHELLO, capi.EVAL_HASHNET, **kw) as eng:
        want = [eng.run_iteration(n, first_game=f) for n, f in ((400, 0), (150, 1000))]
    with SP.Engine(capi.GAME_OTHELLO, capi.EVAL_HASHNET, **kw) as eng:
        eng.stream_samples(400 * 8 * 70)
        for (n, f), ref in zip(((400, 0), (150, 1000)), want):
            eng.begin_iteration(f, n)
            chunks = []
            while True:
                for _ in range(8):
                    eng.round()
                playing, failed = eng.poll()
                chunks.append(eng.stream_info()["games_done"])
                if playing == 0:
                    break
            got = eng.collect_samples()
            assert 0 < chunks[len(chunks) // 2] < n          # half way through, some games had left and some had not
            for a, b in zip(got, ref):
                assert np.array_equal(a, b)
        assert eng.stream_info()["chunks_while_playing"] > 4
        eng.stream_samples(1000)                              # far too small
        with pytest.raises(capi.SprlError):
            eng.run_iteration(40)
        eng.stream_samples(0)
        assert eng.run_iteration(40)[0].shape[0] > 40 * 8 * 20


def test_device_resident_samples_alias_the_host_copy():
    """N1: samples handed over on the device are the arrays collect_samples() copies to the host."""
    import torch
    with SP.Engine(capi.GAME_OTHELLO, capi.EVAL_HASHNET, seed=2, sims=40, max_batch=8, max_queue=4, num_slots=6, max_games=6) as eng:
        states, dists, outcomes = eng.run_iteration(6)
        ds, dd, do = eng.collect_samples_device()
        assert ds.is_cuda and ds.shape == states.shape and dd.shape == dists.shape and do.shape == outcomes.shape
        assert np.array_equal(ds.cpu().numpy(), states) and np.array_equal(dd.cpu().numpy(), dists)
        assert np.array_equal(do.cpu().numpy(), outcomes)
        loss = (dd * torch.log(dd.clamp_min(1e-9))).sum()          # usable by torch without a copy
        assert torch.isfinite(loss)


# ------------------------------------------------------- next rows: DROP_PARENT, OthelloHeuristic, match play
@pytest.mark.parametrize("game,ev,initq,sims,b,q,alpha,ngames,slots", [
    (capi.GAME_OTHELLO, capi.EVAL_HASHNET, "drop", 200, 8, 4, 0.3, 12, 5),
    (capi.GAME_OTHELLO, capi.EVAL_OTHELLO_HEURISTIC, "parent", 120, 8, 4, 0.3, 10, 10),
    (capi.GAME_OTHELLO, capi.EVAL_OTHELLO_HEURISTIC, "drop", 64, 4, 2, 0.3, 6, 3),
    (capi.GAME_C4, capi.EVAL_HASHNET, "drop", 256, 8, 4, 0.5, 12, 12),
    (capi.GAME_GO7, capi.EVAL_HASHNET, "drop", 80, 16, 8, 0.2, 4, 4),
])
def test_drop_parent_and_heuristic_vs_oracle(game, ev, initq, sims, b, q, alpha, ngames, slots):
    """InitQ::DROP_PARENT (uct/UCTNode.hpp:152-163,196-206) and networks/OthelloHeuristic.cpp on the device."""
    seed, first = 99, 20
    oq = {"drop": O.OQ_DROP_PARENT, "parent": O.OQ_PARENT}[initq]
    ref = O.selfplay(game, O_EVALS[ev], seed, first, ngames, sims, b, q, 0.25, alpha, init_q=oq, max_moves_per_game=170)
    got = run_engine(game, ev, seed, first, ngames, sims, b, q, 0.25, alpha, 1, 1, INITQ[initq], num_slots=slots)
    compare_selfplay(ref, got)


def test_heuristic_is_othello_only():
    with pytest.raises(capi.SprlError):
        SP.Engine(capi.GAME_C4, capi.EVAL_OTHELLO_HEURISTIC, num_slots=2)


def run_match(game, agents, seed, first_game, ngames, sims, b, q, pairs=None):
    """Match play through the C ABI with Evaluate.cpp's constants (noise on, eps 0.25, alpha 0.1, uWeight 1.0)."""
    pairs = pairs or ngames
    with SP.Engine(game, capi.EVAL_UNIFORM, seed=seed, sims=sims, max_batch=b, max_queue=q, dir_eps=0.25, dir_alpha=0.1,
                   u_weight=1.0, add_noise=1, num_slots=2 * pairs, max_games=ngames, record_stats=1) as eng:
        got = eng.run_match(agents, ngames, first_game=first_game)
        got.update(eng.move_stats(ngames))
    return got


def gpu_agents(cmd):
    return [dict(evaluator=EVALS[cmd["evaluators"][k]], hash_salt=G.HASH_SALT.get(cmd["evaluators"][k], 0),
                 use_sym=cmd["sym"][k], init_q=INITQ[cmd["initq"][k]]) for k in range(2)]


@pytest.mark.parametrize("name", G.MATCH_FIXTURES)
def test_match_golden(name):
    """Evaluate.cpp's match path against the verbatim reference: every root statistic, action and winner."""
    cmd, ref = G.load("match_" + name)
    got = run_match(GAMES[cmd["game"]], gpu_agents(cmd), cmd["seed"], cmd["first_game"], cmd["ngames"], cmd["sims"],
                    cmd["max_batch"], cmd["max_queue"])
    ref = dict(ref, game_winner=ref["game_winner"].astype(np.int8))
    G.assert_trace_equal(ref, got, MATCH_KEYS)


@pytest.mark.parametrize("game,evs,syms,qs,sims,b,q,ngames,pairs", [
    (capi.GAME_OTHELLO, ("hash", "hash1"), (1, 1), ("parent", "zero"), 100, 8, 4, 16, 5),     # pairs reused by several games
    (capi.GAME_OTHELLO, ("heuristic", "hash"), (1, 0), ("drop", "parent"), 60, 8, 4, 8, 8),
    (capi.GAME_C4, ("hash", "uniform"), (1, 1), ("parent", "parent"), 128, 8, 4, 24, 24),
    (capi.GAME_GO7, ("hash", "hash1"), (1, 1), ("parent", "parent"), 48, 16, 8, 3, 3),
    (capi.GAME_GO9, ("hash1", "hash"), (0, 1), ("zero", "parent"), 32, 16, 8, 2, 1),
])
def test_match_vs_oracle(game, evs, syms, qs, sims, b, q, ngames, pairs):
    seed, first = 7, 11                                   # odd first game: agent 1 opens game 0
    oq = {"drop": O.OQ_DROP_PARENT, "parent": O.OQ_PARENT, "zero": O.OQ_ZERO}
    o_agents = [dict(evaluator=O_EVALS[EVALS[evs[k]]], hash_salt=G.HASH_SALT.get(evs[k], 0), use_sym=syms[k], init_q=oq[qs[k]])
                for k in range(2)]
    g_agents = [dict(evaluator=EVALS[evs[k]], hash_salt=G.HASH_SALT.get(evs[k], 0), use_sym=syms[k], init_q=INITQ[qs[k]])
                for k in range(2)]
    ref = O.match(game, o_agents, seed, first, ngames, sims, b, q, max_moves_per_game=170)
    got = run_match(game, g_agents, seed, first, ngames, sims, b, q, pairs=pairs)
    ref["game_winner"] = ref["game_winner"].astype(np.int8)
    G.assert_trace_equal(ref, got, MATCH_KEYS)
    assert got["wins"] == ref["wins"] and got["draws"] == ref["draws"]
    assert got["wins"][0] + got["wins"][1] + got["draws"] == ngames


def test_match_move_without_any_visit_is_the_first_legal_action():
    """With sims <= max_queue an agent's search ends after the descent that evaluates its (always fresh) root: every edge
    has 0 visits.  The reference's std::max_element then returns action 0 whether or not it is legal
    (agents/UCTNetworkAgent.hpp:92-93) and walks into an illegal child; the engine plays the first LEGAL action instead
    (search.cu: finalize_match_move) -- the one documented departure of match play, pinned here: every move of every game
    has all-zero visit counts and is the lowest legal action, and the games end with a result."""
    agents = [dict(evaluator=capi.EVAL_UNIFORM, hash_salt=0, use_sym=0, init_q=capi.INITQ_PARENT)] * 2
    got = run_match(capi.GAME_OTHELLO, agents, 3, 0, 4, 1, 1, 1)
    n = len(got["move_action"])
    assert n > 4 * 20
    assert not got["move_N"].any()
    for m in range(n):
        legal = np.flatnonzero(got["move_P"][m] > 0)
        assert legal.size > 0 and got["move_action"][m] == legal[0]
    assert got["wins"][0] + got["wins"][1] + got["draws"] == 4


@pytest.mark.parametrize("game,sims,b,q,ngames,pairs,graph,second", [
    (capi.GAME_OTHELLO, 64, 8, 4, 6, 3, False, "net"),
    (capi.GAME_OTHELLO, 48, 8, 4, 4, 4, True, "net"),          # round + both forwards replayed as one CUDA graph
    (capi.GAME_C4, 80, 8, 4, 8, 8, False, "uniform"),          # a network against the uniform evaluator
])
def test_match_external_evaluators_bit_exact(game, sims, b, q, ngames, pairs, graph, second):
    """Two networks in one match: each reads its half of the leaf batch (planes written by the search kernel) and
    writes its half of the logits / values; integer-exact networks, so the oracle's callbacks agree bit for bit."""
    import torch
    gi = capi.game_info(game)
    nets = [IntegerNet(2 * gi.history + 1, gi.cells, gi.actions, seed=5 + k) for k in range(2)]
    o_agents = [dict(evaluator=O.OE_CALLBACK, eval_fn=nets[0].numpy, use_sym=1, init_q=O.OQ_PARENT),
                dict(evaluator=O.OE_CALLBACK, eval_fn=nets[1].numpy, use_sym=1, init_q=O.OQ_ZERO)]
    g_agents = [dict(evaluator=capi.EVAL_EXTERNAL, use_sym=1, init_q=capi.INITQ_PARENT),
                dict(evaluator=capi.EVAL_EXTERNAL, use_sym=1, init_q=capi.INITQ_ZERO)]
    if second == "uniform":
        o_agents[1] = dict(evaluator=O.OE_UNIFORM, use_sym=1, init_q=O.OQ_ZERO)
        g_agents[1] = dict(evaluator=capi.EVAL_UNIFORM, use_sym=1, init_q=capi.INITQ_ZERO)
    ref = O.match(game, o_agents, 3, 0, ngames, sims, b, q, max_moves_per_game=170)
    dev = torch.device("cuda", 0)
    with SP.Engine(game, capi.EVAL_EXTERNAL, seed=3, sims=sims, max_batch=b, max_queue=q, dir_eps=0.25, dir_alpha=0.1,
                   u_weight=1.0, add_noise=1, num_slots=2 * pairs, max_games=ngames, record_stats=1) as eng:
        eng.attach_match_evaluators([nets[0].torch_fn(dev), nets[1].torch_fn(dev) if second == "net" else None],
                                    use_cuda_graph=graph)
        got = eng.run_match(g_agents, ngames)
        got.update(eng.move_stats(ngames))
        if graph:
            # a second match on the same engine and the same captured graph, other agent options and game ids
            o2 = [dict(o_agents[0], use_sym=0, init_q=O.OQ_ZERO), dict(o_agents[1], init_q=O.OQ_PARENT)]
            g2 = [dict(g_agents[0], use_sym=0, init_q=capi.INITQ_ZERO), dict(g_agents[1], init_q=capi.INITQ_PARENT)]
            ref2 = O.match(game, o2, 3, 77, ngames - 1, sims, b, q, max_moves_per_game=170)
            got2 = eng.run_match(g2, ngames - 1, first_game=77)
            got2.update(eng.move_stats(ngames - 1))
            ref2["game_winner"] = ref2["game_winner"].astype(np.int8)
            G.assert_trace_equal(ref2, got2, MATCH_KEYS)
    ref["game_winner"] = ref["game_winner"].astype(np.int8)
    G.assert_trace_equal(ref, got, MATCH_KEYS)
    assert got["wins"] == ref["wins"] and got["draws"] == ref["draws"]


@pytest.mark.parametrize("game,ev,sims,alpha,ngames", [(capi.GAME_OTHELLO, "hash", 120, 0.3, 8), (capi.GAME_OTHELLO, "uniform", 64, 0.3, 6),
                                                       (capi.GAME_C4, "hash", 128, 0.5, 10), (capi.GAME_GO7, "hash", 60, 0.2, 3)])
def test_fix_symmetry_mask_option_vs_oracle(game, ev, sims, alpha, ngames):
    """The non-default repair of quirk Q3 (the legal mask is symmetrised with the state): bit-exact against the oracle
    run with the same option, and every visited move of every root then has a positive prior."""
    oe = O.OE_HASHNET if ev == "hash" else O.OE_UNIFORM
    b, q = (16, 8) if game == capi.GAME_GO7 else (8, 4)
    ref = O.selfplay(game, oe, 31, 0, ngames, sims, b, q, 0.25, alpha, add_noise=False, fix_symmetry_mask=True, max_moves_per_game=170)
    got = run_engine(game, EVALS[ev], 31, 0, ngames, sims, b, q, 0.25, alpha, 0, 1, capi.INITQ_PARENT, fix_symmetry_mask=1)
    compare_selfplay(ref, got)
    assert (got["move_P"][got["move_N"] > 0] > 0).all()
    if game == capi.GAME_OTHELLO:      # with the quirk, roots whose legal set is not symmetric lose priors
        quirk = O.selfplay(game, oe, 31, 0, ngames, sims, b, q, 0.25, alpha, add_noise=False, max_moves_per_game=170)
        assert not np.array_equal(quirk["move_P"][:8], got["move_P"][:8])


def test_python_run_worker_writes_the_reference_files(tmp_path):
    """SPRL::runWorker's file contract through the Python worker: iteration 0 with the uniform evaluator, iteration 1
    with the controller's traced module (run by the library evaluator), three .npy files per iteration."""
    import torch
    from sprl_b200.network import make_network, trace_network
    root = str(tmp_path)
    os.makedirs(os.path.join(root, "data", "models", "unit"))
    trace_network(make_network("othello", 0), "cpu").save(os.path.join(root, "data", "models", "unit", "traced_unit_iteration_0.pt"))
    save_dir = os.path.join(root, "data", "games", "unit", "0", "3")
    SP.run_worker("unit", save_dir, capi.GAME_OTHELLO, 2, 12, 32, 1, 1, 12, 48, 8, 4, 0.25, 0.3, root=root, wait_interval=0.1, settle=0.0)
    for it in (0, 1):
        base = os.path.join(save_dir, f"unit_iteration_{it}")
        s, d, o = np.load(base + "_states.npy"), np.load(base + "_distributions.npy"), np.load(base + "_outcomes.npy")
        assert s.shape[1:] == (3, 8, 8) and d.shape == (s.shape[0], 65) and o.shape == (s.shape[0],)
        assert s.shape[0] % 8 == 0 and s.shape[0] >= 12 * 8 * 20
        assert np.allclose(d.sum(1), 1, atol=1e-5) and set(np.unique(o)) <= {-1.0, 0.0, 1.0}
        assert open(base + "_outcomes.npy", "rb").read(8) == b"\x93NUMPY\x01\x00"
