"""The search kernel at the two edges the other parity tests never reach, bit for bit against the CPU oracle.

Deep descents.  select_leaf records the edges of a descent for the one-lane-per-level backup (backup_path) only up to
DESCENT_MAX = 32; a descent of 32 or more edges is backed up by walking parent links (backup), for terminal leaves,
gray leaves and leaves queued for the evaluator alike.  HashNet, uniform and heuristic evaluators keep descents under
30 edges at the usual settings; a network with a sharp policy (a trained one, or the spiked one below) goes deeper
than 32 on most moves.

Wide leaf queues.  search_batch deduplicates the queue of one batch over its first 32 entries only: a copy among them
shares the first copy's evaluator row and counts as a duplicate; every entry from the 33rd on gets its own row
(popc(first_mask) + q - 32) and its own planes, whether or not it repeats a leaf.

The CPU tests ask the oracle whether each configuration really reaches the edge it is here for, so that the GPU tests
cannot pass without exercising it.  Every GPU run is also checked for writes outside the engine's pools."""
import functools

import numpy as np
import pytest

import golden_util as G
import oracle_py as O
from integer_net import IntegerNet
from sprl_b200 import capi

DESCENT_MAX = 32
MAX_MOVES = {"othello": 130, "go": 200, "go9": 330}        # oracle capacity per game (moves)
GAME_IDS = {"othello": O.OG_OTHELLO, "go": O.OG_GO7, "go9": O.OG_GO9}
O_INITQ = {"parent": O.OQ_PARENT, "zero": O.OQ_ZERO, "drop": O.OQ_DROP_PARENT}
G_INITQ = {"parent": capi.INITQ_PARENT, "zero": capi.INITQ_ZERO, "drop": capi.INITQ_DROP_PARENT}
EXACT_KEYS = ["game_moves", "game_rng_draws", "move_N", "move_W", "move_P", "move_root_N", "move_root_W",
              "move_action", "move_traversals", "move_player", "states", "outcomes"]
MATCH_KEYS = ["game_moves", "game_winner", "game_rng_draws", "move_N", "move_W", "move_P", "move_root_N", "move_root_W",
              "move_action", "move_traversals", "move_player"]
STEP_KEYS = ["game_moves", "move_N", "move_W", "move_P", "move_root_N", "move_root_W", "move_action", "move_traversals",
             "move_player"]


# ---------------------------------------------------------------------------------------------- evaluators
class SpikeNet:
    """Logits c[i] = -i: after masking, the lowest-indexed legal action takes almost all of the prior, so the search
    follows one line deep down the tree.  With `wide`, c[i] + clamp(x @ Wp / 8, -4, 4) with Wp in {-1, 0, 1}, so that a
    leaf reading another leaf's evaluator row changes the result.  The value is IntegerNet's value head: not zero, so
    that the sign of every backed-up term matters.  The spiked network scales it by `vscale` = 1/1024 instead of 1/64,
    small enough that the priors still lead the search deep on Othello; on Go even that keeps descents short, so the
    spiked Go networks answer 0.  Every partial sum is an integer times a power of two and the final
    add is one fp32 add, so numpy and torch (TF32 off) agree bit for bit; the logits stay within [-85, 4], so every
    legal exp() is a normal float even on Go 9x9's 82 actions."""

    def __init__(self, game, seed, wide, vscale=1.0 / 64):
        gi = O.game_info(game)
        planes = (2 * gi.history + 1) * gi.cells
        self.c = -np.arange(gi.actions, dtype=np.float32)
        self.wp = np.random.RandomState(seed).randint(-1, 2, size=(planes, gi.actions)).astype(np.float32) if wide else None
        self.wv = IntegerNet(2 * gi.history + 1, gi.cells, gi.actions, seed=seed).wv
        self.vscale = vscale

    def numpy(self, x):
        flat = np.asarray(x, np.float32).reshape(x.shape[0], -1)
        value = np.clip((flat @ self.wv) * np.float32(self.vscale), -1, 1) if self.vscale else np.zeros(len(flat), np.float32)
        if self.wp is None:
            return np.repeat(self.c[None], flat.shape[0], 0), value
        return self.c + np.clip((flat @ self.wp) * np.float32(0.125), -4, 4), value

    def torch_fn(self, dev):
        import torch
        torch.backends.cuda.matmul.allow_tf32 = False
        c = torch.from_numpy(self.c).to(dev)
        wp = None if self.wp is None else torch.from_numpy(self.wp).to(dev)
        wv, vscale = torch.from_numpy(self.wv).to(dev), self.vscale

        def fn(x):
            flat = x.reshape(x.shape[0], -1)
            value = torch.clamp((flat @ wv) * vscale, -1, 1) if vscale else torch.zeros(x.shape[0], device=x.device)
            if wp is None:
                return c.expand(x.shape[0], -1).clone(), value
            return c + torch.clamp((flat @ wp) * 0.125, -4, 4), value
        return fn


# ---------------------------------------------------------------------------------------------- configurations
# ev: "spike" (constant logits), "net" (input-dependent logits), "hash" (HashNet on the device).  Agent k of a match has
# its own network weights.
# Self-play: seed 3, first game 0, eps 0.25, alpha 0.3.
def cfg(game, sims, b, q, ngames, ev="spike", noise=1, sym=1, iq="parent", slots=None, u_weight=1.1, **engine):
    return dict(game=game, sims=sims, b=b, q=q, ngames=ngames, ev=ev, noise=noise, sym=sym, iq=iq, slots=slots or ngames,
                u_weight=u_weight, engine=engine)


DEEP = {
    "othello_plain": cfg("othello", 200, 8, 4, 3, noise=0, sym=0),
    "othello_noise": cfg("othello", 200, 8, 4, 3, sym=0),
    "othello_zero": cfg("othello", 300, 8, 4, 4, sym=0, iq="zero"),
    "othello_drop": cfg("othello", 300, 8, 4, 4, sym=0, iq="drop"),
    "othello_slots": cfg("othello", 200, 8, 4, 4, sym=0, slots=2),            # retained deep chains compacted, slots reused
    "othello_graph": cfg("othello", 200, 8, 4, 3, noise=0, sym=0, graph=True),
    "go": cfg("go", 300, 16, 8, 2),
    "go9": cfg("go9", 300, 16, 8, 1),
    # rounds_per_launch applies to the device evaluators only (an external network is called between launches).
    # HashNet with u_weight 0 picks by Q alone and also goes deep; 8 rounds a launch apply queued deep leaves in the
    # launch that queued them.  One slot for two games.
    "othello_hash_rounds": cfg("othello", 1000, 4, 2, 2, ev="hash", noise=0, sym=0, slots=1, u_weight=0.0,
                               rounds_per_launch=8),
}
OTHELLO_DEEP = [k for k in DEEP if k.startswith("othello")]

# (b, q): m = min(b, q) copies of each fresh root in its first batch.  (40, 64): the queue never fills.
WIDE_BQ = [(32, 32), (40, 33), (64, 48), (300, 255), (40, 64)]
WIDE = {}
for _b, _q in WIDE_BQ:
    for _g in ("othello", "go"):
        for _ev in ("hash", "net"):
            if (_b, _q) == (40, 64) and (_g, _ev) != ("othello", "hash"):
                continue
            WIDE[f"{_g}_{_ev}_{_b}_{_q}"] = cfg(_g, max(2 * _b, 96), _b, _q, 2 if _g == "othello" else 1, ev=_ev)
WIDE["othello_spike_deep_400_40_33"] = cfg("othello", 400, 40, 33, 3, sym=0)    # deep and wide at once

# Match play (Evaluate.cpp's constants: noise on, eps 0.25, alpha 0.1, uWeight 1.0): seed 7, first game 11.
def mcfg(game, sims, b, q, ngames, evs, iqs=("parent", "zero"), syms=(0, 0), pairs=None):
    return dict(game=game, sims=sims, b=b, q=q, ngames=ngames, evs=evs, iqs=iqs, syms=syms, pairs=pairs or ngames)


MATCH_DEEP = {
    "othello_spike": mcfg("othello", 200, 8, 4, 4, ("spike", "spike")),
    "othello_spike_wide": mcfg("othello", 300, 40, 33, 4, ("spike", "spike"), pairs=2),
}
MATCH_WIDE = {}
for _b, _q in WIDE_BQ[:4]:
    for _g in ("othello", "go"):
        for _ev in ("hash", "net"):
            MATCH_WIDE[f"{_g}_{_ev}_{_b}_{_q}"] = mcfg(_g, max(2 * _b, 96), _b, _q, 2, (_ev, _ev), syms=(1, 0))


# ---------------------------------------------------------------------------------------------- the oracle side
@functools.lru_cache(maxsize=None)
def spike_net(game, ev, side=0):
    vscale = 1.0 / 64 if ev == "net" else (1.0 / 1024 if game == "othello" else 0.0)
    return SpikeNet(GAME_IDS[game], 100 + 10 * GAME_IDS[game] + side, wide=ev == "net", vscale=vscale)


def oracle_selfplay(c, caller_moves=False):
    return _oracle_selfplay(tuple(sorted((k, v) for k, v in c.items() if k != "engine")), caller_moves)


@functools.lru_cache(maxsize=None)
def _oracle_selfplay(key, caller_moves):
    c = dict(key)
    game = GAME_IDS[c["game"]]
    ev = O.OE_HASHNET if c["ev"] == "hash" else O.OE_CALLBACK
    fn = None if c["ev"] == "hash" else spike_net(c["game"], c["ev"]).numpy
    return O.selfplay(game, ev, 3, 0, c["ngames"], c["sims"], c["b"], c["q"], 0.25, 0.3, add_noise=bool(c["noise"]),
                      use_sym=bool(c["sym"]), init_q=O_INITQ[c["iq"]], u_weight=c["u_weight"], eval_fn=fn,
                      caller_moves=caller_moves, max_moves_per_game=MAX_MOVES[c["game"]], search_stats=True)


def o_agent(c, k):
    ev = c["evs"][k]
    a = dict(use_sym=c["syms"][k], init_q=O_INITQ[c["iqs"][k]])
    if ev == "hash":
        return dict(a, evaluator=O.OE_HASHNET, hash_salt=k)
    return dict(a, evaluator=O.OE_CALLBACK, eval_fn=spike_net(c["game"], ev, k).numpy)


@functools.lru_cache(maxsize=None)
def _oracle_match(name, table):
    c = (MATCH_DEEP if table == "deep" else MATCH_WIDE)[name]
    game = GAME_IDS[c["game"]]
    ref = O.match(game, [o_agent(c, 0), o_agent(c, 1)], 7, 11, c["ngames"], c["sims"], c["b"], c["q"],
                  max_moves_per_game=MAX_MOVES[c["game"]], search_stats=True)
    ref["game_winner"] = ref["game_winner"].astype(np.int8)
    return ref


def deep_descents(st):
    return int(st["depth_hist"][DESCENT_MAX:].sum())


# ---------------------------------------------------------------------------------------------- CPU: the oracle counters
def test_oracle_counters_are_consistent():
    """The search-shape counters add up: one histogram entry per descent, every deep descent in exactly one ending, no
    queue longer than max_queue, and the first-32 duplicates a subset of all duplicates (self-play and match play)."""
    ref = oracle_selfplay(DEEP["othello_noise"])
    st = ref["stats"]
    assert st["depth_hist"].sum() == st["total_traversals"] == ref["move_traversals"].sum()
    assert st["leaves_terminal"] + st["leaves_gray"] + st["leaves_empty"] == st["total_traversals"]
    assert st["deep_terminal"] + st["deep_gray"] + st["deep_queued"] == deep_descents(st)
    assert st["select_depth_max"] == np.flatnonzero(st["depth_hist"]).max()
    assert st["select_depth_sum"] == (np.arange(O.DEPTH_BINS) * st["depth_hist"]).sum()
    assert st["queue_max"] <= 4 and 0 < st["dup_first32"] == st["dup_total"]
    m = _oracle_match("othello_spike", "deep")["stats"]
    assert m["depth_hist"].sum() == m["total_traversals"] == _oracle_match("othello_spike", "deep")["move_traversals"].sum()
    assert m["deep_terminal"] + m["deep_gray"] + m["deep_queued"] == deep_descents(m)
    assert m["leaves_terminal"] + m["leaves_gray"] + m["leaves_empty"] == m["total_traversals"]


@pytest.mark.parametrize("name", list(DEEP) + ["othello_spike_deep_400_40_33"])
def test_deep_configuration_goes_deeper_than_the_recorded_path(name):
    st = oracle_selfplay(DEEP.get(name) or WIDE[name])["stats"]
    assert st["depth_hist"][DESCENT_MAX + 1:].sum() > 0, st["select_depth_max"]
    assert deep_descents(st) > 0


@pytest.mark.parametrize("name", list(MATCH_DEEP))
def test_deep_match_configuration_goes_deeper_than_the_recorded_path(name):
    st = _oracle_match(name, "deep")["stats"]
    assert st["depth_hist"][DESCENT_MAX + 1:].sum() > 0 and st["deep_queued"] > 0


def test_othello_deep_configurations_cover_every_ending_and_the_boundary():
    """Together the Othello deep runs back up terminal, gray and queued leaves below depth 32 by parent links, and
    reach depth 31 (the last descent that fills all 32 lanes of backup_path), 32 (the first that falls back) and 33."""
    tot = {k: 0 for k in ("deep_terminal", "deep_gray", "deep_queued")}
    hist = np.zeros(O.DEPTH_BINS, np.int64)
    for name in OTHELLO_DEEP + ["othello_spike_deep_400_40_33"]:
        st = oracle_selfplay(DEEP.get(name) or WIDE[name])["stats"]
        for k in tot:
            tot[k] += st[k]
        hist += st["depth_hist"]
    assert all(v > 0 for v in tot.values()), tot
    assert (hist[DESCENT_MAX - 1:DESCENT_MAX + 2] > 0).all(), hist[DESCENT_MAX - 1:DESCENT_MAX + 2]


def test_stepwise_deep_configuration_goes_deep():
    st = oracle_selfplay(DEEP["othello_noise"], caller_moves=True)["stats"]
    assert st["depth_hist"][DESCENT_MAX + 1:].sum() > 0


@pytest.mark.parametrize("name", list(WIDE))
def test_wide_configuration_queues_past_the_compared_entries(name):
    c = WIDE[name]
    st = oracle_selfplay(c)["stats"]
    m = min(c["b"], c["q"])
    assert st["queue_max"] == m
    if m > 32:
        assert st["dup_total"] > st["dup_first32"]
    else:
        assert st["dup_total"] == st["dup_first32"] > 0


@pytest.mark.parametrize("name", list(MATCH_WIDE))
def test_wide_match_configuration_queues_past_the_compared_entries(name):
    c = MATCH_WIDE[name]
    st = _oracle_match(name, "wide")["stats"]
    assert st["queue_max"] == min(c["b"], c["q"])
    assert (st["dup_total"] > st["dup_first32"]) == (min(c["b"], c["q"]) > 32)


def test_max_queue_above_255_is_refused():
    """Queue offsets and path lengths are stored in bytes: 255 leaves per tree and batch is the limit (checked before
    any device work, so this runs without a GPU)."""
    import ctypes as C
    lib = capi.load()
    h = C.c_void_p()
    conf = capi.default_config(capi.GAME_OTHELLO)
    conf.max_batch, conf.max_queue = 300, 256
    assert lib.sprl_create(C.byref(conf), C.byref(h)) == capi.SPRL_E_INVALID and not h
    assert b"255" in lib.sprl_last_error()


# ---------------------------------------------------------------------------------------------- GPU
def check_stats(st, rs):
    """Engine counters against the oracle's; a duplicate is counted among the first 32 entries of a batch only."""
    assert st["sims"] == rs["total_traversals"] and st["evals"] == rs["total_evals"]
    assert st["depth_sum"] == int(rs["select_depth_sum"]) and st["legal_sum"] == int(rs["select_legal_sum"])
    assert st["leaves_terminal"] == rs["leaves_terminal"] and st["leaves_gray"] == rs["leaves_gray"]
    assert st["leaves_duplicate"] == rs["dup_first32"]


def engine(c, evaluator, **kw):
    from sprl_b200 import selfplay as SP
    return SP.Engine(GPU_GAMES[c["game"]], evaluator,
                     seed=3, sims=c["sims"], max_batch=c["b"], max_queue=c["q"], dir_eps=0.25, dir_alpha=0.3,
                     add_noise=c["noise"], use_sym=c["sym"], init_q=G_INITQ[c["iq"]], u_weight=c["u_weight"],
                     num_slots=c["slots"], max_games=c["ngames"], record_stats=1, **kw)


GPU_GAMES = {"othello": capi.GAME_OTHELLO, "go": capi.GAME_GO7, "go9": capi.GAME_GO9}


def run_selfplay(c):
    import torch
    graph = c["engine"].get("graph", False)
    extra = {k: v for k, v in c["engine"].items() if k != "graph"}
    hash_ev = c["ev"] == "hash"
    with engine(c, capi.EVAL_HASHNET if hash_ev else capi.EVAL_EXTERNAL, **extra) as eng:
        if not hash_ev:
            eng.attach_network(spike_net(c["game"], c["ev"]).torch_fn(torch.device("cuda", 0)), use_cuda_graph=graph)
        states, dists, outcomes = eng.run_iteration(c["ngames"])
        got = eng.move_stats(c["ngames"])
        pools, damaged = eng.check_guards()
        assert pools > 20 and damaged == 0
        got.update(states=states, distributions=dists, outcomes=outcomes, stats=eng.stats())
    return got


def compare_selfplay(ref, got):
    G.assert_trace_equal(ref, got, EXACT_KEYS)
    G.assert_trace_equal(ref, got, ["distributions"], exact=False)
    check_stats(got["stats"], ref["stats"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(DEEP))
def test_deep_selfplay_vs_oracle(name):
    c = DEEP[name]
    compare_selfplay(oracle_selfplay(c), run_selfplay(c))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(WIDE))
def test_wide_queue_selfplay_vs_oracle(name):
    c = WIDE[name]
    compare_selfplay(oracle_selfplay(c), run_selfplay(c))


def run_match(c, ngames=None):
    import torch
    from sprl_b200 import selfplay as SP
    ngames = ngames or c["ngames"]
    external = any(ev != "hash" for ev in c["evs"])
    g_agents = [dict(evaluator=capi.EVAL_HASHNET if ev == "hash" else capi.EVAL_EXTERNAL, hash_salt=k, use_sym=c["syms"][k],
                     init_q=G_INITQ[c["iqs"][k]]) for k, ev in enumerate(c["evs"])]
    with SP.Engine(GPU_GAMES[c["game"]], capi.EVAL_EXTERNAL if external else capi.EVAL_UNIFORM, seed=7, sims=c["sims"],
                   max_batch=c["b"], max_queue=c["q"], dir_eps=0.25, dir_alpha=0.1, u_weight=1.0, add_noise=1,
                   num_slots=2 * c["pairs"], max_games=ngames, record_stats=1) as eng:
        if external:
            dev = torch.device("cuda", 0)
            eng.attach_match_evaluators([None if ev == "hash" else spike_net(c["game"], ev, k).torch_fn(dev)
                                         for k, ev in enumerate(c["evs"])], use_cuda_graph=False)
        got = eng.run_match(g_agents, ngames, first_game=11)
        got.update(eng.move_stats(ngames))
        pools, damaged = eng.check_guards()
        assert pools > 20 and damaged == 0
        got["stats"] = eng.stats()
    return got


def compare_match(ref, got):
    G.assert_trace_equal(ref, got, MATCH_KEYS)
    assert got["wins"] == ref["wins"] and got["draws"] == ref["draws"]
    check_stats(got["stats"], ref["stats"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MATCH_DEEP))
def test_deep_match_vs_oracle(name):
    compare_match(_oracle_match(name, "deep"), run_match(MATCH_DEEP[name]))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MATCH_WIDE))
def test_wide_queue_match_vs_oracle(name):
    compare_match(_oracle_match(name, "wide"), run_match(MATCH_WIDE[name]))


@pytest.mark.gpu
def test_deep_stepwise_trees_vs_oracle():
    """begin_trees / search / advance with the spiked network, a caller playing the first most-visited action."""
    import torch
    from test_gpu_parity import walk_trees
    c = DEEP["othello_noise"]
    ref = oracle_selfplay(c, caller_moves=True)
    with engine(c, capi.EVAL_EXTERNAL) as eng:
        eng.attach_network(spike_net(c["game"], c["ev"]).torch_fn(torch.device("cuda", 0)), use_cuda_graph=False)
        got = walk_trees(eng, c["ngames"], c["sims"], 0)
        assert eng.check_guards()[1] == 0
    G.assert_trace_equal(ref, got, STEP_KEYS)


def _device_rows(eng):
    """The engine's device row counter (uint32[2]: rows of the last search launch, agent 0 / agent 1)."""
    import torch

    class _View:
        def __init__(self, ptr):
            self.__cuda_array_interface__ = dict(shape=(2,), typestr="<i4", data=(ptr, False), version=3, strides=None,
                                                 stream=None)
    torch.cuda.synchronize()
    return torch.as_tensor(_View(eng._nn["rows"]), device=torch.device("cuda", 0)).cpu().numpy().copy()


@pytest.mark.gpu
@pytest.mark.parametrize("game", ["othello", "go"])
@pytest.mark.parametrize("b,q", WIDE_BQ + [(8, 4)])
def test_first_launch_rows_of_fresh_trees(game, b, q):
    """A fresh root is queued m = min(b, q) times in its tree's first batch: the copies among the first 32 entries share
    one evaluator row, every later copy has its own, so the launch hands out 1 + max(0, m - 32) rows per tree -- in
    self-play, and in match play per side (only the side to move searches; agent 1's rows start at q_half)."""
    import torch
    from sprl_b200 import selfplay as SP
    m = min(b, q)
    per_tree = 1 + max(0, m - 32)
    ngames = 3
    dev = torch.device("cuda", 0)
    net = spike_net(game, "net")
    with SP.Engine(GPU_GAMES[game], capi.EVAL_EXTERNAL, seed=3, sims=2 * b, max_batch=b, max_queue=q, num_slots=ngames,
                   max_games=ngames) as eng:
        eng.attach_network(net.torch_fn(dev), use_cuda_graph=False)
        eng.set_stream(torch.cuda.current_stream(dev).cuda_stream)
        eng.begin_iteration(0, ngames)
        eng.round()
        rows = _device_rows(eng)
        assert eng.stats()["leaves_duplicate"] == ngames * (min(m, 32) - 1)
        assert eng.check_guards()[1] == 0
    assert rows[0] == ngames * per_tree and rows[1] == 0, rows
    # match play: game t's side to move first is agent t % 2
    agents = (capi.AgentConfig * 2)(*[capi.AgentConfig(evaluator=capi.EVAL_EXTERNAL, use_sym=1, init_q=capi.INITQ_PARENT,
                                                       hash_salt=0) for _ in range(2)])
    first = 4
    with SP.Engine(GPU_GAMES[game], capi.EVAL_EXTERNAL, seed=3, sims=2 * b, max_batch=b, max_queue=q, num_slots=2 * ngames,
                   max_games=ngames, u_weight=1.0, dir_alpha=0.1) as eng:
        eng.attach_match_evaluators([net.torch_fn(dev), net.torch_fn(dev)], use_cuda_graph=False)
        eng.set_stream(torch.cuda.current_stream(dev).cuda_stream)
        capi.check(eng.lib.sprl_match_begin(eng.handle, agents, first, ngames))
        eng.round()
        rows = _device_rows(eng)
        assert eng.check_guards()[1] == 0
    odd = sum((first + g) % 2 for g in range(ngames))
    assert rows[0] == (ngames - odd) * per_tree and rows[1] == odd * per_tree, rows
