"""Self-play, match play and step-wise trees through the library's evaluator network (EvalNet, csrc/evalnet.cu), bit for
bit against the CPU oracle.

bench.py, the Python worker and the C++ GridNetwork run their network through EvalNet: the engine writes leaf planes,
calls sprl_evalnet_forward_counted with its row count on the device (agent 1 of a match: the second counter, its own
half of the batch), usually replayed in a CUDA graph, and reads logits / values back in place.  Here the oracle's
callback evaluator is a second EvalNet of the same module on the same GPU, fed the planes the oracle writes.  A board's
outputs are the same bits wherever it sits in the batch and whatever the batch size (checked first, for every evaluator
used below), so any difference between the two traces is a fault in how the engine hands leaves to the evaluator and
reads its outputs back -- a leaf reading another leaf's row, a stale row, one agent's half of a match batch counted or
read as the other's, wrong planes -- not rounding.  Unlike the integer-valued test networks, a real network gives
logits and values that are arbitrary floats, so det_expf and the order of the backup's sums see general arguments.

The oracle runs first, then the engine: the engine's evaluator is another instance, whose captured graph holds buffers
sized for the engine's batch.  The CPU tests drive the oracle with each configuration's fp32 CPU forward (trajectories
differ from the GPU's only in rounding) and check that the configuration reaches what it is here for."""
import functools

import numpy as np
import pytest
import torch

import golden_util as G
import oracle_py as O
from sprl_b200 import capi
from sprl_b200.evalnet import EvalNet
from sprl_b200.network import BasicGridNetwork, make_network
from test_evalnet import randomized
from test_gpu_parity import MATCH_KEYS, STEP_KEYS, compare_selfplay, walk_trees

AUTO, STREAMING = capi.EVALNET_PATH_AUTO, capi.EVALNET_PATH_STREAMING
FP32, FP16 = capi.EVALNET_PRECISION_FP32_SPLIT, capi.EVALNET_PRECISION_FP16
# game: (engine id, oracle id, rows, cols, oracle capacity in moves per game)
GAMES = {"othello": (capi.GAME_OTHELLO, O.OG_OTHELLO, 8, 8, 130), "c4": (capi.GAME_C4, O.OG_C4, 6, 7, 50),
         "go7": (capi.GAME_GO7, O.OG_GO7, 7, 7, 200), "go9": (capi.GAME_GO9, O.OG_GO9, 9, 9, 330)}
INITQ = {"parent": (capi.INITQ_PARENT, O.OQ_PARENT), "zero": (capi.INITQ_ZERO, O.OQ_ZERO),
         "drop": (capi.INITQ_DROP_PARENT, O.OQ_DROP_PARENT)}
SHARP_MIN, SHARP_MAX = -80.0, 88.0       # the sharp head's logits reach below SHARP_MIN and stay under SHARP_MAX


# ---------------------------------------------------------------------------------------------- networks
def sharpen(net):
    """policy_fc times 4 plus a bias ramp of -1.3 i: logits from about -85 to 2, so exp() of a prior runs over most of the
    range where it is a normal float (expf overflows above 88.7)."""
    with torch.no_grad():
        net.policy_fc.weight.mul_(4.0)
        net.policy_fc.bias.mul_(4.0).add_(-1.3 * torch.arange(net.policy_fc.out_features, dtype=torch.float32))
    return net


def _wide_othello():
    torch.manual_seed(12)
    return randomized(BasicGridNetwork(8, 8, 65, 1, 2, 128).eval(), 112)


# name: (game, builder).  Every network has randomized BatchNorm statistics (test_evalnet.randomized).
NETWORKS = {
    "othello": ("othello", lambda: randomized(make_network("othello", 0), 100)),
    "othello_b": ("othello", lambda: randomized(make_network("othello", 1), 101)),
    "wide": ("othello", _wide_othello),                                                  # 2x128: the k_evalnet<., 128> tower
    "sharp": ("othello", lambda: sharpen(randomized(make_network("othello", 6), 6))),
    "c4": ("c4", lambda: randomized(make_network("c4", 3), 103)),
    "go7": ("go7", lambda: randomized(make_network("go7", 4), 104)),
    "go9": ("go9", lambda: randomized(make_network("go9", 5), 105)),
    "go9_b": ("go9", lambda: randomized(make_network("go9", 7), 107)),
}


@functools.lru_cache(maxsize=None)
def network(name):
    return NETWORKS[name][1]()


# evaluator setting: (network, path, precision)
SETTINGS = {
    "othello": ("othello", AUTO, FP32),
    "othello_b": ("othello_b", AUTO, FP32),
    "streaming": ("othello", STREAMING, FP32),
    "fp16": ("othello", AUTO, FP16),
    "wide": ("wide", AUTO, FP32),
    "sharp": ("sharp", AUTO, FP32),
    "c4": ("c4", AUTO, FP32),
    "go7": ("go7", AUTO, FP32),
    "go9": ("go9", AUTO, FP32),
    "go9_b": ("go9_b", AUTO, FP32),
}


def board(setting):
    _, _, rows, cols, _ = GAMES[NETWORKS[SETTINGS[setting][0]][0]]
    return rows, cols


def make_evalnet(module, rows, cols, path=AUTO, precision=FP32):
    ev = EvalNet(module, device=0, rows=rows, cols=cols)
    if path != AUTO:
        ev.set_path(path)
    if precision != FP32:
        ev.set_precision(precision)
    return ev


def setting_evalnet(setting, module=None):
    name, path, precision = SETTINGS[setting]
    return make_evalnet(module if module is not None else network(name), *board(setting), path, precision)


# ---------------------------------------------------------------------------------------------- the oracle's evaluator
class OracleEvaluator:
    """The oracle's callback evaluator: numpy planes [n, planes, rows, cols] -> (logits [n, A], values [n]) through
    `forward`.  Records the calls, the rows and the range of the logits it returned."""

    def __init__(self, forward, evalnet=None):
        self.forward, self.evalnet = forward, evalnet
        self.calls = self.rows = 0
        self.lo, self.hi = np.inf, -np.inf

    def __call__(self, x):
        logits, value = self.forward(np.ascontiguousarray(x, np.float32))
        self.calls += 1
        self.rows += x.shape[0]
        self.lo, self.hi = min(self.lo, float(logits.min())), max(self.hi, float(logits.max()))
        return logits, value

    def close(self):
        """status() of the evaluator (fails on an out-of-range activation or a pipeline time-out), then frees it."""
        if self.evalnet is not None:
            self.evalnet.status()
            self.evalnet.close()


def gpu_evaluator(module, rows, cols, path=AUTO, precision=FP32):
    """A separate EvalNet of `module` for the oracle: planes to the GPU, one forward of the oracle's batch, back."""
    ev = make_evalnet(module, rows, cols, path, precision)

    def forward(x):
        logits, value = ev(torch.from_numpy(x).cuda())
        return logits.cpu().numpy(), value.cpu().numpy().reshape(-1)
    return OracleEvaluator(forward, ev)


def cpu_evaluator(module):
    """The fp32 CPU forward of the same module (the CPU tests)."""
    def forward(x):
        with torch.no_grad():
            logits, value = module(torch.from_numpy(x))
        return logits.numpy(), value.numpy().reshape(-1)
    return OracleEvaluator(forward)


def oracle_evaluator(setting, on_gpu):
    name, path, precision = SETTINGS[setting]
    return gpu_evaluator(network(name), *board(setting), path, precision) if on_gpu else cpu_evaluator(network(name))


# ---------------------------------------------------------------------------------------------- configurations
def cfg(game, ev, sims, b, q, alpha, ngames, compare=None, slots=None, first=0, stride=1, graph=True, noise=1, sym=1,
        iq="parent", fix_mask=0, attach_as=None):
    """Self-play (seed 21, eps 0.25).  compare: the first games compared with the oracle (all by default); stride: game
    ids first, first + stride, ...; attach_as: the network the engine's evaluator is built from before update() loads
    the setting's network into it, after attach and before the graph is captured (bench.py's broadcast_weights)."""
    return dict(game=game, ev=ev, sims=sims, b=b, q=q, alpha=alpha, ngames=ngames, compare=compare or ngames,
                slots=slots or ngames, first=first, stride=stride, graph=graph, noise=noise, sym=sym, iq=iq,
                fix_mask=fix_mask, attach_as=attach_as)


SELFPLAY = {
    # bench.py's headline configuration (400 sims, 8 / 4, D4, Dirichlet 0.25 / 0.3, graph): 256 concurrent games, the
    # first 3 compared -- a game must not depend on its neighbours
    "headline": cfg("othello", "othello", 400, 8, 4, 0.3, 256, compare=3),
    # bench.py's steady state: game stride 2 from an odd first game, fewer slots than games, update() before capture
    "steady": cfg("othello", "othello", 200, 8, 4, 0.3, 5, slots=2, first=1, stride=2, attach_as="othello_b"),
    "nograph": cfg("othello", "othello", 160, 8, 4, 0.3, 3, graph=False),
    "streaming": cfg("othello", "streaming", 160, 8, 4, 0.3, 3),
    "fp16": cfg("othello", "fp16", 160, 8, 4, 0.3, 3),
    "wide": cfg("othello", "wide", 160, 8, 4, 0.3, 3),
    "c4": cfg("c4", "c4", 200, 8, 4, 0.5, 4),
    "go7": cfg("go7", "go7", 64, 16, 8, 0.2, 2),
    # Go 9x9 (two-word bitboards; roots with more than 32 legal actions): bench.py's batch 16 / queue 8 / alpha 0.2
    "go9": cfg("go9", "go9", 48, 16, 8, 0.2, 1),
    "zero": cfg("othello", "othello", 120, 8, 4, 0.3, 2, iq="zero"),
    "drop": cfg("othello", "othello", 120, 8, 4, 0.3, 2, iq="drop"),
    "fix_mask": cfg("othello", "othello", 120, 8, 4, 0.3, 2, noise=0, fix_mask=1),
    "plain": cfg("othello", "othello", 120, 8, 4, 0.3, 2, noise=0, sym=0),
    "sharp": cfg("othello", "sharp", 200, 8, 4, 0.3, 2),
}
SEED = 21


def game_ids(c):
    return [c["first"] + k * c["stride"] for k in range(c["compare"])]


def oracle_selfplay(c, ev, first_game, ngames, caller_moves=False):
    _, og, _, _, cap = GAMES[c["game"]]
    return O.selfplay(og, O.OE_CALLBACK, SEED, first_game, ngames, c["sims"], c["b"], c["q"], 0.25, c["alpha"],
                      add_noise=bool(c["noise"]), use_sym=bool(c["sym"]), init_q=INITQ[c["iq"]][1], eval_fn=ev,
                      max_moves_per_game=cap, fix_symmetry_mask=bool(c["fix_mask"]), caller_moves=caller_moves)


STAT_KEYS = (("sims", "total_traversals"), ("evals", "total_evals"), ("leaves_terminal", "leaves_terminal"),
             ("leaves_gray", "leaves_gray"), ("depth_sum", "select_depth_sum"), ("legal_sum", "select_legal_sum"))


def oracle_games(c, ev):
    """The oracle's games of the configuration's compared ids, one run per id when the ids are not consecutive; traces
    concatenated in id order, statistics summed."""
    ids = game_ids(c)
    if c["stride"] == 1:
        return oracle_selfplay(c, ev, ids[0], len(ids))
    runs = [oracle_selfplay(c, ev, g, 1) for g in ids]
    ref = {k: np.concatenate([r[k] for r in runs]) for k in runs[0] if k != "stats"}
    ref["stats"] = {o: sum(r["stats"][o] for r in runs) for _, o in STAT_KEYS}
    return ref


def first_games(got, k, samples_per_move):
    """The trace of the first k games of an engine run."""
    m = int(got["game_moves"][:k].sum())
    out = {key: v[:k] for key, v in got.items() if key.startswith("game_")}
    out.update({key: v[:m] for key, v in got.items() if key.startswith("move_")})
    out.update({key: got[key][:m * samples_per_move] for key in ("states", "distributions", "outcomes")})
    return out


def check_stats(st, rs):
    for mine, theirs in STAT_KEYS:
        assert st[mine] == int(rs[theirs]), (mine, st[mine], rs[theirs])


def selfplay_engine(c, num_slots, max_games):
    from sprl_b200 import selfplay as SP
    return SP.Engine(GAMES[c["game"]][0], capi.EVAL_EXTERNAL, seed=SEED, sims=c["sims"], max_batch=c["b"], max_queue=c["q"],
                     dir_eps=0.25, dir_alpha=c["alpha"], add_noise=c["noise"], use_sym=c["sym"], init_q=INITQ[c["iq"]][0],
                     fix_symmetry_mask=c["fix_mask"], num_slots=num_slots, max_games=max_games, record_stats=1)


def finish(eng, ngames, samples):
    states, dists, outcomes = samples
    got = eng.move_stats(ngames)
    pools, damaged = eng.check_guards()             # no kernel wrote outside its pools
    assert pools > 20 and damaged == 0
    got.update(states=states, distributions=dists, outcomes=outcomes, stats=eng.stats())
    return got


def run_selfplay(c):
    """The engine's run of configuration c through an attached EvalNet of its setting."""
    ev = setting_evalnet(c["ev"], network(c["attach_as"]) if c["attach_as"] else None)
    with selfplay_engine(c, c["slots"], c["ngames"]) as eng:
        if c["stride"] != 1:
            eng.set_game_stride(c["stride"])
        eng.attach_evalnet(ev, use_cuda_graph=c["graph"])
        if c["attach_as"]:
            ev.update(network(SETTINGS[c["ev"]][0]))
        got = finish(eng, c["ngames"], eng.run_iteration(c["ngames"], first_game=c["first"]))
    ev.status()
    ev.close()
    return got


# match play (Evaluate.cpp's constants: noise on, eps 0.25, alpha 0.1, uWeight 1.0): seed 7, first game 11 (odd: agent 1
# opens game 0).  An agent is an evaluator setting, "hash" or "uniform".
def mcfg(game, evs, sims, b, q, ngames, pairs, graph=True, iqs=("parent", "zero"), syms=(1, 1)):
    return dict(game=game, evs=evs, sims=sims, b=b, q=q, ngames=ngames, pairs=pairs, graph=graph, iqs=iqs, syms=syms)


MATCH = {
    "nets_graph": mcfg("othello", ("othello", "othello_b"), 100, 8, 4, 6, 2),
    "nets_no_graph": mcfg("othello", ("othello", "othello_b"), 100, 8, 4, 6, 2, graph=False, syms=(1, 0)),
    "hash_vs_net": mcfg("othello", ("hash", "othello"), 100, 8, 4, 4, 2),
    "c4_net_vs_uniform": mcfg("c4", ("c4", "uniform"), 128, 8, 4, 6, 3),
    "go9": mcfg("go9", ("go9", "go9_b"), 32, 16, 8, 2, 1),
}
DEVICE_EVALS = {"hash": (capi.EVAL_HASHNET, O.OE_HASHNET), "uniform": (capi.EVAL_UNIFORM, O.OE_UNIFORM)}


def oracle_match(c, evaluators):
    agents = []
    for k, ev in enumerate(c["evs"]):
        a = dict(use_sym=c["syms"][k], init_q=INITQ[c["iqs"][k]][1])
        agents.append(dict(a, evaluator=DEVICE_EVALS[ev][1]) if ev in DEVICE_EVALS else
                      dict(a, evaluator=O.OE_CALLBACK, eval_fn=evaluators[k]))
    _, og, _, _, cap = GAMES[c["game"]]
    ref = O.match(og, agents, 7, 11, c["ngames"], c["sims"], c["b"], c["q"], max_moves_per_game=cap, search_stats=True)
    ref["game_winner"] = ref["game_winner"].astype(np.int8)
    return ref


def run_match(c):
    from sprl_b200 import selfplay as SP
    evs = [None if ev in DEVICE_EVALS else setting_evalnet(ev) for ev in c["evs"]]
    agents = [dict(evaluator=DEVICE_EVALS[ev][0] if ev in DEVICE_EVALS else capi.EVAL_EXTERNAL, hash_salt=0,
                   use_sym=c["syms"][k], init_q=INITQ[c["iqs"][k]][0]) for k, ev in enumerate(c["evs"])]
    with SP.Engine(GAMES[c["game"]][0], capi.EVAL_EXTERNAL, seed=7, sims=c["sims"], max_batch=c["b"], max_queue=c["q"],
                   dir_eps=0.25, dir_alpha=0.1, u_weight=1.0, add_noise=1, num_slots=2 * c["pairs"], max_games=c["ngames"],
                   record_stats=1) as eng:
        eng.attach_match_evaluators(evs, use_cuda_graph=c["graph"])
        got = eng.run_match(agents, c["ngames"], first_game=11)
        got.update(eng.move_stats(c["ngames"]))
        pools, damaged = eng.check_guards()
        assert pools > 20 and damaged == 0
        got["stats"] = eng.stats()
    for ev in evs:
        if ev is not None:
            ev.status()
            ev.close()
    return got


# step-wise trees: the caller plays the first most-visited action; fewer trees than slots
STEPWISE = cfg("othello", "othello", 64, 8, 4, 0.3, 3, slots=5, first=200)


def engine_batches(setting):
    """(evaluator batch, max_queue) of every engine that runs the setting in this module."""
    out = {(c["slots"] * c["q"], c["q"]) for c in list(SELFPLAY.values()) + [STEPWISE] if c["ev"] == setting}
    out |= {(2 * c["pairs"] * c["q"], c["q"]) for c in MATCH.values() if setting in c["evs"]}
    return sorted(out)


# ---------------------------------------------------------------------------------------------- CPU: what the configurations reach
@functools.lru_cache(maxsize=None)
def cpu_oracle(name):
    c = SELFPLAY[name]
    ev = oracle_evaluator(c["ev"], on_gpu=False)
    return oracle_games(c, ev), ev


def test_every_setting_is_used():
    for setting in SETTINGS:
        assert engine_batches(setting), setting


def test_go9_roots_have_more_than_32_legal_actions():
    """Go 9x9 roots with more than 32 legal actions take the n > 32 branch of evaluate_leaf, here with real priors."""
    ref, ev = cpu_oracle("go9")
    legal = (ref["move_P"] > 0).sum(1)
    assert (legal > 32).sum() >= 10, legal
    assert ev.calls > 0


def test_sharp_head_spans_the_range_of_expf():
    """The sharp head's logits reach below -80 and stay under 88: det_expf sees most of the range where its result is a
    normal float, and never overflows."""
    _, ev = cpu_oracle("sharp")
    assert ev.lo < SHARP_MIN and ev.hi < SHARP_MAX, (ev.lo, ev.hi)


def test_steady_state_reuses_every_slot():
    """In the steady-state configuration every slot plays several games: a slot starts the next game id when its game
    ends (a move takes the same number of search rounds in every game, so game lengths in moves order the ends)."""
    c = SELFPLAY["steady"]
    ref, _ = cpu_oracle("steady")
    moves = ref["game_moves"]
    assert len(moves) == c["ngames"] > c["slots"]
    free_at, played = [0] * c["slots"], [0] * c["slots"]
    for m in moves:
        s = int(np.argmin(free_at))
        free_at[s] += int(m)
        played[s] += 1
    assert min(played) >= 2, played


# ---------------------------------------------------------------------------------------------- GPU: the premise
def _row_independence(ev, planes, rows, cols, batch, max_queue, seed):
    g = torch.Generator().manual_seed(seed)
    big = max(batch, 1501)
    x = (torch.rand(big, planes, rows, cols, generator=g) > 0.5).float().cuda()
    want_l, want_v = ev(x)
    # one forward at the engine's batch size
    l, v = ev(x[:batch])
    assert torch.equal(l, want_l[:batch]) and torch.equal(v, want_v[:batch])
    # the oracle's batches: 1 .. max_queue boards from anywhere in the batch
    for n in range(1, max_queue + 1):
        idx = torch.randperm(big, generator=g)[:n].cuda()
        l, v = ev(x[idx])
        assert torch.equal(l, want_l[idx]) and torch.equal(v, want_v[idx]), n
    # a permutation of the large batch
    perm = torch.randperm(big, generator=g).cuda()
    l, v = ev(x[perm])
    assert torch.equal(l, want_l[perm]) and torch.equal(v, want_v[perm])
    # the engine's call: the counted forward over its batch buffer, the row count on the device
    logits = torch.empty(batch, want_l.shape[1], device="cuda")
    value = torch.empty(batch, device="cuda")
    d_rows = torch.zeros(1, dtype=torch.int32, device="cuda")
    for count in sorted({1, max_queue, batch // 2 + 1, batch}):
        d_rows.fill_(count)
        logits.fill_(float("nan"))
        value.fill_(float("nan"))
        ev.forward_ptr(x.data_ptr(), batch, logits.data_ptr(), value.data_ptr(), torch.cuda.current_stream().cuda_stream,
                       d_rows=d_rows.data_ptr())
        torch.cuda.synchronize()
        assert torch.equal(logits[:count], want_l[:count]) and torch.equal(value[:count], want_v[:count].reshape(-1)), count
        assert torch.isnan(logits[count:]).all() and torch.isnan(value[count:]).all(), count
    ev.status()


@pytest.mark.gpu
@pytest.mark.parametrize("setting", list(SETTINGS))
def test_evaluator_outputs_do_not_depend_on_the_batch(setting):
    """Every evaluator setting below: a board's outputs from batches of 1 .. max_queue rows (the oracle's calls), from a
    permuted large batch and from the counted forward (the engine's call) are the bits of one forward at the engine's batch
    size.  The fp16 opt-in mode holds the same property, for every network that runs on the resident kernel."""
    name, path, precision = SETTINGS[setting]
    rows, cols = board(setting)
    planes = network(name).conv.in_channels
    ev = setting_evalnet(setting)
    modes = [precision]
    if precision == FP32 and path == AUTO and ev.phases > 0:
        modes.append(FP16)
    for mode in modes:
        ev.set_precision(mode)
        for k, (batch, q) in enumerate(engine_batches(setting)):
            _row_independence(ev, planes, rows, cols, batch, q, seed=31 * k + mode)
    ev.close()


# ---------------------------------------------------------------------------------------------- GPU: self-play
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SELFPLAY))
def test_selfplay_through_evalnet_vs_oracle(name):
    c = SELFPLAY[name]
    ev = oracle_evaluator(c["ev"], on_gpu=True)
    ref = oracle_games(c, ev)
    ev.close()
    assert ev.calls > 0
    if c["ev"] == "sharp":
        assert ev.lo < SHARP_MIN and ev.hi < SHARP_MAX, (ev.lo, ev.hi)
    got = run_selfplay(c)
    if c["compare"] < c["ngames"]:
        got = dict(first_games(got, c["compare"], 8 if c["sym"] else 1), stats=None)
    compare_selfplay(ref, got)
    if got["stats"] is not None:
        check_stats(got["stats"], ref["stats"])


@pytest.mark.gpu
def test_selfplay_after_update_vs_oracle():
    """Network A for one iteration (graph captured), then update(B): the next iteration is the oracle's with B."""
    c = cfg("othello", "othello_b", 120, 8, 4, 0.3, 3, slots=2, first=40)
    ev = oracle_evaluator("othello_b", on_gpu=True)
    ref = oracle_games(c, ev)
    ev.close()
    mine = setting_evalnet("othello")
    with selfplay_engine(c, c["slots"], c["ngames"]) as eng:
        eng.attach_evalnet(mine, use_cuda_graph=True)
        eng.run_iteration(c["ngames"], first_game=0)
        mine.update(network("othello_b"))
        eng.reset_stats()
        got = finish(eng, c["ngames"], eng.run_iteration(c["ngames"], first_game=c["first"]))
    mine.status()
    mine.close()
    compare_selfplay(ref, got)
    check_stats(got["stats"], ref["stats"])


# ---------------------------------------------------------------------------------------------- GPU: match play
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MATCH))
def test_match_through_evalnet_vs_oracle(name):
    c = MATCH[name]
    evs = [None if ev in DEVICE_EVALS else oracle_evaluator(ev, on_gpu=True) for ev in c["evs"]]
    ref = oracle_match(c, evs)
    for ev in evs:
        if ev is not None:
            ev.close()
            assert ev.calls > 0
    got = run_match(c)
    G.assert_trace_equal(ref, got, MATCH_KEYS)
    assert got["wins"] == ref["wins"] and got["draws"] == ref["draws"]
    check_stats(got["stats"], ref["stats"])


# ---------------------------------------------------------------------------------------------- GPU: step-wise trees
@pytest.mark.gpu
def test_stepwise_trees_through_evalnet_vs_oracle():
    c = STEPWISE
    ev = oracle_evaluator(c["ev"], on_gpu=True)
    ref = oracle_selfplay(c, ev, c["first"], c["ngames"], caller_moves=True)
    ev.close()
    mine = setting_evalnet(c["ev"])
    with selfplay_engine(c, c["slots"], c["slots"]) as eng:
        eng.attach_evalnet(mine, use_cuda_graph=False)
        got = walk_trees(eng, c["ngames"], c["sims"], c["first"])
        assert eng.check_guards()[1] == 0
    mine.status()
    mine.close()
    G.assert_trace_equal(ref, got, [k for k in STEP_KEYS if k != "game_winner"])
