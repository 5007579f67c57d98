"""The C++ side of the drop-in boundary on the GPU (sprl_b200/host): the worker executables and a move loop over the
veneer's UCTTree -- their outputs against the Python engine on the same stream ids and against the golden traces of the
verbatim reference.

The binaries are built by __graft_entry__.build() (`make -C sprl_b200/host all check`); what is missing is built here."""
import os
import struct
import subprocess

import numpy as np
import pytest

import golden_util as G
from sprl_b200 import capi
from sprl_b200 import selfplay as SP

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "sprl_b200", "host")
BIN = os.path.join(HOST, "bin")


def binary(name, target):
    path = os.path.join(BIN, name)
    if not os.path.exists(path):
        subprocess.run(["make", "-C", HOST, target], check=True, capture_output=True)
    assert os.path.exists(path), f"{path} is missing: run __graft_entry__.build()"
    return path


def load_triple(base):
    return tuple(np.load(base + suffix) for suffix in ("_states.npy", "_distributions.npy", "_outcomes.npy"))


def test_othworker_files_equal_the_engine_on_the_same_streams(tmp_path):
    """bin/OTHWorker (runWorker of selfplay/GridWorker.hpp:84-198 over the C ABI), sized by environment variables:
    iteration 0 with the uniform evaluator, its three .npy files bit-identical to Engine.run_iteration on the stream
    ids task 5 of 16 plays (5, 21, 37, ...)."""
    exe = binary("OTHWorker", "all")
    env = dict(os.environ, SPRL_RUN_NAME="hosttest", SPRL_NUM_GROUPS="4", SPRL_NUM_ITERS="1", SPRL_INIT_NUM_GAMES="6",
               SPRL_INIT_UCT_TRAVERSALS="96", SPRL_INIT_MAX_BATCH_SIZE="8", SPRL_INIT_MAX_QUEUE_SIZE="4", SPRL_SEED="77",
               SPRL_NUM_SLOTS="4")
    r = subprocess.run([exe, "5", "16"], cwd=tmp_path, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "Task 5 of 16, in group 1." in r.stdout and "Using initial network..." in r.stdout
    got = load_triple(str(tmp_path / "data" / "games" / "hosttest" / "1" / "5" / "hosttest_iteration_0"))
    with SP.Engine(capi.GAME_OTHELLO, capi.EVAL_UNIFORM, seed=77, sims=96, max_batch=8, max_queue=4, dir_eps=0.25, dir_alpha=0.3,
                   num_slots=4, max_games=6) as eng:
        eng.set_game_stride(16)
        want = eng.run_iteration(6, first_game=5)
    for a, b in zip(got, want):
        assert a.dtype == np.float32 and np.array_equal(a, b)
    assert got[0].shape[1:] == (3, 8, 8) and got[1].shape[1] == 65 and got[0].shape[0] % 8 == 0


def read_treewalk(path):
    raw = open(path, "rb").read()
    ngames, A = struct.unpack_from("<ii", raw, 0)
    at = 8
    out = dict(game_moves=[], game_winner=[], move_N=[], move_W=[], move_P=[], move_root_N=[], move_root_W=[], move_action=[],
               move_traversals=[], move_player=[])
    for _ in range(ngames):
        moves, winner = struct.unpack_from("<ii", raw, at)
        at += 8
        out["game_moves"].append(moves)
        out["game_winner"].append(winner)
        for _ in range(moves):
            f = np.frombuffer(raw, np.float32, 3 * A + 2, at)
            at += 4 * (3 * A + 2)
            action, trav, player = struct.unpack_from("<iii", raw, at)
            at += 12
            out["move_N"].append(f[:A]); out["move_W"].append(f[A:2 * A]); out["move_P"].append(f[2 * A:3 * A])
            out["move_root_N"].append(f[3 * A]); out["move_root_W"].append(f[3 * A + 1])
            out["move_action"].append(action); out["move_traversals"].append(trav); out["move_player"].append(player)
    assert at == len(raw)
    kinds = dict(game_moves=np.int32, game_winner=np.int32, move_action=np.int32, move_traversals=np.int32, move_player=np.int8)
    return {k: np.array(v, kinds.get(k, np.float32)) for k, v in out.items()}


@pytest.mark.parametrize("name", [n for n in G.TREEWALK_FIXTURES if not n.startswith("go9")])
def test_veneer_ucttree_move_loop_matches_the_reference(name, tmp_path):
    """tests/hostcheck/treewalk.cpp: a C++ move loop written against uct/UCTTree.hpp's public surface
    (searchAndGetLeaves / evaluateAndBackpropLeaves / getDecisionNode / advanceDecision), compiled against the veneer,
    against the golden trace the verbatim reference produced with the same loop."""
    exe = binary("treewalk", "check")
    cmd, ref = G.load("treewalk_" + name)
    out = str(tmp_path / "walk.bin")
    args = [exe, cmd["game"], cmd["seed"], cmd["first_game"], cmd["ngames"], cmd["sims"], cmd["max_batch"], cmd["max_queue"],
            cmd["eps"], cmd["alpha"], cmd["noise"], cmd["sym"], cmd["initq"], out]
    r = subprocess.run([str(x) for x in args], env=dict(os.environ, SPRL_SEED=str(cmd["seed"])), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    got = read_treewalk(out)
    G.assert_trace_equal(ref, got, ["game_moves", "game_winner", "move_N", "move_W", "move_P", "move_root_N", "move_root_W",
                                    "move_action", "move_traversals", "move_player"])


def test_host_gamenode_and_gridstate_follow_the_device_rules():
    """The veneer's GameNode / GridState (games/GameNode.hpp:50-200, games/GridState.hpp:56-115) node by node against one
    sprl_env_line call per game, for Othello, Connect Four and Go: tests/hostcheck/gamenode.cpp."""
    r = subprocess.run([binary("gamenode", "check"), "7"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "gamenode ok" in r.stdout


def test_host_inetwork_evaluate_matches_the_module(tmp_path):
    """INetwork::evaluate(states, masks) for host callers (networks/INetwork.hpp:25-27): the veneer's GridNetwork embeds
    GridStates, runs the traced module on the GPU and applies the reference's exp / mask / normalise on the host
    (networks/GridNetwork.hpp:72-142); tests/hostcheck/netcheck.cpp evaluates 300 positions of random Othello games, PyTorch
    recomputes them from the same module on the CPU.  RandomNetwork: uniform over the legal actions."""
    import torch
    from sprl_b200.network import make_network, trace_network
    net = make_network("othello", 3)
    pt = str(tmp_path / "net.pt")
    trace_network(net, "cpu").save(pt)
    prefix = str(tmp_path / "out")
    r = subprocess.run([binary("netcheck", "check"), pt, "300", "11", prefix], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout + r.stderr)[-2000:]
    assert "300 + 300 evaluations counted" in r.stdout
    cells, player, mask, policy, value, uniform = (np.load(prefix + f"_{k}.npy") for k in ("cells", "player", "mask", "policy", "value", "uniform"))
    mine = (cells == player[:, None]).astype(np.float32).reshape(-1, 8, 8)
    theirs = (cells == (1 - player)[:, None]).astype(np.float32).reshape(-1, 8, 8)
    turn = np.broadcast_to((player == 0).astype(np.float32)[:, None, None], mine.shape)
    with torch.no_grad():
        logits, v = net(torch.from_numpy(np.stack([mine, theirs, turn], 1).copy()))
    want = np.exp(logits.numpy()) * mask
    want /= want.sum(1, keepdims=True)
    assert np.abs(policy - want).max() <= 1e-6 and np.abs(value - v.numpy().reshape(-1)).max() <= 1e-6
    assert np.allclose(policy.sum(1), 1.0, atol=1e-6) and not (policy[mask == 0] != 0).any()
    assert np.allclose(uniform, mask / mask.sum(1, keepdims=True), atol=1e-7)
