"""The evaluator network with a 128-channel tower (csrc/evalnet.cu: k_evalnet<., 128> and k_heads<128>): validation of
the width, accuracy against the fp64 forward on both lattices and at the shape limits, batches around k_heads' 32-board
step, row independence, the device-side row count, update() under a captured graph, and self-play and the C++ veneer
with a 2x128 Othello evaluator.

The accuracy rule is the one of test_evalnet_edges.py: |d| <= 2e-6 * max(1, A) against the fp64 forward, where A is the
largest |BatchNorm output|, A < 4,094, and status() clean."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch
from torch import nn

from sprl_b200 import capi
from sprl_b200.evalnet import EvalNet, network_params
from sprl_b200.network import BasicGridNetwork
from test_evalnet import randomized
from test_evalnet_edges import assert_close, boards, fp64_forward, layer_shifts

WIDE = 128
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def wide_net(rows, cols, policy_channels, planes, blocks, actions, seed=0, channels=WIDE):
    """BasicGridNetwork of a 128-channel tower with randomized BatchNorm (an even plane count replaces the stem)."""
    torch.manual_seed(seed)
    net = BasicGridNetwork(rows, cols, actions, (planes - 1) // 2, blocks, channels, num_policy_channels=policy_channels)
    if planes % 2 == 0:
        net.conv = nn.Conv2d(planes, channels, 3, 1, 1)
    return randomized(net.eval(), seed + 100)


def othello_wide(seed=0):
    return wide_net(8, 8, 2, 3, 2, 65, seed=seed)


def create(net, rows, cols):
    lib = capi.load()
    p, keep = network_params(net.state_dict(), rows=rows, cols=cols)
    h = C.c_void_p()
    rc = lib.sprl_evalnet_create(0, C.byref(p), C.byref(h))
    return lib, rc, h


def rc_of(fn, *args):
    try:
        fn(*args)
    except capi.SprlError as e:
        return e.code
    return capi.SPRL_OK


def heads_smem_bytes_wide(policy_channels, cells):
    """Shared memory of k_heads<128> (heads_smem_bytes in csrc/evalnet.cu): policy weights [K][84], value weights
    [cells][128], two 32-board activation buffers, the hidden layer [32][129] and the lone-tail weights [K]."""
    hp_stride, hb, vh, k = 84, 32, WIDE, policy_channels * cells
    return 4 * (k * hp_stride + cells * vh + 2 * hb * (policy_channels + 1) * cells + hb * (vh + 1) + k)


def max_cells_wide(policy_channels):
    return max(c for c in range(1, 129) if heads_smem_bytes_wide(policy_channels, c) <= 227 * 1024)


# ------------------------------------------------------------------ validation (no GPU needed)
@pytest.mark.parametrize("shape", [(8, 8, 2, 3, 2, 65), (6, 7, 2, 3, 2, 7), (9, 9, 2, 17, 6, 82), (3, 5, 1, 21, 7, 84)],
                         ids=lambda s: "x".join(map(str, s)))
def test_wide_network_passes_validation(shape):
    """Without a GPU create() gets past validation and reports SPRL_E_NOGPU; with one it creates the evaluator."""
    rows, cols = shape[:2]
    lib, rc, h = create(wide_net(*shape), rows, cols)
    assert rc != capi.SPRL_E_INVALID, lib.sprl_last_error()
    if rc == capi.SPRL_OK:
        assert h
        lib.sprl_evalnet_destroy(h)
    else:
        assert rc == capi.SPRL_E_NOGPU and not h, (rc, lib.sprl_last_error())


@pytest.mark.parametrize("channels", [96, 192])
def test_other_widths_are_refused(channels):
    lib, rc, h = create(wide_net(8, 8, 2, 3, 1, 65, channels=channels), 8, 8)
    assert rc == capi.SPRL_E_INVALID and not h
    assert b"64 or 128 channels" in lib.sprl_last_error()


@pytest.mark.parametrize("channels,hidden", [(WIDE, 64), (64, WIDE)])
def test_value_hidden_must_match_the_tower(channels, hidden):
    net = wide_net(8, 8, 2, 3, 1, 65, channels=channels)
    net.value_fc1 = nn.Linear(64, hidden)
    net.value_fc2 = nn.Linear(hidden, 1)
    lib, rc, h = create(net, 8, 8)
    assert rc == capi.SPRL_E_INVALID and not h
    assert b"value hidden" in lib.sprl_last_error()


def test_k_heads_shared_memory_limits_the_wide_board():
    """With a 128-wide value hidden layer k_heads stages 32 boards a step: two policy channels fit 227 KB up to 110
    cells (Go 9x9 included), one policy channel the whole 128-cell tile."""
    assert max_cells_wide(2) == 110
    assert max_cells_wide(1) == 128


# ------------------------------------------------------------------ accuracy against fp64
# (rows, cols, policy channels, planes, blocks, actions)
WIDE_SHAPES = [
    (8, 8, 2, 3, 2, 65),          # Othello
    (6, 7, 2, 3, 2, 7),           # Connect Four
    (7, 7, 2, 17, 6, 50),         # Go 7x7 (pair lattice), 17 planes
    (9, 9, 2, 17, 6, 82),         # Go 9x9 (linear lattice)
    (8, 8, 2, 3, 0, 65),          # blocks: 0
    (9, 9, 2, 3, 1, 82),          # ... 1 on the linear lattice
    (8, 8, 1, 3, 7, 64),          # ... 7, one policy channel
    (5, 8, 2, 21, 1, 41),         # planes: 21
    (6, 6, 2, 2, 1, 37),          # ... an even count
    (10, 11, 2, 3, 1, 84),        # the largest board k_heads<128> takes with two policy channels (110 cells)
    (16, 8, 1, 3, 1, 84),         # a full 128-lane tile, one policy channel
]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", WIDE_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_wide_shape_sweep(shape):
    rows, cols, pc, planes, blocks, actions = shape
    net = wide_net(rows, cols, pc, planes, blocks, actions, seed=rows * 31 + cols)
    x = boards(net, 37, rows, cols, seed=planes)
    want_l, want_v, a = fp64_forward(net, x)
    ev = EvalNet(net, device=0, rows=rows, cols=cols)
    assert ev.phases == 0                                      # AUTO runs the streaming kernel
    l, v = ev(x.cuda())
    assert l.shape == (37, actions) and v.shape == (37, 1)
    ev.status()
    assert_close(l, v, want_l, want_v, a)
    ev.close()


@pytest.mark.gpu
def test_wide_board_too_large_for_k_heads_is_refused():
    assert max_cells_wide(2) < 8 * 14
    lib, rc, h = create(wide_net(8, 14, 2, 3, 1, 84), 8, 14)
    assert rc == capi.SPRL_E_INVALID and not h
    assert b"do not fit k_heads' shared memory" in lib.sprl_last_error()
    lib, rc, h = create(wide_net(8, 14, 1, 3, 1, 84), 8, 14)   # one policy channel: the same board fits
    assert rc == capi.SPRL_OK and h
    lib.sprl_evalnet_destroy(h)


@pytest.mark.gpu
def test_wide_network_runs_on_the_streaming_kernel_only():
    net = othello_wide()
    ev = EvalNet(net, device=0)
    assert ev.phases == 0
    assert rc_of(ev.set_path, capi.EVALNET_PATH_RESIDENT) == capi.SPRL_E_STATE
    assert rc_of(ev.set_precision, capi.EVALNET_PRECISION_FP16) == capi.SPRL_E_STATE
    assert ev.phases == 0
    ev.set_path(capi.EVALNET_PATH_STREAMING)
    ev.set_path(capi.EVALNET_PATH_AUTO)
    info = ev.info()
    assert info["ring_stages"] >= 4 and info["smem_bytes"] <= 227 * 1024
    ev.close()


# ------------------------------------------------------------------ batches
WIDE_BATCHES = [1, 2, 3, 31, 32, 33, 63, 64, 65, 129]
BIG_ODD = 4099


def _batch_net(kind):
    if kind == "8x8":
        return othello_wide(seed=31), 8, 8
    return wide_net(9, 9, 2, 17, 2, 82, seed=32), 9, 9


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["8x8", "linear"])
def test_wide_batch_edges(kind):
    """Batches around a tile pair and k_heads' 32-board step, and an odd batch over 4,096: every batch gives the bits of
    the same rows in the largest one, and sampled rows of that one match fp64."""
    net, rows, cols = _batch_net(kind)
    x = boards(net, BIG_ODD, rows, cols, seed=1)
    xg = x.cuda()
    ev = EvalNet(net, device=0, rows=rows, cols=cols)
    l_all, v_all = ev(xg)
    small = max(WIDE_BATCHES)
    want_l, want_v, a = fp64_forward(net, x[:small])
    for n in WIDE_BATCHES:
        l, v = ev(xg[:n])
        assert l.shape == (n, want_l.shape[1])
        assert_close(l, v, want_l[:n], want_v[:n], a)
        assert torch.equal(l, l_all[:n]) and torch.equal(v, v_all[:n])
    idx = torch.arange(small, BIG_ODD, 61)
    want_l, want_v, a = fp64_forward(net, x[idx])
    assert_close(l_all[idx.cuda()], v_all[idx.cuda()], want_l, want_v, a)
    ev.status()
    ev.close()


@pytest.mark.gpu
def test_wide_othello_at_the_mean_leaf_batch():
    """61,952 rows (the benchmark's mean leaf batch): a row sample against fp64, and those rows evaluated on their own
    give the same bits."""
    net = othello_wide(seed=33)
    n = 61952
    x = boards(net, n, 8, 8, seed=2)
    ev = EvalNet(net, device=0)
    l_all, v_all = ev(x.cuda())
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:256]
    want_l, want_v, a = fp64_forward(net, x[idx])
    assert_close(l_all[idx.cuda()], v_all[idx.cuda()], want_l, want_v, a)
    l_s, v_s = ev(x[idx].cuda())
    assert torch.equal(l_s, l_all[idx.cuda()]) and torch.equal(v_s, v_all[idx.cuda()])
    ev.status()
    ev.close()


# ------------------------------------------------------------------ determinism and the device-side row count
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["8x8", "linear"])
def test_wide_outputs_do_not_depend_on_the_row(kind):
    """A board's outputs are the same bits wherever it sits in the batch, whoever its tile partner is (8x8 lattice) and
    whatever the grid size."""
    net, rows, cols = _batch_net(kind)
    ev = EvalNet(net, device=0, rows=rows, cols=cols)
    g = torch.Generator().manual_seed(5)
    x = boards(net, 1501, rows, cols, seed=3).cuda()
    perm = torch.randperm(x.shape[0], generator=g).cuda()
    l0, v0 = ev(x)
    l1, v1 = ev(x[perm])
    assert torch.equal(l0[perm], l1) and torch.equal(v0[perm], v1)
    l2, v2 = ev(x[:77])
    assert torch.equal(l0[:77], l2) and torch.equal(v0[:77], v2)
    ev.status()
    ev.close()


COUNTED_BATCH = 67


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["8x8", "linear"])
def test_wide_forward_counted(kind):
    """The row count read on the device: rows [0, min(count, batch)) get the plain forward's bits, the other rows are
    not written.  Then the same inside a captured CUDA graph, the count changed between replays."""
    net, rows, cols = _batch_net(kind)
    ev = EvalNet(net, device=0, rows=rows, cols=cols)
    x = boards(net, COUNTED_BATCH, rows, cols, seed=4).cuda()
    want_l, want_v = ev(x)
    logits = torch.empty_like(want_l)
    value = torch.empty(COUNTED_BATCH, device="cuda")
    d_rows = torch.zeros(1, dtype=torch.int32, device="cuda")
    stream = lambda: torch.cuda.current_stream().cuda_stream

    def run():
        ev.forward_ptr(x.data_ptr(), COUNTED_BATCH, logits.data_ptr(), value.data_ptr(), stream(), d_rows=d_rows.data_ptr())

    def check(count):
        n = min(count, COUNTED_BATCH)
        assert torch.equal(logits[:n], want_l[:n]) and torch.equal(value[:n], want_v[:n].reshape(-1)), count
        assert torch.isnan(logits[n:]).all() and torch.isnan(value[n:]).all(), count

    counts = [0, 1, COUNTED_BATCH // 2, COUNTED_BATCH, COUNTED_BATCH + 5]
    for count in counts:
        d_rows.fill_(count)
        logits.fill_(float("nan"))
        value.fill_(float("nan"))
        run()
        torch.cuda.synchronize()
        check(count)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        run()
    for count in counts[::-1] + counts:
        d_rows.fill_(count)
        logits.fill_(float("nan"))
        value.fill_(float("nan"))
        graph.replay()
        torch.cuda.synchronize()
        check(count)
    ev.status()
    del graph
    ev.close()


# ------------------------------------------------------------------ update()
def _update_nets(kind):
    """(A, B, rows, cols): two 128-channel networks of one shape whose per-layer weight shifts differ."""
    if kind == "8x8":
        torch.manual_seed(40)
        a = BasicGridNetwork(8, 8, 65, 1, 2, WIDE).eval()
        return a, othello_wide(seed=41), 8, 8
    torch.manual_seed(42)
    a = BasicGridNetwork(9, 9, 82, 8, 2, WIDE).eval()
    return a, wide_net(9, 9, 2, 17, 2, 82, seed=43), 9, 9


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["8x8", "linear"])
def test_wide_update_reaches_a_captured_graph(kind):
    """A graph captured with network A and replayed after update(B) computes B: the same bits as a fresh evaluator of B."""
    a, b, rows, cols = _update_nets(kind)
    assert layer_shifts(a) != layer_shifts(b)
    n = 300
    x = boards(a, n, rows, cols, seed=6)
    want_l, want_v, amax = fp64_forward(b, x)
    xg = x.cuda()
    ev = EvalNet(a, device=0, rows=rows, cols=cols)
    logits = torch.empty(n, want_l.shape[1], device="cuda")
    value = torch.empty(n, device="cuda")
    stream = lambda: torch.cuda.current_stream().cuda_stream
    ev.forward_ptr(xg.data_ptr(), n, logits.data_ptr(), value.data_ptr(), stream())      # sizes the buffers
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ev.forward_ptr(xg.data_ptr(), n, logits.data_ptr(), value.data_ptr(), stream())
    graph.replay()
    torch.cuda.synchronize()
    l_a = logits.clone()

    ev.update(b)
    logits.fill_(float("nan"))
    value.fill_(float("nan"))
    graph.replay()
    torch.cuda.synchronize()
    ev.status()
    fresh = EvalNet(b, device=0, rows=rows, cols=cols)
    l_b, v_b = fresh(xg)
    fresh.status()
    assert (l_a - l_b).abs().max().item() > 1e-3
    assert torch.equal(logits, l_b) and torch.equal(value, v_b.reshape(-1))
    assert_close(logits, value, want_l, want_v, amax)
    del graph
    ev.close()
    fresh.close()


@pytest.mark.gpu
def test_update_refuses_a_change_of_width():
    wide = othello_wide()
    narrow = wide_net(8, 8, 2, 3, 2, 65, channels=64)
    for first, second in ((wide, narrow), (narrow, wide)):
        ev = EvalNet(first, device=0)
        with pytest.raises(capi.SprlError) as e:
            ev.update(second)
        assert e.value.code == capi.SPRL_E_INVALID and "shape changed" in str(e.value)
        ev.close()


# ------------------------------------------------------------------ end to end
@pytest.mark.gpu
def test_selfplay_with_a_wide_evaluator_tracks_libtorch():
    """Self-play with a 2x128 Othello evaluator: the first move's root priors match the LibTorch path of the same
    module, and two runs with the same seed give the same samples."""
    from sprl_b200 import selfplay as SP
    from sprl_b200.network import trace_network
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    net = othello_wide(seed=44)
    kw = dict(seed=8, sims=48, max_batch=8, max_queue=4, num_slots=16, max_games=16, record_stats=1, add_noise=0)
    out = {}
    for kind in ("evalnet", "evalnet_again", "libtorch"):
        with SP.Engine(capi.GAME_OTHELLO, capi.EVAL_EXTERNAL, **kw) as eng:
            if kind.startswith("evalnet"):
                ev = EvalNet(net, device=0)
                eng.attach_evalnet(ev, use_cuda_graph=True)
            else:
                eng.attach_network(trace_network(net, torch.device("cuda", 0)), use_cuda_graph=False)
            samples = eng.run_iteration(16)
            out[kind] = (eng.move_stats(16), samples)
        if kind.startswith("evalnet"):
            ev.status()
            ev.close()
    (ma, sa), (mb, sb) = out["evalnet"], out["libtorch"]
    first_a = np.concatenate([[0], np.cumsum(ma["game_moves"])[:-1]])
    first_b = np.concatenate([[0], np.cumsum(mb["game_moves"])[:-1]])
    assert np.allclose(ma["move_P"][first_a], mb["move_P"][first_b], atol=1e-5)
    for g, w in zip(sa, out["evalnet_again"][1]):
        assert np.array_equal(g, w)
    states, dists, outcomes = sa
    assert states.shape[0] == dists.shape[0] == outcomes.shape[0] and states.shape[0] % 8 == 0
    assert np.allclose(dists.sum(1), 1.0, atol=1e-5) and set(np.unique(outcomes)) <= {-1.0, 0.0, 1.0}


@pytest.mark.gpu
def test_host_network_with_a_wide_module_uses_the_kernel(tmp_path):
    """The C++ veneer's GridNetwork with a traced 2x128 Othello module takes the tcgen05 evaluator (not the LibTorch
    fallback) and INetwork::evaluate matches PyTorch on the CPU."""
    from sprl_b200.network import trace_network
    host = os.path.join(ROOT, "sprl_b200", "host")
    binary = os.path.join(host, "bin", "netcheck")
    if not os.path.exists(binary):
        subprocess.run(["make", "-C", host, "check"], check=True, capture_output=True)
    net = othello_wide(seed=45)
    pt = str(tmp_path / "net.pt")
    trace_network(net, "cpu").save(pt)
    prefix = str(tmp_path / "out")
    r = subprocess.run([binary, pt, "300", "11", prefix], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout + r.stderr)[-2000:]
    assert "Evaluator: tcgen05 network kernel" in r.stdout, r.stdout[-2000:]
    assert "300 + 300 evaluations counted" in r.stdout
    cells, player, mask, policy, value = (np.load(prefix + f"_{k}.npy") for k in ("cells", "player", "mask", "policy", "value"))
    mine = (cells == player[:, None]).astype(np.float32).reshape(-1, 8, 8)
    theirs = (cells == (1 - player)[:, None]).astype(np.float32).reshape(-1, 8, 8)
    turn = np.broadcast_to((player == 0).astype(np.float32)[:, None, None], mine.shape)
    with torch.no_grad():
        logits, v = net(torch.from_numpy(np.stack([mine, theirs, turn], 1).copy()))
    want = np.exp(logits.numpy()) * mask
    want /= want.sum(1, keepdims=True)
    assert np.abs(policy - want).max() <= 1e-6 and np.abs(value - v.numpy().reshape(-1)).max() <= 1e-6
    assert np.allclose(policy.sum(1), 1.0, atol=1e-6) and not (policy[mask == 0] != 0).any()
