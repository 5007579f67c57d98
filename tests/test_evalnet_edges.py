"""The evaluator network (csrc/evalnet.cu, csrc/evalnet_resident.cuh) at the edges of what its C ABI accepts: board shapes
on both lattices, plane / block / action / policy-channel limits, batch sizes around tile pairs, quads and k_heads' 64-board
step, CTA pairs that loop over quads, the device-side row count of sprl_evalnet_forward_counted, and sprl_evalnet_update
under a captured CUDA graph.

Reference: the fp64 CPU forward of the same `BasicGridNetwork` with non-trivial BatchNorm.  The fp16 split keeps ~22
significant bits of every operand, so the error is bounded relative to the largest intermediate activation `A` (the
largest |BatchNorm output| of the fp64 forward): |d| <= 2e-6 * max(1, A).  Every case also asserts A < 4,094 (the split's
range, so the case tests accuracy and not range) and calls status(), which fails on an out-of-range report or a
pipeline-barrier time-out."""
import ctypes as C
import math

import numpy as np
import pytest
import torch
from torch import nn

from sprl_b200 import capi
from sprl_b200.evalnet import EvalNet, network_params
from sprl_b200.network import BasicGridNetwork, make_network
from test_evalnet import randomized

TOL, TOL_PATHS, TOL_FP16 = 2e-6, 1e-6, 5e-3
HALF_RANGE = 4094.0                      # 65504 / 2^ACT_SHIFT: the largest activation the fp16 split represents


def grid_net(rows, cols, policy_channels, planes, blocks, actions, seed=0):
    """BasicGridNetwork of any shape the evaluator accepts, with randomized BatchNorm.  An even plane count cannot be
    built from a history size: the stem is replaced (network_params reads in_planes from its weight)."""
    torch.manual_seed(seed)
    net = BasicGridNetwork(rows, cols, actions, (planes - 1) // 2, blocks, 64, num_policy_channels=policy_channels)
    if planes % 2 == 0:
        net.conv = nn.Conv2d(planes, 64, 3, 1, 1)
    return randomized(net.eval(), seed + 100)


def planes_of(net):
    return net.conv.in_channels


def boards(net, n, rows, cols, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(n, planes_of(net), rows, cols, generator=g) > 0.5).float()


def fp64_forward(net, x):
    """(logits, value, A): the fp64 forward of `net` and the largest |BatchNorm output| in it."""
    acts = []
    hooks = [m.register_forward_hook(lambda _m, _i, out: acts.append(out.abs().max().item()))
             for m in net.modules() if isinstance(m, nn.BatchNorm2d)]
    try:
        with torch.no_grad():
            want_l, want_v = net.double()(x.double())
    finally:
        net.float()
        for h in hooks:
            h.remove()
    return want_l, want_v, max(acts)


def err(got, want):
    return (got.cpu().double().reshape(want.shape) - want).abs().max().item()


def assert_close(got_l, got_v, want_l, want_v, a, tol=TOL):
    assert a < HALF_RANGE, a
    bound = tol * max(1.0, a)
    el, ev_ = err(got_l, want_l), err(got_v, want_v)
    assert el <= bound and ev_ <= bound, (el, ev_, bound)


def layer_shifts(net, eps=1e-5):
    """Per-layer power of two the evaluator scales the folded weights by (weight_shift in csrc/evalnet.cu): the one that
    brings the layer's largest |weight| into (2^9, 2^10].  Stem, the tower's convolutions, then the 1x1 heads."""
    def fold(conv, bn):
        scale = bn.weight.detach().double() / torch.sqrt(bn.running_var.double() + eps)
        return (conv.weight.detach().double() * scale.view(-1, 1, 1, 1)).float()
    convs = [(net.conv, net.bn)] + [(getattr(b, f"conv{i}"), getattr(b, f"bn{i}")) for b in net.residual_blocks for i in (1, 2)]
    ws = [fold(c, b) for c, b in convs]
    ws.append(torch.cat([net.policy_conv.weight.detach().reshape(-1), net.value_conv.weight.detach().reshape(-1)]))
    return [max(-40, min(40, 10 - math.frexp(w.abs().max().item())[1])) for w in ws]


def heads_smem_bytes(policy_channels, cells):
    """Shared memory of k_heads (heads_smem_bytes in csrc/evalnet.cu): policy weights [K][84], value weights [cells][64],
    two 64-board activation buffers, the hidden layer [64][65] and the lone-tail weights [K]."""
    hp_stride, hb, k = 84, 64, policy_channels * cells
    return 4 * (k * hp_stride + cells * 64 + 2 * hb * (policy_channels + 1) * cells + hb * 65 + k)


K_HEADS_SMEM = 227 * 1024


def max_cells(policy_channels):
    return max(c for c in range(1, 129) if heads_smem_bytes(policy_channels, c) <= K_HEADS_SMEM)


# ------------------------------------------------------------------ validation limits, both sides
# (rows, cols, policy channels, planes, blocks, actions); every accepted shape keeps the others at small values
ACCEPTED = [
    (3, 5, 2, 3, 7, 10),          # blocks: 7
    (3, 5, 2, 3, 0, 10),          # ... and none
    (3, 5, 2, 21, 1, 10),         # in_planes: 21
    (3, 5, 2, 1, 1, 10),          # ... and 1
    (3, 5, 2, 2, 1, 10),          # ... an even count
    (3, 5, 2, 3, 1, 84),          # actions: 84
    (3, 5, 2, 3, 1, 1),           # ... and 1
    (3, 5, 1, 3, 1, 10),          # policy channels: 1 and 2
    (1, 16, 2, 3, 1, 10),         # cols: 16
    (16, 8, 1, 3, 1, 10),         # cells: 128
    (8, 16, 1, 3, 1, 10),
    (7, 12, 2, 3, 1, 10),         # two policy channels: 84 cells, the largest board k_heads stages with rows <= 16 wide
]
REFUSED = [
    (3, 5, 2, 3, 8, 10),          # blocks: 8
    (3, 5, 2, 22, 1, 10),         # in_planes: 22
    (3, 5, 2, 3, 1, 85),          # actions: 85
    (3, 5, 3, 3, 1, 10),          # policy channels: 3
    (1, 17, 2, 3, 1, 10),         # cols: 17
    (1, 129, 1, 3, 1, 10),        # cells: 129 (and cols)
    (9, 15, 1, 3, 1, 10),         # cells: 135, cols <= 16
    (11, 12, 1, 3, 1, 10),        # cells: 132, cols <= 16
]


def _create(shape):
    rows, cols, pc, planes, blocks, actions = shape
    torch.manual_seed(0)
    net = BasicGridNetwork(rows, cols, actions, (planes - 1) // 2, blocks, 64, num_policy_channels=pc)
    if planes % 2 == 0:
        net.conv = nn.Conv2d(planes, 64, 3, 1, 1)
    lib = capi.load()
    p, keep = network_params(net.state_dict(), rows=rows, cols=cols)
    assert (p.rows, p.cols, p.policy_channels, p.in_planes, p.blocks, p.actions) == shape
    h = C.c_void_p()
    rc = lib.sprl_evalnet_create(0, C.byref(p), C.byref(h))
    return lib, rc, h


@pytest.mark.parametrize("shape", ACCEPTED, ids=lambda s: "x".join(map(str, s)))
def test_evalnet_accepts_shapes_at_the_limits(shape):
    """Without a GPU create() gets past validation and reports SPRL_E_NOGPU; with one it creates the evaluator."""
    lib, rc, h = _create(shape)
    assert rc != capi.SPRL_E_INVALID, lib.sprl_last_error()
    if rc == capi.SPRL_OK:
        assert h
        lib.sprl_evalnet_destroy(h)
    else:
        assert rc == capi.SPRL_E_NOGPU and not h, (rc, lib.sprl_last_error())


@pytest.mark.parametrize("shape", REFUSED, ids=lambda s: "x".join(map(str, s)))
def test_evalnet_refuses_shapes_past_the_limits(shape):
    lib, rc, h = _create(shape)
    assert rc == capi.SPRL_E_INVALID and not h, (rc, lib.sprl_last_error())


def test_k_heads_shared_memory_limits_the_board():
    """Two policy channels fit k_heads' 227 KB up to 87 cells, one policy channel the whole 128-cell tile."""
    assert max_cells(2) == 87
    assert max_cells(1) == 128


@pytest.mark.gpu
def test_evalnet_refuses_boards_too_large_for_k_heads():
    assert 8 * 11 > max_cells(2) >= 7 * 12
    lib, rc, h = _create((8, 11, 2, 3, 1, 10))
    assert rc == capi.SPRL_E_INVALID and not h
    assert b"do not fit k_heads' shared memory" in lib.sprl_last_error()
    lib, rc, h = _create((8, 11, 1, 3, 1, 10))        # one policy channel: the same board fits
    assert rc == capi.SPRL_OK and h
    lib.sprl_evalnet_destroy(h)


# ------------------------------------------------------------------ shape sweep on both kernels and both precisions
SHAPES = [
    # 8x8 lattice (two boards per tile)
    (1, 1, 2, 1, 1, 1),
    (3, 3, 2, 3, 2, 10),
    (1, 8, 2, 3, 2, 9),
    (8, 1, 2, 3, 2, 9),
    (7, 6, 2, 3, 2, 7),
    (5, 8, 2, 21, 7, 41),
    (8, 8, 1, 2, 2, 64),          # no lone tail in k_heads, an even plane count
    (8, 8, 2, 3, 2, 66),
    (8, 8, 2, 3, 2, 84),          # k_heads' HP_STRIDE padding
    # linear lattice (one board per tile, cell = TMEM lane)
    (10, 8, 2, 3, 2, 81),
    (7, 12, 2, 3, 2, 84),
    (1, 16, 2, 3, 2, 17),         # 16 columns: vertical taps use the whole zero padding
    (2, 16, 2, 3, 2, 33),
    (16, 8, 1, 3, 2, 84),         # a full 128-lane tile
    (8, 16, 1, 3, 2, 84),
    (11, 11, 1, 17, 6, 84),
    (128, 1, 1, 3, 1, 84),        # one column: no cell has a left or right neighbour
    (9, 9, 2, 21, 7, 82),
]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_evalnet_shape_sweep(shape):
    rows, cols, pc, planes, blocks, actions = shape
    net = grid_net(rows, cols, pc, planes, blocks, actions, seed=rows * 31 + cols)
    x = boards(net, 37, rows, cols, seed=planes)
    want_l, want_v, a = fp64_forward(net, x)
    xg = x.cuda()
    ev = EvalNet(net, device=0, rows=rows, cols=cols)
    assert ev.phases > 0                                       # AUTO runs the resident-weight kernel
    l_res, v_res = ev(xg)
    assert l_res.shape == (37, actions) and v_res.shape == (37, 1)
    ev.status()
    assert_close(l_res, v_res, want_l, want_v, a)

    ev.set_path(capi.EVALNET_PATH_STREAMING)
    assert ev.phases == 0
    l_str, v_str = ev(xg)
    ev.status()
    assert_close(l_str, v_str, want_l, want_v, a)
    bound = TOL_PATHS * max(1.0, a)
    assert (l_res - l_str).abs().max().item() <= bound and (v_res - v_str).abs().max().item() <= bound

    ev.set_path(capi.EVALNET_PATH_AUTO)
    ev.set_precision(capi.EVALNET_PRECISION_FP16)
    l16, v16 = ev(xg)
    l16b, v16b = ev(xg[:20])                                   # another batch size: the same bits
    ev.status()
    assert_close(l16, v16, want_l, want_v, a, tol=TOL_FP16)
    assert torch.equal(l16b, l16[:20]) and torch.equal(v16b, v16[:20])
    ev.close()


# ------------------------------------------------------------------ batch and grid edges
EDGE_BATCHES = [1, 2, 3, 7, 8, 9, 63, 64, 65, 129]


def _edge_net(kind):
    if kind == "8x8":                                          # Othello's shape with one residual block
        return grid_net(8, 8, 2, 3, 1, 65, seed=21), 8, 8
    return randomized(make_network("go9", 3), 22), 9, 9        # linear lattice, six blocks


@pytest.mark.gpu
@pytest.mark.parametrize("path", [capi.EVALNET_PATH_AUTO, capi.EVALNET_PATH_STREAMING], ids=["resident", "streaming"])
@pytest.mark.parametrize("kind", ["8x8", "linear"])
def test_evalnet_batch_edges(kind, path):
    """Batches around a tile pair (two boards per tile on the 8x8 lattice), a quad of four tiles and k_heads' 64-board step."""
    net, rows, cols = _edge_net(kind)
    x = boards(net, max(EDGE_BATCHES), rows, cols, seed=1)
    want_l, want_v, a = fp64_forward(net, x)
    ev = EvalNet(net, device=0, rows=rows, cols=cols)
    ev.set_path(path)
    xg = x.cuda()
    l_all, v_all = ev(xg)
    for n in EDGE_BATCHES:
        l, v = ev(xg[:n])
        assert l.shape == (n, want_l.shape[1])
        assert_close(l, v, want_l[:n], want_v[:n], a)
        assert torch.equal(l, l_all[:n]) and torch.equal(v, v_all[:n])
    ev.status()
    ev.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind,rows,cols,batch", [("go7", 7, 7, 1801), ("go9", 9, 9, 1203)])
def test_evalnet_pairs_loop_over_quads(kind, rows, cols, batch, monkeypatch):
    """Seven-phase networks at batches where every CTA pair of the resident kernel takes several quads (more than 296
    tiles on 148 SMs), and every CTA of the streaming kernel several tiles.  A second evaluator capped at ONE CTA pair
    (SPRL_EVALNET_MAX_CTAS=2, read once by create) walks every quad itself and must give the same bits."""
    net = randomized(make_network(kind, 4), 23)
    x = boards(net, batch, rows, cols, seed=2)
    want_l, want_v, a = fp64_forward(net, x)
    xg = x.cuda()
    ev = EvalNet(net, device=0, rows=rows, cols=cols)
    assert ev.phases == 7
    l_res, v_res = ev(xg)
    ev.status()
    assert_close(l_res, v_res, want_l, want_v, a)
    ev.set_path(capi.EVALNET_PATH_STREAMING)
    l_str, v_str = ev(xg)
    ev.status()
    assert_close(l_str, v_str, want_l, want_v, a)
    ev.close()

    monkeypatch.setenv("SPRL_EVALNET_MAX_CTAS", "2")
    capped = EvalNet(net, device=0, rows=rows, cols=cols)
    monkeypatch.delenv("SPRL_EVALNET_MAX_CTAS")
    l_cap, v_cap = capped(xg)
    capped.status()
    assert torch.equal(l_cap, l_res) and torch.equal(v_cap, v_res)
    capped.close()


@pytest.mark.gpu
@pytest.mark.parametrize("path", [capi.EVALNET_PATH_AUTO, capi.EVALNET_PATH_STREAMING], ids=["resident", "streaming"])
def test_evalnet_outputs_do_not_depend_on_the_row_linear_lattice(path):
    """Go 9x9: a board's outputs are the same bits wherever it sits in the batch and whatever the grid size."""
    net = randomized(make_network("go9", 1), 24)
    ev = EvalNet(net, device=0, rows=9, cols=9)
    ev.set_path(path)
    g = torch.Generator().manual_seed(5)
    x = boards(net, 777, 9, 9, seed=3).cuda()
    perm = torch.randperm(x.shape[0], generator=g).cuda()
    l0, v0 = ev(x)
    l1, v1 = ev(x[perm])
    assert torch.equal(l0[perm], l1) and torch.equal(v0[perm], v1)
    l2, v2 = ev(x[:77])
    assert torch.equal(l0[:77], l2) and torch.equal(v0[:77], v2)
    ev.status()
    ev.close()


# ------------------------------------------------------------------ sprl_evalnet_forward_counted
COUNTED_BATCH = 67


def _counted(ev, x, d_rows, logits, value):
    ev.forward_ptr(x.data_ptr(), x.shape[0], logits.data_ptr(), value.data_ptr(),
                   torch.cuda.current_stream().cuda_stream, d_rows=d_rows.data_ptr())


def _check_counted(count, logits, value, want_l, want_v):
    n = min(count, COUNTED_BATCH)
    assert torch.equal(logits[:n], want_l[:n]) and torch.equal(value[:n], want_v[:n].reshape(-1)), count
    assert torch.isnan(logits[n:]).all() and torch.isnan(value[n:]).all(), count       # rows past the count: untouched


@pytest.mark.gpu
@pytest.mark.parametrize("path", [capi.EVALNET_PATH_AUTO, capi.EVALNET_PATH_STREAMING], ids=["resident", "streaming"])
@pytest.mark.parametrize("kind", ["8x8", "linear"])
def test_evalnet_forward_counted(kind, path):
    """The row count read on the device (the engine's leaf count): rows [0, min(count, batch)) get the plain forward's
    bits, every other row is left as it was.  Then the same inside a captured CUDA graph, the count changed between
    replays."""
    net, rows, cols = _edge_net(kind)
    ev = EvalNet(net, device=0, rows=rows, cols=cols)
    ev.set_path(path)
    x = boards(net, COUNTED_BATCH, rows, cols, seed=4).cuda()
    want_l, want_v = ev(x)
    logits = torch.empty_like(want_l)
    value = torch.empty(COUNTED_BATCH, device="cuda")
    d_rows = torch.zeros(1, dtype=torch.int32, device="cuda")
    counts = [0, 1, COUNTED_BATCH // 2, COUNTED_BATCH, COUNTED_BATCH + 5]
    for count in counts:
        d_rows.fill_(count)
        logits.fill_(float("nan"))
        value.fill_(float("nan"))
        _counted(ev, x, d_rows, logits, value)
        torch.cuda.synchronize()
        _check_counted(count, logits, value, want_l, want_v)

    d_rows.fill_(COUNTED_BATCH)
    _counted(ev, x, d_rows, logits, value)                     # the full batch once before capture (buffers are sized)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        _counted(ev, x, d_rows, logits, value)
    for count in counts[::-1] + counts:
        d_rows.fill_(count)
        logits.fill_(float("nan"))
        value.fill_(float("nan"))
        graph.replay()
        torch.cuda.synchronize()
        _check_counted(count, logits, value, want_l, want_v)
    ev.status()
    del graph
    ev.close()


# ------------------------------------------------------------------ sprl_evalnet_update under a captured graph
def _update_nets(kind):
    """(A, B, rows, cols, phases): two networks of one shape whose per-layer weight shifts differ."""
    if kind == "othello":                                      # two blocks: two resident phases
        return make_network("othello", 0), randomized(make_network("othello", 2), 2), 8, 8, 2
    if kind == "noblocks":                                     # stem and heads only: one phase
        torch.manual_seed(0)
        a = BasicGridNetwork(8, 8, 65, 1, 0, 64).eval()
        torch.manual_seed(1)
        return a, randomized(BasicGridNetwork(8, 8, 65, 1, 0, 64).eval(), 1), 8, 8, 1
    return make_network("go9", 0), randomized(make_network("go9", 2), 2), 9, 9, 7      # six blocks: seven phases


@pytest.mark.gpu
@pytest.mark.parametrize("path", [capi.EVALNET_PATH_AUTO, capi.EVALNET_PATH_STREAMING], ids=["resident", "streaming"])
@pytest.mark.parametrize("kind", ["othello", "noblocks", "go9"])
def test_evalnet_update_reaches_a_captured_graph(kind, path):
    """A graph captured with network A and replayed after update(B) computes B: the same bits as a fresh evaluator of B.
    A and B scale their weights by different powers of two, so a replay that kept A's scales would be off by a power
    of two in those layers."""
    a, b, rows, cols, phases = _update_nets(kind)
    assert layer_shifts(a) != layer_shifts(b)
    x = boards(a, 300, rows, cols, seed=6)
    want_l, want_v, amax = fp64_forward(b, x)
    xg = x.cuda()
    ev = EvalNet(a, device=0, rows=rows, cols=cols)
    ev.set_path(path)
    assert ev.phases == (phases if path == capi.EVALNET_PATH_AUTO else 0)
    logits = torch.empty(300, want_l.shape[1], device="cuda")
    value = torch.empty(300, device="cuda")
    stream = lambda: torch.cuda.current_stream().cuda_stream
    ev.forward_ptr(xg.data_ptr(), 300, logits.data_ptr(), value.data_ptr(), stream())     # sizes the buffers
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ev.forward_ptr(xg.data_ptr(), 300, logits.data_ptr(), value.data_ptr(), stream())
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
    fresh.set_path(path)
    l_b, v_b = fresh(xg)
    fresh.status()
    assert (l_a - l_b).abs().max().item() > 1e-3              # A and B are different networks
    assert torch.equal(logits, l_b) and torch.equal(value, v_b.reshape(-1))
    assert_close(logits, value, want_l, want_v, amax)
    del graph
    ev.close()
    fresh.close()


@pytest.mark.gpu
def test_selfplay_after_update_matches_a_fresh_evaluator():
    """Self-play through an attached evaluator keeps its CUDA graph across run_iteration calls.  After update(B) the next
    iteration must produce the samples of a fresh engine with a fresh evaluator of B (same seed, same games)."""
    from sprl_b200 import selfplay as SP
    a, b, _, _, _ = _update_nets("othello")
    assert layer_shifts(a) != layer_shifts(b)
    kw = dict(seed=7, sims=48, max_batch=8, max_queue=4, num_slots=64, max_games=64)
    n = 64
    ev = EvalNet(a, device=0)
    with SP.Engine(capi.GAME_OTHELLO, capi.EVAL_EXTERNAL, **kw) as eng:
        eng.attach_evalnet(ev, use_cuda_graph=True)
        eng.run_iteration(n, first_game=0)
        ev.update(b)
        got = eng.run_iteration(n, first_game=n)
    ev.status()
    ev.close()
    ev_b = EvalNet(b, device=0)
    with SP.Engine(capi.GAME_OTHELLO, capi.EVAL_EXTERNAL, **kw) as eng:
        eng.attach_evalnet(ev_b, use_cuda_graph=True)
        want = eng.run_iteration(n, first_game=n)
    ev_b.status()
    ev_b.close()
    assert got[0].shape[0] > n * 8 * 20
    for g, w in zip(got, want):
        assert np.array_equal(g, w)
