#!/usr/bin/env python
"""Benchmark of the self-play hot path (BASELINE.json: Othello 8x8, 400 sims/move,
8-fold symmetrised, virtual-loss leaf batching 8/4).

  python bench.py --gpus N --steps K --warmup W            our arm (one process per GPU)
  python bench.py --impl reference --gpus N --steps K ...   the reference's CPU worker on the host cores

A *step* of our arm is `--rounds` search rounds of `--slots` concurrent games in
continuous play (a slot starts its next game when one ends): every round is one
search launch over all trees (select / expand / backup / re-root), one forward of the
reference's network (same architecture and weights as the traced module; run by the
library's tcgen05 kernel with fp32-level split-fp16 arithmetic, or by LibTorch/cuDNN fp32
with --evaluator libtorch) on the leaf batch those trees produced, and the application
of its outputs in the next launch.  `value` is MCTS simulations per second,
whole job, from device counters over exactly K timed steps; moves/s etc. ride along.
`e2e` is the same metric through the public API with host buffers: each e2e step loads
the network weights from pinned host memory, plays `--e2e-games` full games from the
start position to the end, and copies the sample arrays back to the host.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SIMS, MAX_BATCH, MAX_QUEUE, EPS, ALPHA = 400, 8, 4, 0.25, 0.3
WORKLOAD = "othello8x8_selfplay_400sims_batch8_queue4_d4sym_net2x64_fp32"
NET_FLOP_PER_LEAF = 2 * (64 * 27 * 64 + 4 * 64 * 64 * 9 * 64 + 3 * 64 * 64 + 128 * 65 + 64 * 64 + 64)   # 19.1 MFLOP (SURVEY 8d)
NET_KIND, GAME_NAME, BOARD, PLANES, ACTIONS, METRIC, MAX_PLIES = "othello", "GAME_OTHELLO", (8, 8), 3, 65, "othello_selfplay_mcts_sims_per_sec", 66


def net_flop_per_leaf(rows, cols, planes, blocks, actions, ch=64):
    cells = rows * cols
    return 2 * (ch * 9 * planes * cells + 2 * blocks * ch * ch * 9 * cells + 3 * ch * cells + 2 * cells * actions + cells * ch + ch)


def select_workload(name):
    """BASELINE.json's headline configuration (default) or config 5 (Go 9x9: GoWorker.cpp:12-27 constants -- alpha 0.2,
    batch 16 / queue 8 -- with 400 sims/move, the reference's 6-block network shape, subtree reuse and Dirichlet noise on)."""
    global SIMS, MAX_BATCH, MAX_QUEUE, EPS, ALPHA, WORKLOAD, NET_FLOP_PER_LEAF, NET_KIND, GAME_NAME, BOARD, PLANES, ACTIONS, METRIC, MAX_PLIES
    if name == "othello":
        return
    if name != "go9":
        raise SystemExit(f"unknown workload {name}")
    SIMS, MAX_BATCH, MAX_QUEUE, EPS, ALPHA = 400, 16, 8, 0.25, 0.2
    WORKLOAD = "go9x9_selfplay_400sims_batch16_queue8_d4sym_net6x64_fp32_komi7.5"
    NET_KIND, GAME_NAME, BOARD, PLANES, ACTIONS, METRIC, MAX_PLIES = "go9", "GAME_GO9", (9, 9), 17, 82, "go9_selfplay_mcts_sims_per_sec", 163
    NET_FLOP_PER_LEAF = net_flop_per_leaf(9, 9, 17, 6, 82)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="othello", choices=["othello", "go9"], help="othello = BASELINE.json's headline configuration; go9 = its config 5")
    ap.add_argument("--slots", type=int, default=16384, help="concurrent games per GPU")
    ap.add_argument("--rounds", type=int, default=256, help="search rounds per step")
    ap.add_argument("--e2e-games", type=int, default=16384, help="games per e2e step per GPU")
    ap.add_argument("--e2e-slots", type=int, default=16384, help="concurrent games of the e2e engine (fewer than games: slots refill, finished games stream out)")
    ap.add_argument("--e2e-no-stream", action="store_true", help="collect the samples at the end into pageable memory (round-1 behaviour)")
    ap.add_argument("--e2e-steps", type=int, default=1)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--evaluator", default="evalnet", choices=["evalnet", "libtorch"],
                    help="network forward: the library's tcgen05 kernel (default) or the traced module through LibTorch/cuDNN")
    ap.add_argument("--evaluator-precision", default="fp32", choices=["fp32", "fp16"],
                    help="fp32 = the reference's precision (split fp16 x3, the headline); fp16 = the opt-in single-pass mode of the library "
                         "evaluator: NOT the reference's precision, printed as a different metric")
    ap.add_argument("--ref-seconds", type=float, default=20.0, help="timed window of the cpu_baseline leg (one core), seconds")
    ap.add_argument("--ref-window", type=float, default=60.0, help="timed window of --impl reference (every core), seconds")
    ap.add_argument("--ref-test-sims", type=int, default=0, help="smoke tests only: sims/move of the reference worker")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what they computed as DIR/<name>.npy "
                    "(float32, at most 60 MB; rank 0), to compare two builds output for output")
    args = ap.parse_args()
    select_workload(args.workload)
    if args.workload == "go9":          # smaller defaults: a Go 9x9 tree slab is 6.5 MB, a sample row 5.8 KB
        if args.slots == 16384:
            args.slots = 4096
        if args.e2e_games == 16384:
            args.e2e_games, args.e2e_slots = 1024, 1024
        args.no_cpu_baseline = True     # the reference arm exists for the headline workload (and Connect Four, tools/bench_configs.py)
    return args


# ------------------------------------------------------------------------ clocks sampler
class ClockSampler:
    """Samples nvidia-smi clocks and throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.limit")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) >= 7:
                self.rows.append(parts)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, watts, limit = [], None, set(), [], None
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except ValueError:
                continue
            try:
                watts.append(float(r[2])); limit = float(r[7]) if len(r) > 7 else None
            except ValueError:
                pass
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        watts.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
                "power_w": watts[len(watts) // 2] if watts else None, "power_limit_w": limit}


def bytes_per_sim(D, L, e, planes_cells=192, A=65):
    """Algorithmic HBM bytes of one simulation (SURVEY.md 8d): D select levels that each read a
    16 B node header + 16 B board pair + 4 B link and 12 B of P/W/N per legal child, the leaf's
    virtual loss, one step + new node, the evaluator-side traffic of the fraction e of
    simulations that need an evaluation, and the backup."""
    return D * (16 + 12 * L + 4 + 16) + 16 + (16 + 16 + 8 + 16) + e * (4 * planes_cells + 4 * (A + 1) + 16 * L) + (D + 1) * 8


# ------------------------------------------------------------------------------ our arm
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from sprl_b200 import capi
    from sprl_b200 import selfplay as SP
    from sprl_b200.network import make_network, trace_network, num_parameters

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus > 1 and world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} needs torchrun with {args.gpus} ranks (WORLD_SIZE={world})")
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    torch.backends.cudnn.allow_tf32 = False          # the reference evaluates in fp32
    torch.backends.cuda.matmul.allow_tf32 = False

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- the evaluator: the reference's network shape, random init, traced as the controller does
    net = make_network(NET_KIND, seed=0)
    n_params = num_parameters(net)
    module = trace_network(net, dev)
    flat_params = [p for p in module.parameters()] + [b for b in module.buffers()]
    weight_bytes = sum(t.numel() * t.element_size() for t in flat_params)

    from sprl_b200.evalnet import EvalNet
    evalnet = EvalNet(net, device=local, rows=BOARD[0], cols=BOARD[1]) if args.evaluator == "evalnet" else None
    fp16_eval = args.evaluator_precision == "fp16"
    if fp16_eval:
        if evalnet is None:
            raise SystemExit("--evaluator-precision fp16 needs --evaluator evalnet")
        evalnet.set_precision(capi.EVALNET_PRECISION_FP16)

    def attach(engine):
        if evalnet is not None:
            engine.attach_evalnet(evalnet, use_cuda_graph=not args.no_graph)
        else:
            engine.attach_network(module, use_cuda_graph=not args.no_graph)

    def broadcast_weights(generation):
        """New generation: rank 0 draws fresh random-init weights, NCCL broadcasts the flat
        parameter + buffer vector (SURVEY.md 8e); every rank updates its module in place."""
        if rank == 0:
            fresh = make_network(NET_KIND, seed=1000 + generation)
            src = [p for p in fresh.parameters()] + [b for b in fresh.buffers()]
            flat = torch.cat([t.detach().reshape(-1).float() for t in src]).to(dev)
        else:
            flat = torch.empty(sum(t.numel() for t in flat_params), device=dev)
        if world > 1:
            dist.broadcast(flat, 0)
        at = 0
        with torch.no_grad():
            for t in flat_params:
                n = t.numel()
                t.copy_(flat[at:at + n].reshape(t.shape).to(t.dtype))
                at += n
        if evalnet is not None:
            evalnet.update(module)          # fold BN, split hi/lo, re-pack in place (device addresses stay valid)

    # ---- evaluator accuracy on this box: ours vs the fp64 forward of the same network (CPU)
    eval_err = None
    if evalnet is not None and rank == 0:
        xs = (torch.rand(512, PLANES, *BOARD) > 0.5).float()
        with torch.no_grad():
            want = make_network(NET_KIND, seed=0).double()(xs.double())[0]
            got = evalnet(xs.to(dev))[0].cpu().double()
        eval_err = float((got - want).abs().max())
        assert eval_err < (2e-2 if fp16_eval else 1e-4), f"evaluator deviates from the fp64 forward by {eval_err}"

    # ---- steady-state engine: continuous play, games sharded by id % world
    games_cap = args.slots * 24
    eng = SP.Engine(getattr(capi, GAME_NAME), capi.EVAL_EXTERNAL, device=local, seed=0, sims=SIMS, max_batch=MAX_BATCH,
                    max_queue=MAX_QUEUE, dir_eps=EPS, dir_alpha=ALPHA, num_slots=args.slots, max_games=games_cap)
    eng.set_game_stride(world)
    attach(eng)
    broadcast_weights(0)
    with torch.cuda.device(dev):
        eng.set_stream(torch.cuda.current_stream(dev).cuda_stream)
        eng.begin_iteration(rank, games_cap)
        if not args.no_graph:
            eng._capture()
        graph = eng._nn["graph"]

        def step():
            for _ in range(args.rounds):
                if graph is not None:
                    graph.replay()
                else:
                    eng._round_with_network()

        for _ in range(args.warmup):
            step()
        barrier()
        eng.reset_stats()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(args.steps):
            step()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        clocks = sampler.stop() if rank == 0 else None
        st = eng.stats()
        playing, failed = eng.poll()
        assert failed == 0 and playing == args.slots, (playing, failed)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, eng)

        # ---- roofline leg: the search launch alone, timed with events on its stream
        n_probe = 64
        eng.reset_stats()
        evs = [tuple(torch.cuda.Event(enable_timing=True) for _ in range(3)) for _ in range(n_probe)]
        for a, b, c in evs:
            a.record()
            eng.round()
            b.record()
            eng._forward()
            c.record()
        torch.cuda.synchronize(dev)
        k_ms = sum(a.elapsed_time(b) for a, b, c in evs) / n_probe
        nn_ms = sum(b.elapsed_time(c) for a, b, c in evs) / n_probe     # the forward of exactly the leaves each launch queued
        pst = eng.stats()
    eng.close()

    # totals over ranks
    tot = torch.tensor([st["sims"], st["moves"], st["evals"], st["games"], st["leaves_duplicate"]], dtype=torch.float64, device=dev)
    tmax = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    sims, moves, evals, games, dups = [float(x) for x in tot.tolist()]
    ms = float(tmax.item())
    value = sims / (ms / 1e3)

    D = pst["depth_sum"] / max(1, pst["sims"])
    L = pst["legal_sum"] / max(1, pst["nodes_visited"])
    ef = pst["evals"] / max(1, pst["sims"])
    bps = bytes_per_sim(D, L, ef, planes_cells=PLANES * BOARD[0] * BOARD[1], A=ACTIONS)
    sims_per_launch = pst["sims"] / n_probe
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
    # DRAM bytes per launch from the committed `ncu --set full` captures (profiles/ncu_traffic.json), used only when the
    # capture was taken at this run's size
    ncu_traffic = {}
    try:
        ncu_traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except Exception:
        pass

    def traffic_of(kernel):
        t = ncu_traffic.get(kernel)
        return t["dram_bytes_per_launch"] if t and t.get("slots") == args.slots else None
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = bps * sims_per_launch / (k_ms / 1e3) / 1e9
    roofline_search = {"kernel": "k_round<%s>" % ("Othello" if NET_KIND == "othello" else "Go<9>"), "bound": "hbm", "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s",
                       "frac": round(achieved / peak, 5), "traffic": traffic_of("k_round"), "peak_source": peak_src,
                       "algorithmic_bytes_per_launch": round(bps * sims_per_launch, 1),
                       "launch_ms": round(k_ms, 4), "sims_per_launch": round(sims_per_launch, 1), "bytes_per_sim": round(bps, 1),
                       "select_depth": round(D, 3), "legal_per_node": round(L, 3), "evals_per_sim": round(ef, 4),
                       "sampled_launches": n_probe, "share_of_round": round(k_ms / (k_ms + nn_ms), 4),
                       "probe_note": "the two legs are timed un-graphed, with CUDA events between the launches of 64 extra rounds: their "
                                     "sum runs 2-3 % above ms_per_step / rounds_per_step (event records and launch gaps the graph does not have)"}
    batch_rows = args.slots * MAX_QUEUE
    if evalnet is not None:
        # dominant kernel of the step: the evaluator's forward over the rows in use (the leaves the launch queued)
        tpeak = float(peaks.get("bf16_tflops_sustained", 1400.0))
        batch_rows = (pst["evals"] - pst["leaves_duplicate"]) / n_probe     # a leaf queued twice in a batch (quirk Q4) takes one row
        tf = batch_rows * NET_FLOP_PER_LEAF / (nn_ms / 1e3) / 1e12
        roofline = {"kernel": "k_evalnet_resident" if evalnet.phases else "k_evalnet", "launches_per_forward": max(1, evalnet.phases), "bound": "tensor", "achieved": round(tf, 2), "peak": tpeak, "unit": "TFLOP/s",
                    "frac": round(tf / tpeak, 5), "traffic": traffic_of("k_evalnet_resident" if evalnet.phases else "k_evalnet"), "peak_source": peak_src + " bf16 sustained",
                    "launch_ms": round(nn_ms, 4), "leaves_per_launch": round(batch_rows, 1), "leaf_batch_capacity": args.slots * MAX_QUEUE, "flop_per_leaf": NET_FLOP_PER_LEAF,
                    "note": "launch_ms = one forward = the conv tower (launches_per_forward launches of the kernel) + k_heads; "
                            "achieved = algorithmic fp32 FLOPs / time against the measured bf16 peak; the kernel issues 3x that "
                            "as fp16 MMAs (hi/lo split of both operands: hi*hi + hi*lo + lo*hi, fp32 accumulate) to keep fp32-level "
                            "accuracy, so issued_frac is the tensor-pipe utilisation",
                    "issued_tflops": round((1 if fp16_eval else 3) * tf, 1), "issued_frac": round((1 if fp16_eval else 3) * tf / tpeak, 4),
                    "share_of_round": round(nn_ms / (k_ms + nn_ms), 4)}
    else:
        roofline = dict(roofline_search, network_forward_ms=round(nn_ms, 4))
    result = {
        "metric": METRIC + ("_fp16_evaluator" if fp16_eval else ""), "value": round(value, 1), "unit": "sims/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": ("fp16 network (single pass, fp32 accumulate; NOT the reference's fp32: a different metric, never the headline), tree statistics fp32" if fp16_eval else
                  "fp32 (tree statistics fp32; network split-fp16 x3 on tcgen05, fp32 accumulate, max |dlogit| ~1e-7 vs fp64)") if evalnet is not None else "fp32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD + ("_FP16EVAL" if fp16_eval else ""), "sims_per_move": SIMS, "max_batch": MAX_BATCH, "max_queue": MAX_QUEUE,
                   "slots_per_gpu": args.slots, "rounds_per_step": args.rounds, "network_params": n_params,
                   "sharding": "game_id % world, no data collective; NCCL broadcast of weights per generation",
                   "l2": "working set (tree slabs %.1f GB + leaf batch) exceeds the 126 MB L2" % (st["device_bytes"] / 1e9),
                   "cuda_graph": not args.no_graph, "evaluator": args.evaluator,
                   "evaluator_max_abs_logit_err_vs_fp64": eval_err},
        "moves_per_sec": round(moves / (ms / 1e3), 1), "evals_per_sec": round(evals / (ms / 1e3), 1),
        "samples_per_sec": round(8 * moves / (ms / 1e3), 1), "games_finished": int(games),
        "evals_per_sim": round(evals / max(1.0, sims), 4), "eval_rows_per_sim": round((evals - dups) / max(1.0, sims), 4),
        "duplicate_leaf_fraction": round(dups / max(1.0, evals), 4),
        # per round: k_round, k_flip, the conv tower (one k_evalnet_resident launch per residual block, or one k_evalnet), k_heads
        "gpu_launches": int(args.steps * args.rounds * world * ((2 + max(1, evalnet.phases) + 1) if evalnet is not None else 2)),
        "roofline": roofline, "roofline_search": roofline_search, "clocks": clocks,
    }

    if not args.no_e2e:
        e2e = run_e2e(args, local, module, flat_params, weight_bytes, barrier, evalnet, rank, world)     # every rank, on its own shard
        agg = torch.tensor([e2e.pop("_sims"), e2e.pop("_moves")], dtype=torch.float64, device=dev)
        tm = torch.tensor([e2e.pop("_ms")], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(agg)
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        e2e["value"] = round(float(agg[0]) / (float(tm) / 1e3), 1)
        e2e["moves_per_sec"] = round(float(agg[1]) / (float(tm) / 1e3), 1)
        e2e["ms_per_step"] = round(float(tm) / args.e2e_steps, 1)
        result["e2e"] = e2e
    if rank == 0 and world == 1 and not args.no_cpu_baseline:      # the reported CPU baseline: rank 0 at N = 1 only
        result["cpu_baseline"] = cpu_baseline(args, threads=1, seconds=args.ref_seconds)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        emit(result)


DUMP_BYTES_PER_GROUP = 30 * 10**6      # two groups of arrays: --dump-outputs writes at most 60 MB


def dump_outputs(out_dir, eng):
    """--dump-outputs: what the timed steps computed, as float32 .npy files, for comparing two builds on identical inputs.
    eval_inputs / eval_logits / eval_values: the leaf batch of the last round and the network's outputs for it.  The
    search kernel hands out batch rows in no fixed order, so the rows are sorted by their bytes.
    samples_states / samples_distributions / samples_outcomes: the sample rows of every game finished so far, in the
    reference's order (games, moves, symmetries).  A group larger than DUMP_BYTES_PER_GROUP keeps a fixed, seeded
    sample of its rows, in order."""
    import numpy as np
    import torch
    nn = eng._nn
    torch.cuda.synchronize(nn["dev"])

    def keep(n, row_bytes):
        cap = DUMP_BYTES_PER_GROUP // row_bytes
        return np.arange(n) if n <= cap else np.sort(np.random.default_rng(0).choice(n, cap, replace=False))

    class Counter:                 # __cuda_array_interface__ over the device count of rows the last launch queued
        __cuda_array_interface__ = dict(shape=(1,), typestr="<i4", data=(nn["rows"], False), version=3, strides=None, stream=None)
    rows = int(torch.as_tensor(Counter(), device=nn["dev"]).item())
    x = nn["inp"][:rows].reshape(rows, -1).cpu().numpy()
    logits = nn["logits"][:rows].cpu().numpy()
    flat = np.ascontiguousarray(np.concatenate([x, logits, nn["value"][:rows].cpu().numpy().reshape(rows, 1)], 1))
    flat = flat[np.argsort(flat.view(np.dtype((np.void, flat.shape[1] * 4))).ravel(), kind="stable")]
    flat = flat[keep(rows, flat.shape[1] * 4)]
    P, A = x.shape[1], logits.shape[1]
    out = {"eval_inputs": flat[:, :P].reshape((-1,) + tuple(nn["inp"].shape[1:])), "eval_logits": flat[:, P:P + A],
           "eval_values": flat[:, P + A]}

    states, dists, outcomes = eng.collect_samples_device()
    idx = torch.from_numpy(keep(states.shape[0], 4 * (int(np.prod(states.shape[1:])) + dists.shape[1] + 1))).to(states.device)
    out.update(samples_states=states[idx], samples_distributions=dists[idx], samples_outcomes=outcomes[idx])
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        a = a.cpu().numpy() if isinstance(a, torch.Tensor) else a
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, np.float32))


def run_e2e(args, local, module, flat_params, weight_bytes, barrier, evalnet, rank=0, world=1):
    """Full generations through the public API with host buffers.  Every e2e step is one generation as SURVEY.md 8(d)
    config 4 / 8(e) describe it: rank 0 holds the new network's weights in host memory and broadcasts the flat parameter +
    buffer vector (NCCL at N > 1), every rank folds / packs / uploads them, plays its shard of the generation's games
    (ids rank, rank + world, ...) start to finish, streams the samples to page-locked host arrays, and the ranks
    all-gather their sample counts (the row ranges of the generation's arrays)."""
    import torch.distributed as dist
    from sprl_b200 import shard
    import numpy as np
    import torch
    from sprl_b200 import capi
    from sprl_b200 import selfplay as SP
    dev = torch.device("cuda", local)
    host_weights = [t.detach().cpu().pin_memory() for t in flat_params]
    G = args.e2e_games
    with SP.Engine(getattr(capi, GAME_NAME), capi.EVAL_EXTERNAL, device=local, seed=1, sims=SIMS, max_batch=MAX_BATCH,
                   max_queue=MAX_QUEUE, dir_eps=EPS, dir_alpha=ALPHA, num_slots=min(G, args.e2e_slots), max_games=G) as eng:
        if not args.e2e_no_stream:
            # page-locked sample arrays, registered once (as a worker would keep them across iterations): finished games
            # are embedded and copied while the others play; an Othello game has at most 60 placements + passes
            eng.stream_samples(G * 8 * MAX_PLIES)
        if evalnet is not None:
            eng.attach_evalnet(evalnet, use_cuda_graph=not args.no_graph)
            host_state = {k: v.detach().cpu().numpy() for k, v in module.state_dict().items()}
            weight_bytes = evalnet.info()["upload_bytes"]
        else:
            eng.attach_network(module, use_cuda_graph=not args.no_graph)

        eng.set_game_stride(world)
        names = [k for k, _ in module.state_dict().items()]
        shapes = [tuple(v.shape) for _, v in module.state_dict().items()]
        flat_host = torch.cat([v.detach().reshape(-1).float().cpu() for _, v in module.state_dict().items()]).pin_memory()
        counts = []

        def one(first):
            if world > 1:
                # the generation's weights: host (rank 0) -> device -> NCCL broadcast -> every rank's host copy for the packer
                flat = flat_host.to(dev, non_blocking=True) if rank == 0 else torch.empty(flat_host.numel(), device=dev)
                dist.broadcast(flat, 0)
                flat_cpu = flat.cpu()
            else:
                flat_cpu = flat_host
            if evalnet is not None:
                at, state = 0, {}
                for k, shp in zip(names, shapes):
                    n = int(np.prod(shp)) if shp else 1
                    state[k] = flat_cpu[at:at + n].reshape(shp).numpy()
                    at += n
                evalnet.update(state)               # host weights -> folded / packed -> device, inside the timed region
            else:
                with torch.no_grad():
                    for t, h in zip(flat_params, host_weights):
                        t.copy_(h, non_blocking=True)
            out = eng.run_iteration(G, first_game=first * world + rank)
            counts.append(shard.gather_sample_counts(out[0].shape[0], device=dev))     # all-gather of one int64 per rank
            return out

        # warm-up: a short iteration with the same engine (graph capture, cuDNN autotune)
        one(0) if args.e2e_steps > 1 else eng.run_iteration(min(G, 64), first_game=0)
        barrier()
        eng.reset_stats()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d2h = 0
        e0.record()
        for i in range(args.e2e_steps):
            states, dists, outcomes = one(10_000 * (i + 1))
            d2h += states.nbytes + dists.nbytes + outcomes.nbytes
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        st = eng.stats()
        eng_info = eng.stream_info()
    return {"value": None, "unit": "sims/s", "h2d_bytes_per_step": int(weight_bytes),
            "d2h_bytes_per_step": int(d2h / args.e2e_steps), "moves_per_sec": None,
            "games_per_step_per_gpu": G, "slots_per_gpu": min(G, args.e2e_slots), "steps": args.e2e_steps, "ms_per_step": None,
            "streamed_chunks_while_playing": None if args.e2e_no_stream else eng_info["chunks_while_playing"],
            "collectives_per_step": "none (1 rank)" if world == 1 else f"NCCL broadcast of {flat_host.numel() * 4} weight bytes + all-gather of {world} sample counts",
            "sample_rows_per_rank_last_step": counts[-1] if counts else None,
            "note": "public API (Engine.run_iteration) with host buffers: weights from host memory (fold + pack + H2D), full games "
                    "start to finish incl. the tail where few games are left, every sample row D2H into page-locked host arrays "
                    "(finished games stream out while the others play)",
            "_sims": float(st["sims"]), "_moves": float(st["moves"]), "_ms": float(ms)}


# ----------------------------------------------------------------- reference / CPU baseline
def ref_worker_path():
    return os.path.join(ROOT, "oracle", "_ref", "ref_worker")


def traced_model_file():
    import torch
    from sprl_b200.network import make_network, trace_network
    path = os.path.join(tempfile.gettempdir(), f"sprl_bench_othello_{os.getpid()}.pt")
    trace_network(make_network("othello", seed=0), "cpu").save(path)
    return path


def cpu_baseline(args, threads, seconds, game="othello"):
    """Times the reference's CPU worker path (oracle/_ref/ref_worker: unmodified reference sources + LibTorch on the
    CPU), `threads` single-threaded processes (one per host core, the reference's deployment model).  Protocol of
    BASELINE.md section 3: every process plays one discarded warm-up game, then full games through the reference's own
    SPRL::runIteration until `seconds` of wall time have passed (the game in progress is finished and counted)."""
    sims = args.ref_test_sims or SIMS
    if not os.path.exists(ref_worker_path()):
        r = cpu_baseline_port(sims, seconds)
    else:
        r = cpu_baseline_reference(threads, seconds, game, sims)
    if args.ref_test_sims:
        r["test_override"] = f"{sims} sims/move instead of {SIMS} (smoke test of the arm, not a measurement)"
    return r


def cpu_baseline_reference(threads, seconds, game, sims):
    model = traced_model_file()
    t0 = time.time()
    procs = [subprocess.Popen([ref_worker_path(), game, model, "0", str(100000 * (i + 1)), str(sims), str(MAX_BATCH), str(MAX_QUEUE),
                               str(EPS), str(ALPHA), str(seconds)], stdout=subprocess.PIPE, text=True) for i in range(threads)]
    outs = [json.loads(p.communicate()[0].strip().split("\n")[-1]) for p in procs]
    wall = time.time() - t0
    os.unlink(model)
    # every process has its own window (it ends at a game boundary): the aggregate is the sum of the per-process rates
    sims_s = sum(o["sims"] / o["seconds"] for o in outs)
    moves_s = sum(o["moves"] / o["seconds"] for o in outs)
    window = sum(o["seconds"] for o in outs) / len(outs)
    r = {"value": round(sims_s, 1), "unit": "sims/s", "cores": threads, "kind": "reference",
         "moves_per_sec": round(moves_s, 2), "per_core": round(sims_s / threads, 1), "window_seconds": round(window, 2),
         "games": sum(o["games"] for o in outs), "sims_per_move": round(sum(o["sims_per_move"] for o in outs) / len(outs), 2),
         "sample": f"{threads} process(es), each: one discarded warm-up game, then {min(o['games'] for o in outs)}-{max(o['games'] for o in outs)} full "
                   f"game(s) through the reference's runIteration in a {window:.1f} s window, {sims} sims/move, traced 2x64 net on CPU "
                   f"(LibTorch, 1 thread each); {wall:.1f} s wall in all",
         "cpu": cpu_model(), "host_cores": os.cpu_count()}
    return r


def cpu_baseline_port(sims, seconds):
    """Fallback when oracle/_ref was not built: the plain-C oracle port, one thread, full games at `sims` sims/move until
    `seconds` of wall time have passed (the game in progress is finished and counted)."""
    import numpy as np
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_py as O
    from sprl_b200.network import make_network
    torch.set_num_threads(1)
    net = make_network("othello", seed=0)

    def fn(x):
        with torch.no_grad():
            lg, v = net(torch.from_numpy(np.array(x)))
        return lg.numpy(), v.numpy().reshape(-1)

    def play(game):
        return O.selfplay(O.OG_OTHELLO, O.OE_CALLBACK, 0, game, 1, sims, MAX_BATCH, MAX_QUEUE, EPS, ALPHA, eval_fn=fn)

    play(0)                     # discarded warm-up game, as in the reference protocol
    games = moves = sims_done = 0
    t0 = time.time()
    while True:
        r = play(1 + games)
        games += 1
        moves += int(r["game_moves"].sum())
        sims_done += r["stats"]["total_traversals"]
        dt = time.time() - t0
        if dt >= seconds:
            break
    return {"value": round(sims_done / dt, 1), "unit": "sims/s", "cores": 1, "kind": "port",
            "moves_per_sec": round(moves / dt, 2), "window_seconds": round(dt, 2), "games": games,
            "sims_per_move": round(sims_done / moves, 2),
            "sample": f"one discarded warm-up game, then {games} full game(s) at {sims} sims/move through the C oracle with "
                      f"the network on CPU via a Python callback, one thread, in a {dt:.1f} s window"}


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation on all host cores of the box.  One measurement: every
    core plays a discarded warm-up game (the W warm-up steps), then full games in one window of --ref-window seconds (at
    least 60, BASELINE.md section 3); a step is 1/K of that window."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload != "othello":
        emit({"impl": "reference", "unavailable": "the reference arm times the headline workload (Othello); Go 9x9 needs the two-constant reference copy with LibTorch"})
        return
    threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else os.cpu_count()
    m = cpu_baseline(args, threads, args.ref_window)
    out = {"impl": "reference", "metric": "othello_selfplay_mcts_sims_per_sec", "value": m["value"], "unit": "sims/s",
           "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
           "ms_per_step": round(m.get("window_seconds", 0.0) * 1e3 / max(1, args.steps), 1),
           "config": {"workload": WORKLOAD, "sims_per_move": SIMS, "max_batch": MAX_BATCH, "max_queue": MAX_QUEUE},
           "moves_per_sec": m.get("moves_per_sec"),
           "cpu_baseline": {k: m[k] for k in m if k not in ("moves_per_sec",)},
           "e2e": {"value": m["value"], "unit": "sims/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(out)


def emit(obj):
    """The one JSON line of the contract, on the real stdout."""
    sys.stdout.flush()
    os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(obj), flush=True)


if __name__ == "__main__":
    # libraries (NCCL's version banner, torch) write to stdout: keep fd 1 clean for the JSON line
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
