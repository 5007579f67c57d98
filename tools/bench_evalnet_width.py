"""Evaluator forward at tower widths 64 and 128: the library's tcgen05 kernels against LibTorch fp32 on the same module.

    python tools/bench_evalnet_width.py [--out FILE]

Prints the GPU's name, power limit and SM clock, then one JSON line per network:
  * Othello 2 blocks x 64 / x 128 channels at 61,952 rows (bench.py's mean leaf batch), Go 9x9 6 x 64 / x 128 at 32,768;
  * `lib_ms`: sprl_evalnet_forward (AUTO path: the resident kernel for 64 channels, the streaming one for 128), CUDA
    events over >= 200 launches after warm-up;
  * `torch_ms`: the traced module through LibTorch, fp32 with cuDNN and TF32 off (ATen's own convolution), and
    `torch_cudnn_ms`: the same with cuDNN on (still fp32, TF32 off) -- the LibTorch fallback the C++ veneer takes for a
    network the library refuses; fewer launches (each takes up to seconds), after one warm-up;
  * `lib_err` / `torch_err`: max |d logit| and |d value| against the fp64 CPU forward on a 128-row sample, and `A`, the
    largest |BatchNorm output| of that sample (the library's error bound is 2e-6 * max(1, A));
  * `mflop_per_leaf` from the shapes, and the rates both give.
Last, a short self-play leg (Othello, 400 sims/move, batch 8, queue 4, 16,384 games) with a 2x64 and a 2x128 evaluator
attached through Engine.attach_evalnet and replayed as one CUDA graph, as bench.py does: sims/s of each.

Every number is measured in this one process on one GPU; the inputs are seeded random boards (0/1 planes) and the
networks random-init with randomized BatchNorm."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

from sprl_b200 import capi  # noqa: E402
from sprl_b200 import selfplay as SP  # noqa: E402
from sprl_b200.evalnet import EvalNet  # noqa: E402
from sprl_b200.network import BasicGridNetwork, trace_network  # noqa: E402

CONFIGS = [  # name, rows, cols, planes, blocks, channels, actions, batch
    ("othello_2x64", 8, 8, 3, 2, 64, 65, 61952),
    ("othello_2x128", 8, 8, 3, 2, 128, 65, 61952),
    ("go9_6x64", 9, 9, 17, 6, 64, 82, 32768),
    ("go9_6x128", 9, 9, 17, 6, 128, 82, 32768),
]


def gpu_state():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), f"--query-gpu={q}", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), (x.strip() for x in out.split(","))))
    except Exception as e:          # the timings stand without it; say so
        return {"nvidia-smi": f"unavailable: {e}"}


def flop_per_leaf(rows, cols, planes, blocks, ch, actions):
    cells = rows * cols
    return 2 * (ch * 9 * planes * cells + 2 * blocks * ch * ch * 9 * cells + 3 * ch * cells + 2 * cells * actions + cells * ch + ch)


def make(rows, cols, planes, blocks, ch, actions, seed):
    from test_evalnet import randomized
    torch.manual_seed(seed)
    return randomized(BasicGridNetwork(rows, cols, actions, (planes - 1) // 2, blocks, ch).eval(), seed + 100)


def fp64(net, x):
    from test_evalnet_edges import fp64_forward
    return fp64_forward(net, x)


def time_ms(fn, launches, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(launches):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / launches


def torch_ms(module, x, budget_s):
    """One warm-up, then launches until `budget_s` seconds (at least 2, at most 20)."""
    with torch.no_grad():
        module(x)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        module(x)
        torch.cuda.synchronize()
        one = time.perf_counter() - t0
        n = max(2, min(20, int(budget_s / max(one, 1e-6))))
        return time_ms(lambda: module(x), n, 0), n


def forward_leg(cfg, args):
    name, rows, cols, planes, blocks, ch, actions, batch = cfg
    batch = max(256, int(batch * args.scale))
    net = make(rows, cols, planes, blocks, ch, actions, seed=ch + blocks)
    g = torch.Generator().manual_seed(1)
    x = (torch.rand(batch, planes, rows, cols, generator=g) > 0.5).float()
    sample = torch.randperm(batch, generator=g)[:128]
    want_l, want_v, a = fp64(net, x[sample])
    xg = x.cuda()
    ev = EvalNet(net, device=0, rows=rows, cols=cols)
    logits = torch.empty(batch, actions, device="cuda")
    value = torch.empty(batch, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    lib = lambda: ev.forward_ptr(xg.data_ptr(), batch, logits.data_ptr(), value.data_ptr(), stream)
    lib_ms = time_ms(lib, args.launches, 20)
    clocks = gpu_state()
    ev.status()
    idx = sample.cuda()
    lib_err = [(logits[idx].cpu().double() - want_l).abs().max().item(), (value[idx].cpu().double() - want_v.reshape(-1)).abs().max().item()]
    phases = ev.phases
    ev.close()

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    res = {}
    for cudnn in (False, True):
        # a trace records the cuDNN switch into every convolution it contains: trace under the setting it is timed with
        torch.backends.cudnn.enabled = cudnn
        module = trace_network(net, torch.device("cuda", 0))
        ms, n = torch_ms(module, xg, args.torch_seconds)
        with torch.no_grad():
            tl, tv = module(xg[idx])
        res[cudnn] = (ms, n, [(tl.cpu().double() - want_l).abs().max().item(), (tv.cpu().double() - want_v).abs().max().item()])
        del module
    torch.backends.cudnn.enabled = True
    del xg
    torch.cuda.empty_cache()
    mflop = flop_per_leaf(rows, cols, planes, blocks, ch, actions) / 1e6
    return {
        "net": name, "rows": batch, "channels": ch, "blocks": blocks, "mflop_per_leaf": round(mflop, 1),
        "lib_path": "resident" if phases else "streaming", "lib_ms": round(lib_ms, 3), "lib_launches": args.launches,
        "lib_tflops_fp32_equiv": round(mflop * 1e6 * batch / (lib_ms * 1e-3) / 1e12, 1),
        "torch_ms": round(res[False][0], 2), "torch_launches": res[False][1],
        "torch_cudnn_ms": round(res[True][0], 2), "torch_cudnn_launches": res[True][1],
        "speedup_vs_torch": round(res[False][0] / lib_ms, 1), "speedup_vs_torch_cudnn": round(res[True][0] / lib_ms, 2),
        "lib_err": [float(f"{e:.3g}") for e in lib_err], "torch_err": [float(f"{e:.3g}") for e in res[False][2]],
        "torch_cudnn_err": [float(f"{e:.3g}") for e in res[True][2]], "A": round(a, 2),
        "sm_clock_after_lib": clocks.get("clocks.sm"),
    }


def selfplay_leg(ch, args):
    """bench.py's steady state (400 sims/move, batch 8, queue 4, continuous play in `slots` games) for a 2 x ch network."""
    net = make(8, 8, 3, 2, ch, 65, seed=ch + 7)
    ev = EvalNet(net, device=0)
    slots = args.slots
    eng = SP.Engine(capi.GAME_OTHELLO, capi.EVAL_EXTERNAL, device=0, seed=0, sims=400, max_batch=8, max_queue=4,
                    dir_eps=0.25, dir_alpha=0.3, num_slots=slots, max_games=slots * 24)
    eng.attach_evalnet(ev, use_cuda_graph=True)
    eng.set_stream(torch.cuda.current_stream().cuda_stream)
    eng.begin_iteration(0, slots * 24)
    eng._capture()
    graph = eng._nn["graph"]

    def step():
        for _ in range(args.rounds):
            graph.replay()

    step()
    torch.cuda.synchronize()
    eng.reset_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.sp_steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    st = eng.stats()
    clocks = gpu_state()
    playing, failed = eng.poll()
    eng.close()
    ev.status()
    ev.close()
    assert failed == 0, failed
    return {"selfplay": f"othello_2x{ch}", "sims_per_s": round(st["sims"] / (ms / 1e3), 1), "window_ms": round(ms, 1),
            "rounds": args.rounds * args.sp_steps, "games_finished": int(st["games"]), "slots": slots,
            "sm_clock_after": clocks.get("clocks.sm")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=200, help="timed library forwards per network")
    ap.add_argument("--torch-seconds", type=float, default=3.0, help="time budget of each LibTorch measurement")
    ap.add_argument("--scale", type=float, default=1.0, help="batch sizes x this (rehearsals only)")
    ap.add_argument("--slots", type=int, default=16384)
    ap.add_argument("--rounds", type=int, default=256, help="search rounds per self-play step")
    ap.add_argument("--sp-steps", type=int, default=2, help="timed self-play steps (after one warm-up step)")
    ap.add_argument("--out", help="also write the lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_evalnet_width: no CUDA device")
    lines = [json.dumps({"gpu": gpu_state(), "torch": torch.__version__, "launches": args.launches, "scale": args.scale})]
    print(lines[-1], flush=True)
    for cfg in CONFIGS:
        lines.append(json.dumps(forward_leg(cfg, args)))
        print(lines[-1], flush=True)
    for ch in (64, 128):
        lines.append(json.dumps(selfplay_leg(ch, args)))
        print(lines[-1], flush=True)
    lines.append(json.dumps({"gpu_after": gpu_state()}))
    print(lines[-1], flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
