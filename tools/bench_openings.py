"""Self-play throughput with and without opening lines, at bench.py's configuration (Othello, 400 sims/move, 8 / 4 leaf
batching, D4 symmetry, Dirichlet 0.25 / 0.3, the library evaluator with the 2x64 network, one CUDA graph per round).

    python tools/bench_openings.py [--lines 1000] [--plies 8] [--slots 16384] [--rounds 256] [--steps 3] [--warmup 3] [--repeats 2]

Engines without and with a table of `--lines` lines of `--plies` plies each (prefixes of random play-outs) are timed in
alternation, each over `--steps` steps of `--rounds` graph replays after `--warmup` steps.  Prints one JSON line per
timed engine (sims/s, searched moves, games) and one summary line with the card's name and power limit."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from sprl_b200 import capi  # noqa: E402
from sprl_b200 import selfplay as SP  # noqa: E402
from sprl_b200.evalnet import EvalNet  # noqa: E402
from sprl_b200.network import make_network  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def run(args, lines, net):
    dev = torch.device("cuda", 0)
    games_cap = args.slots * 24
    eng = SP.Engine(capi.GAME_OTHELLO, capi.EVAL_EXTERNAL, seed=0, sims=400, max_batch=8, max_queue=4, dir_eps=0.25,
                    dir_alpha=0.3, num_slots=args.slots, max_games=games_cap)
    try:
        eng.set_openings(lines)
        eng.attach_evalnet(net, use_cuda_graph=True)
        with torch.cuda.device(dev):
            eng.set_stream(torch.cuda.current_stream(dev).cuda_stream)
            eng.begin_iteration(0, games_cap)
            eng._capture()
            graph = eng._nn["graph"]

            def step():
                for _ in range(args.rounds):
                    graph.replay()
            for _ in range(args.warmup):
                step()
            eng.reset_stats()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                step()
            e1.record()
            torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1)
            st = eng.stats()
            playing, failed = eng.poll()
            assert failed == 0 and playing == args.slots, (playing, failed)
        net.status()
        return dict(lines=len(lines), sims_per_sec=round(st["sims"] / (ms / 1e3), 1), seconds=round(ms / 1e3, 3),
                    searched_moves=st["moves"], games=st["games"])
    finally:
        eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lines", type=int, default=1000)
    ap.add_argument("--plies", type=int, default=8)
    ap.add_argument("--slots", type=int, default=16384)
    ap.add_argument("--rounds", type=int, default=256)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=2)
    args = ap.parse_args()
    r = SP.env_rollout(capi.GAME_OTHELLO, 12345, 0, args.lines, record=True)
    starts = [0] + list(r["game_steps"].cumsum()[:-1])
    table = [[int(a) for a in r["action"][s:s + args.plies]] for s in starts]     # every play-out is longer than 9 plies
    net = EvalNet(make_network("othello", seed=0), device=0, rows=8, cols=8)
    results = {0: [], len(table): []}
    for _ in range(args.repeats):
        for lines in ([], table):
            res = run(args, lines, net)
            results[len(lines)].append(res["sims_per_sec"])
            print(json.dumps(res), flush=True)
    net.close()
    print(json.dumps({"card": card(), "slots": args.slots, "plies": args.plies,
                      "sims_per_sec_no_openings": results[0], f"sims_per_sec_{len(table)}_lines": results[len(table)]}))


if __name__ == "__main__":
    main()
