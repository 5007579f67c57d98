"""GPU check of the tcgen05 evaluator against the fp32 PyTorch forward of the same network.
    python tools/check_evalnet.py [batch] [blocks]"""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from sprl_b200.evalnet import EvalNet
from sprl_b200.network import BasicGridNetwork

B = int(sys.argv[1]) if len(sys.argv) > 1 else 256
blocks = int(sys.argv[2]) if len(sys.argv) > 2 else 2
torch.manual_seed(0)
net = BasicGridNetwork(8, 8, 65, 1, blocks, 64).eval()
# non-trivial BatchNorm statistics so that folding is exercised
with torch.no_grad():
    for mod in net.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.running_mean.uniform_(-0.5, 0.5); mod.running_var.uniform_(0.5, 2.0)
            mod.weight.uniform_(0.5, 1.5); mod.bias.uniform_(-0.5, 0.5)
x = (torch.rand(B, 3, 8, 8) > 0.5).float()
with torch.no_grad():
    ref_l, ref_v = net.double()(x.double())
    net.float()
    f32_l, f32_v = net(x)
ev = EvalNet(net, device=0)
xg = x.cuda()
t0 = time.time()
lg, v = ev(xg)
torch.cuda.synchronize()
print(f"first forward {1e3 * (time.time() - t0):.1f} ms, status launches={ev.status()}", flush=True)
el, evv = (lg.cpu().double() - ref_l).abs().max().item(), (v.cpu().double() - ref_v).abs().max().item()
fl, fv = (f32_l.double() - ref_l).abs().max().item(), (f32_v.double() - ref_v).abs().max().item()
print(f"B={B} blocks={blocks}: max|dlogit| vs fp64: ours {el:.3e} (torch fp32 CPU {fl:.3e}); max|dvalue| ours {evv:.3e} (torch {fv:.3e}); "
      f"logit scale {ref_l.abs().max().item():.3f}", flush=True)
if el > 1e-4 or evv > 1e-4:
    bad = (lg.cpu().double() - ref_l).abs().amax(1)
    print("worst boards:", bad.topk(min(8, B)).indices.tolist(), bad.topk(min(8, B)).values.tolist())
    print("ours[0,:8]", lg[0, :8].tolist(), "\nref [0,:8]", ref_l[0, :8].tolist())
    sys.exit(1)
if B >= 4096:
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        ev(xg)
    e0.record()
    for _ in range(10):
        ev(xg)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    flop = (64 * 27 * 64 + 2 * blocks * 64 * 64 * 9 * 64 + 3 * 64 * 64 + 128 * 65 + 64 * 64 + 64) * 2
    print(f"forward B={B}: {ms:.3f} ms, {B / ms * 1e3 / 1e6:.2f} M evals/s, {B * flop / ms / 1e9:.1f} TFLOP/s fp32-equivalent "
          f"({3 * B * flop / ms / 1e9:.1f} TF32 tensor TFLOP/s issued)", flush=True)
ev.status()
print("evalnet ok")
