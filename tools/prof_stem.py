"""Time (or, under ncu, expose) the fast-pathway stem alone at the headline shape.
    python tools/prof_stem.py [batch] [iters] [banded(0|1)]        banded=1: the banded stem instead of the temporal band"""
import os
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

from efficient_slowfast_b200 import runtime as rt
from efficient_slowfast_b200.engine import Plan, stem_route

B = int(sys.argv[1]) if len(sys.argv) > 1 else 64
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 20
banded = int(sys.argv[3]) if len(sys.argv) > 3 else 0
g = torch.Generator().manual_seed(0)
x = torch.randn(B, 3, 32, 224, 224, device="cuda")
w = (torch.randn(8, 3, 5, 7, 7, generator=g) * 0.1).double()
b = (torch.randn(8, generator=g) * 0.1).double()
y = torch.empty(B, 32, 112, 112, 8, dtype=torch.float16, device="cuda")
plan = Plan(torch.device("cuda"), "fp16")
pitch, lpad, twb = stem_route(x.shape, w.shape, (1, 2, 2), (2, 3, 3))
plan.stem_gemm(x, y, w, b, (1, 2, 2), (2, 3, 3), rt.ACT_RELU, pitch, lpad, 0 if banded else twb)
plan.launch_all()
torch.cuda.synchronize()
h = plan.handles[-1]
f = lambda: rt.check(rt.lib().esf_op_launch(h, None))
for _ in range(min(3, iters)):
    f()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(iters):
    f()
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / iters
flops = 2.0 * y.numel() * 3 * 5 * 7 * 7
print("%s batch %d: %.3f ms  %.1f TFLOP/s (true MACs)  %.2f TB/s (packed clip + output)"
      % (plan.meta[-1]["label"], B, ms, flops / ms / 1e9, (x.numel() / 3 * 688 / 224 * 2 / 1 + y.numel() * 2) / ms / 1e9))
