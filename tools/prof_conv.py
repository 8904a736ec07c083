"""Launch one conv layer alone (for ncu / timing):
python tools/prof_conv.py B T H W Cin Cout kT kH kW sT sH sW res(0|1) [reps] [precision] [wfold(0|1)]
wfold=0 runs the dense layer on the plain implicit GEMM where Plan.conv would pick the W-folded one."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from efficient_slowfast_b200 import runtime as rt  # noqa: E402
from efficient_slowfast_b200.engine import Plan  # noqa: E402

a = [int(v) for v in sys.argv[1:14]]
B, T, H, W, cin, cout, kt, kh, kw, st, sh, sw, use_res = a
reps = int(sys.argv[14]) if len(sys.argv) > 14 else 5
precision = sys.argv[15] if len(sys.argv) > 15 else "fp16"
wfold = int(sys.argv[16]) if len(sys.argv) > 16 else 1
groups = int(os.environ.get("ESF_PROF_GROUPS", "1"))
DEV = "cuda:0"
adt = rt.TORCH_DTYPE[precision]
pad = (kt // 2, kh // 2, kw // 2)
To, Ho, Wo = (T + 2 * pad[0] - kt) // st + 1, (H + 2 * pad[1] - kh) // sh + 1, (W + 2 * pad[2] - kw) // sw + 1
g = torch.Generator().manual_seed(0)
plan = Plan(DEV, precision)
x = plan.act(B, T, H, W, cin)
x.copy_(torch.randn(B, T, H, W, cin, generator=g).to(DEV, adt))
y = plan.act(B, To, Ho, Wo, cout)
res = torch.randn(B, To, Ho, Wo, cout, generator=g).to(DEV, adt) if use_res else None
w = torch.randn(cout, cin // groups, kt, kh, kw, generator=g).double() * (2.0 * groups / (cin * kt * kh * kw)) ** 0.5
zero = torch.zeros(cout, dtype=torch.float64)
if wfold:
    plan.conv(x, y, w, zero, stride=(st, sh, sw), padding=pad, groups=groups, act=rt.ACT_RELU, res=res)
else:
    plan.conv_igemm(x, y, w, zero, stride=(st, sh, sw), padding=pad, act=rt.ACT_RELU, res=res)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)
plan.launch_all()
torch.cuda.synchronize()
tot = 0.0
for _ in range(reps):
    flush.fill_(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    plan.launch_all()
    e1.record()
    torch.cuda.synchronize()
    tot += e0.elapsed_time(e1)
ms = tot / reps
m = plan.meta[-1]
print("%s %s: %.3f ms  %.0f GB/s  %.1f TFLOP/s" % (m["kind"], m["label"], ms, m["bytes"] / ms / 1e6, m["flops"] / ms / 1e9))
