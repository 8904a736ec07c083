"""Time the depthwise layers of the efficient backbones alone (CUDA events, L2 flushed between launches):
python tools/prof_dwconv.py [reps] [layer indices]"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from efficient_slowfast_b200 import runtime as rt  # noqa: E402
from efficient_slowfast_b200.engine import Plan  # noqa: E402

# (B, T, H, W, C, kT, stride) -- MobileNetV2 w1.0 two-stream layers at a quarter of the bench batch
LAYERS = [
    (32, 8, 56, 56, 144, 3, 1), (32, 8, 112, 112, 96, 3, 2), (32, 8, 112, 112, 32, 3, 1), (32, 32, 56, 56, 18, 3, 1),
    (32, 32, 28, 28, 162, 3, 2), (32, 32, 112, 112, 12, 3, 2), (32, 32, 112, 112, 4, 3, 1), (32, 32, 56, 56, 36, 3, 2),
    (64, 8, 14, 14, 576, 3, 1), (64, 8, 7, 7, 960, 3, 1), (64, 8, 28, 28, 192, 3, 1), (64, 32, 7, 7, 240, 3, 1),
]
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
if len(sys.argv) > 2:      # only these layers (indices), e.g. for an ncu capture
    LAYERS = [LAYERS[int(i)] for i in sys.argv[2].split(",")]
DEV = "cuda:0"
flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)
g = torch.Generator().manual_seed(0)
total = 0.0
for (B, T, H, W, C, kt, s) in LAYERS:
    plan = Plan(DEV, "fp16")
    st = (1, s, s)
    pad = (kt // 2, 1, 1)
    Ho, Wo = (H + 2 - 3) // s + 1, (W + 2 - 3) // s + 1
    x = plan.act(B, T, H, W, C)
    x.copy_(torch.randn(1, T, H, W, C, generator=g).to(DEV, torch.float16).expand(B, T, H, W, C))
    y = plan.act(B, T, Ho, Wo, C)
    w = torch.randn(C, 1, kt, 3, 3, generator=g).double() * 0.2
    plan.conv(x, y, w, torch.zeros(C, dtype=torch.float64), stride=st, padding=pad, groups=C, act=rt.ACT_RELU)
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
    total += ms
    m = plan.meta[-1]
    print("C=%4d %3dx%3d T=%2d s%d B=%d: %.3f ms  %5.0f GB/s  %5.1f TFLOP/s  (HBM bound %.3f ms)" % (
        C, H, W, T, s, B, ms, m["bytes"] / ms / 1e6, m["flops"] / ms / 1e9, m["bytes"] / 6538e6), flush=True)
    del plan, x, y
print("total %.3f ms" % total)
