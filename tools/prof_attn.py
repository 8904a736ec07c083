"""Launch the fused attention kernel alone (for ncu): python tools/prof_attn.py [d] [T] [HW] [B] [reps]"""
import ctypes
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from efficient_slowfast_b200 import runtime as rt  # noqa: E402

d = int(sys.argv[1]) if len(sys.argv) > 1 else 32
T = int(sys.argv[2]) if len(sys.argv) > 2 else 8
HW = int(sys.argv[3]) if len(sys.argv) > 3 else 56
B = int(sys.argv[4]) if len(sys.argv) > 4 else 2
reps = int(sys.argv[5]) if len(sys.argv) > 5 else 3
DEV = "cuda:0"
L = rt.lib()
N = T * HW * HW
g = torch.Generator().manual_seed(0)
proj = torch.randn(B * N, 4 * d, generator=g).to(DEV)
proj[:, d:3 * d] *= 1.0 / d ** 0.25
alpha = 4
ybuf = torch.zeros(B, T * alpha, HW, HW, 2 * d, dtype=torch.float16, device=DEV)   # FP16: the default storage format
yv = rt.view(ybuf[..., :d])
sc = torch.ones(d, device=DEV)
sh = torch.zeros(d, device=DEV)
s = rt.current_stream_ptr()
packed = torch.empty(L.esf_attn_tc_pack_bytes(B, N, d), dtype=torch.uint8, device=DEV)
rt.check(L.esf_attn_tc_pack(proj.data_ptr(), B, N, d, rt.F16, packed.data_ptr(), s))
h = ctypes.c_void_p()
rt.check(L.esf_attn_tc_create(packed.data_ptr(), B, T, HW, HW, d, 0.5, sc.data_ptr(), sh.data_ptr(), alpha,
                              ctypes.byref(yv), ctypes.byref(h)))
launch = lambda: rt.check(L.esf_op_launch(h, s))
launch()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(reps):
    launch()
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / reps
print("attn tc d=%d N=%d B=%d: %.3f ms  %.2f Texp/s  %.1f TFLOP/s" % (d, N, B, ms, B * N * N / ms / 1e9,
                                                                     4.0 * B * N * N * d / ms / 1e9))
