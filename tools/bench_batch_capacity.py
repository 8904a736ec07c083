"""Batch capacity (cfg.ESF.MAX_BATCH): a variant of a plan family against a dedicated plan of the same batch.

  python tools/bench_batch_capacity.py --out profiles/r8_batch_capacity.json

Model: SlowFastDualAttention 8x8 R50, FP16, 32 x 224^2 clips (the headline workload of bench.py), with the parity
recipe's weights.  The family is compiled for `--capacity` rows (default 64); the comparison runs at `--rows` (default
32).  Reported:
  * time to the first output: host clock around the first forward call at `--rows` rows, ended by a device
    synchronise -- for the dedicated plan the whole compile (weight folding and packing, arena allocation, op
    creation, graph capture) and one run; for the variant its compile and one run, the capacity plan already built;
  * device memory that call adds (torch.cuda.memory_allocated after minus before), and the capacity plan's
    arena_bytes();
  * steady-state forward time of the variant and of the dedicated plan at `--rows`: CUDA events around `--iters`
    forwards on the same input, the two alternated `--repeats` times, best and median window reported;
  * whether the two outputs are bit-identical.
The card's name, power limit and clocks are read in the same run.
"""
import argparse
import json
import os
import statistics
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import efficient_slowfast_b200 as esf  # noqa: E402
from bench_frames_spatial import gpu_info  # noqa: E402
from efficient_slowfast_b200 import workloads as W  # noqa: E402


def build(capacity):
    """(cfg, dedicated model, family model with MAX_BATCH = capacity), same weights, on the GPU."""
    cfg = esf.slowfast_dual_8x8_r50_cfg()
    cfg.NUM_GPUS = 0
    torch.manual_seed(0)
    model = esf.build_model(cfg)
    gold = W.load_golden("dual_r50")
    bn = {k[3:]: v for k, v in gold.items() if k.startswith("bn/")}
    model.load_state_dict(W.seeded_state_dict(model.state_dict(), seed=0, bn_stats=bn), strict=True)
    cfg.ESF.MAX_BATCH = capacity
    fam = model.__class__(cfg)
    fam.load_state_dict(model.state_dict())
    return cfg, model.cuda().eval(), fam.cuda().eval()


def first_output(model, xs):
    """(seconds to the first output, device bytes the call added, output)."""
    torch.cuda.synchronize()
    mem = torch.cuda.memory_allocated()
    t0 = time.perf_counter()
    y = model(xs)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, torch.cuda.memory_allocated() - mem - y.numel() * y.element_size(), y


def window_ms(model, xs, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        model(xs)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--capacity", type=int, default=64)
    ap.add_argument("--rows", type=int, default=32)
    ap.add_argument("--frames", type=int, default=32)
    ap.add_argument("--crop", type=int, default=224)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: nothing here is measured on the CPU")
    if not 1 <= a.rows < a.capacity:
        raise SystemExit("--rows must be in [1, --capacity)")
    res = dict(gpu=gpu_info(), workload=dict(model="SlowFastDualAttention 8x8 R50", precision="fp16",
                                             frames=a.frames, crop=a.crop, capacity=a.capacity, rows=a.rows))
    cfg, model, fam = build(a.capacity)
    alpha = cfg.SLOWFAST.ALPHA
    g = torch.Generator(device="cuda").manual_seed(0)
    fast = torch.randn(a.capacity, 3, a.frames, a.crop, a.crop, device="cuda", generator=g)
    idx = torch.linspace(0, a.frames - 1, a.frames // alpha).long().cuda()
    xs = [fast.index_select(2, idx).contiguous(), fast]
    xb = [x[:a.rows].contiguous() for x in xs]
    with torch.no_grad():
        t_cap, m_cap, _ = first_output(fam, xs)
        cap = next(iter(fam._plans.values()))[1]
        t_var, m_var, y_var = first_output(fam, xb)
        t_ded, m_ded, y_ded = first_output(model, xb)
        ded = next(reversed(model._plans.values()))[1]
        res["first_output_s"] = dict(capacity_plan=t_cap, variant=t_var, dedicated=t_ded)
        res["device_bytes_added"] = dict(capacity_plan=m_cap, variant=m_var, dedicated=m_ded)
        res["arena_bytes"] = dict(capacity_plan=cap.arena_bytes(), dedicated=ded.arena_bytes())
        res["bit_identical"] = bool(torch.equal(y_var, y_ded))
        for m in (fam, model):
            window_ms(m, xb, 3)
        var_ms, ded_ms = [], []
        for _ in range(a.repeats):
            var_ms.append(window_ms(fam, xb, a.iters))
            ded_ms.append(window_ms(model, xb, a.iters))
        res["forward_ms"] = dict(variant=dict(best=min(var_ms), median=statistics.median(var_ms), all=var_ms),
                                 dedicated=dict(best=min(ded_ms), median=statistics.median(ded_ms), all=ded_ms))
        res["plans"] = dict(family_lru_entries=len(fam._plans), variants=sorted(cap.variants))
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
