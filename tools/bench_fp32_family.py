"""The FP32-accurate plan (cfg.ESF.PRECISION = "fp32") against the FP16 plan on the ResNet family's newly covered paths.

  python tools/bench_fp32_family.py --out /tmp/fp32_family.json

(a) SlowFast 4x16 R50 (the stock config: head pool from the 224^2 training crop) at its fully-convolutional test crop:
    B clips of 32 uint8 frames at 256 x 340 through forward_frames(frames, crop_size=256, spatial_idx=(0, 1, 2)) --
    3 views per clip, an 8 x 8 res5 map, Linear + softmax at 2 x 2 positions.
(b) slowfast_r50_g2 (RESNET.NUM_GROUPS 2) at 224^2 with global head pooling.  The FP32 plan runs each grouped 3 x 3
    conv as one dense split GEMM over a block-diagonal weight: twice the MACs of that layer.
Each workload times both precisions with CUDA events after warm-up, in windows of at least a second, alternating the
two plans; the median window is reported.  The card's name and power limit are read in the same run.  Weights are the
recipe's seeded ones (workloads.py): timing does not depend on their values.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from efficient_slowfast_b200 import config as esf_cfg  # noqa: E402
from efficient_slowfast_b200.build import build_model  # noqa: E402
from efficient_slowfast_b200.workloads import (case_model_and_weights, load_golden, pack_pathway_output,  # noqa: E402
                                               seeded_clip, seeded_state_dict)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        return dict(zip(q.split(","), [v.strip() for v in r.stdout.splitlines()[0].split(",")]))
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def window_ms(fn, min_s):
    """One timing window: ms per call of fn, over as many calls as fill at least min_s seconds between two events."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    n = max(1, int(min_s * 1e3 / max(a.elapsed_time(b), 1e-3)) + 1)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def compare(fns, rows, min_s, rounds):
    """fns: precision -> callable; alternates the precisions `rounds` times."""
    for fn in fns.values():     # warm-up: plan build, graph capture, first launches
        for _ in range(3):
            fn()
    times = {p: [] for p in fns}
    for _ in range(rounds):
        for p, fn in fns.items():
            times[p].append(window_ms(fn, min_s))
    out = {}
    for p, ts in times.items():
        ms = statistics.median(ts)
        out[p] = dict(ms_per_call=ms, rows_per_s=rows / ms * 1e3, windows_ms=ts)
    out["fp32_over_fp16"] = out["fp32"]["ms_per_call"] / out["fp16"]["ms_per_call"]
    return out


def fcn_models():
    gold = load_golden("slowfast_r50")        # same parameter shapes as the stock 4x16 config
    bn = {k[3:]: v for k, v in gold.items() if k.startswith("bn/")}
    models = {}
    for prec in ("fp16", "fp32"):
        cfg = esf_cfg.slowfast_4x16_r50_cfg()
        cfg.NUM_GPUS = 0
        cfg.ESF.PRECISION = prec
        torch.manual_seed(0)
        m = build_model(cfg)
        m.load_state_dict(seeded_state_dict(m.state_dict(), seed=0, bn_stats=bn), strict=True)
        models[prec] = m.cuda().eval()
    return cfg, models


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--fcn-batch", type=int, default=8, help="clips per call of (a); 3 views each")
    ap.add_argument("--g2-batch", type=int, default=16)
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: nothing here is measured on the CPU")
    res = dict(gpu=gpu_info(), device=torch.cuda.get_device_name(0))
    with torch.no_grad():
        cfg, models = fcn_models()
        S = int(cfg.DATA.TEST_CROP_SIZE)
        frames = torch.randint(0, 256, (a.fcn_batch, cfg.DATA.NUM_FRAMES, 256, 340, 3), dtype=torch.uint8,
                               generator=torch.Generator().manual_seed(3)).cuda()
        fns = {p: (lambda m=m: m.forward_frames(frames, crop_size=S, spatial_idx=(0, 1, 2))) for p, m in models.items()}
        res["a_slowfast_4x16_r50_fcn_3view"] = dict(
            clips=a.fcn_batch, rows=3 * a.fcn_batch, frames=[256, 340], test_crop=S,
            **compare(fns, 3 * a.fcn_batch, a.min_seconds, a.rounds))
        del models, fns, frames
        torch.cuda.empty_cache()

        models = {p: case_model_and_weights("slowfast_r50_g2", p)[1].cuda().eval() for p in ("fp16", "fp32")}
        xs = [t.cuda() for t in pack_pathway_output(seeded_clip(a.g2_batch, 32, 224, seed=1), 8)]
        fns = {p: (lambda m=m: m(xs)) for p, m in models.items()}
        res["b_slowfast_r50_g2_224"] = dict(clips=a.g2_batch, crop=224,
                                            **compare(fns, a.g2_batch, a.min_seconds, a.rounds))
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
