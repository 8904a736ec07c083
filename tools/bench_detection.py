"""AVA detection throughput of the AVA SLOWFAST_32x2_R50 model (ResNetRoIHead, res5 at stride 1 / dilation 2, 80
sigmoid classes) on one GPU: model(clips, boxes) at batch 16 for 224 x 224 clips and for 256 x 340 AVA test frames, with
4 and 16 boxes per clip.

Per workload: ms per forward (CUDA events around `model(xs, host_boxes)`, the boxes copied from the host each call as
the test loop does), clips/s and boxes/s; the device time of the trunk (`plan.run`: stem packing + graph replay) and of
the box-dependent part (`plan.run_boxes`: RoIAlign + max per pathway + projection) measured separately with events; and
the parity of the timed batch against the FP32 CPU oracle on its first and last clip (the oracle would need minutes
for all 16).  Weights are seeded with the calibrated BN statistics of the slowfast_r50 fixture (same BN keys).  The card
name and power limit are read in the same run.  Prints one JSON line; --out also writes it to a file.

    python tools/bench_detection.py [--batch 16] [--steps 20] [--warmup 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import detection_oracle as DO  # noqa: E402
import efficient_slowfast_b200 as esf  # noqa: E402
from efficient_slowfast_b200 import workloads  # noqa: E402


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], stdout=subprocess.PIPE, text=True, timeout=60).stdout
        pl, mhz = [v.strip() for v in out.strip().split(",")]
        info.update(power_limit_w=float(pl), sm_max_mhz=float(mhz))
    except Exception as e:  # noqa: BLE001
        info["power_limit_w"] = "unavailable: %s" % e
    return info


def boxes_for(B, per_clip, H, W, seed):
    """`per_clip` boxes for every clip: person-sized boxes (15-60 % of the frame) inside the frame."""
    g = torch.Generator().manual_seed(seed)
    K = B * per_clip
    b = torch.arange(B).repeat_interleave(per_clip).float()
    w, h = (0.15 + 0.45 * torch.rand(K, generator=g)) * W, (0.15 + 0.45 * torch.rand(K, generator=g)) * H
    x1, y1 = torch.rand(K, generator=g) * (W - w), torch.rand(K, generator=g) * (H - h)
    return torch.stack([b, x1, y1, x1 + w, y1 + h], 1)


def timed(fn, steps):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(steps):
        fn()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_detection needs a CUDA device")
    cfg = esf.ava_slowfast_32x2_r50_cfg()
    cfg.NUM_GPUS = 1
    torch.manual_seed(0)
    model = esf.build_model(cfg)
    bn = {k[3:]: v for k, v in workloads.load_golden("slowfast_r50").items() if k.startswith("bn/")}
    sd = workloads.seeded_state_dict(model.state_dict(), seed=0, bn_stats=bn)
    model.load_state_dict(sd, strict=True)
    model = model.cuda().eval()
    res = {"model": "AVA SLOWFAST_32x2_R50 (SlowFast R50 + ResNetRoIHead, res5 stride 1 dilation 2)",
           "precision": cfg.ESF.PRECISION, "batch": a.batch, "steps": a.steps, "warmup": a.warmup, "card": card(),
           "workloads": []}
    for H, W in ((224, 224), (256, 340)):
        g = torch.Generator().manual_seed(1)
        fast = torch.randn(a.batch, 3, cfg.DATA.NUM_FRAMES, H, W, generator=g)
        xs_h = workloads.pack_pathway_output(fast, cfg.SLOWFAST.ALPHA)
        xs = [t.cuda() for t in xs_h]
        trunk = None
        for per_clip in (4, 16):
            boxes = boxes_for(a.batch, per_clip, H, W, seed=per_clip)
            boxes_d = boxes.cuda()
            with torch.no_grad():
                for _ in range(a.warmup):
                    model(xs, boxes)
                torch.cuda.synchronize()
                ms = timed(lambda: model(xs, boxes), a.steps)
                y = model(xs, boxes).cpu()
                plan = list(model._plans.values())[-1][1]
                trunk_ms = timed(lambda: plan.run(xs), a.steps)
                roi_ms = timed(lambda: plan.run_boxes(boxes_d), a.steps)
            if trunk is None:     # FP32 CPU oracle trunk of the first and the last clip of the timed batch
                sel = [0, a.batch - 1]
                trunk = DO.trunk(cfg, sd, [t[sel] for t in xs_h])
            rows = torch.cat([torch.nonzero(boxes[:, 0] == c).flatten() for c in (0, a.batch - 1)])
            ob = boxes[rows].clone()
            ob[:, 0] = (ob[:, 0] > 0).float()          # clip index inside the two-clip oracle batch
            want = DO.head(cfg, sd, trunk, ob)
            err = ((y[rows].double() - want.double()).abs().max() / want.double().abs().max()).item()
            K = boxes.shape[0]
            res["workloads"].append(dict(
                frames="%dx%d" % (H, W), slow_fast_frames=[xs[0].shape[2], xs[1].shape[2]], boxes_per_clip=per_clip,
                boxes=K, ms_per_forward=round(ms, 3), clips_per_s=round(a.batch * 1000.0 / ms, 1),
                boxes_per_s=round(K * 1000.0 / ms, 1), trunk_ms=round(trunk_ms, 3), roi_ms=round(roi_ms, 4),
                roi_share_of_trunk=round(roi_ms / trunk_ms, 5), res5_map=list(plan.roi["maps"][0].shape[1:3]),
                oracle_rows=int(rows.numel()), oracle_rel_err=err, finite=bool(torch.isfinite(y).all()),
                plans=len(model._plans)))
            print(json.dumps(res["workloads"][-1]), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
