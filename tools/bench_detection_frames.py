"""AVA detection from uint8 frames against host-prepared FP32 clips: the AVA SLOWFAST_32x2_R50 model at batch 16.

Routes, per decode size (256 x 340 AVA keyframe clips, a pure window at TEST_CROP_SIZE 256; and 240 x 320, resized to
256 x 341), each timed with CUDA events over --steps forwards after --warmup:
- `u8_device`:    model.forward_ava_frames(frames, boxes) on device-resident uint8 frames, the loader's [0, 1] boxes
                  from the host (what the test loop hands over).
- `u8_h2d`:       the same with the uint8 frames copied from pinned host memory in every step.
- `fp32_device`:  model(clips, boxes) on device-resident FP32 [slow, fast] clips prepared on the host by the loader chain
                  (tests/ava_frames_oracle.py), boxes in pixels from the host.
- `fp32_h2d`:     the same with both FP32 clips copied from pinned host memory in every step.
Also: the host preparation time of the FP32 route (the oracle's loader chain for the batch, run once: it is minutes of
CPU for more), the device time of the frame kernels alone (both pathways, CUDA events over --kernel-steps launches) with
the bytes they must move against the 7.7 TB/s data-sheet HBM bandwidth, and whether the two routes' scores are equal.
The card name and power limit are read in the same run.  Prints one JSON line; --out also writes it to a file.

    python tools/bench_detection_frames.py [--batch 16] [--steps 20] [--warmup 5] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import ava_frames_oracle as AO  # noqa: E402
import efficient_slowfast_b200 as esf  # noqa: E402
from bench_detection import card, timed  # noqa: E402
from efficient_slowfast_b200 import frames as FR  # noqa: E402
from efficient_slowfast_b200 import workloads  # noqa: E402

HBM_TBS = 7.7   # NVIDIA's data sheet, one HGX B200 GPU


def loader_boxes(B, per_clip, seed):
    """`per_clip` person-sized boxes per clip in the annotation's [0, 1] coordinates (FP64, as ava_helper reads them)."""
    g = torch.Generator().manual_seed(seed)
    K = B * per_clip
    b = torch.arange(B).repeat_interleave(per_clip).double()
    w, h = 0.15 + 0.45 * torch.rand(K, generator=g, dtype=torch.float64), 0.15 + 0.45 * torch.rand(K, generator=g,
                                                                                                   dtype=torch.float64)
    x1, y1 = torch.rand(K, generator=g, dtype=torch.float64) * (1 - w), torch.rand(K, generator=g,
                                                                                    dtype=torch.float64) * (1 - h)
    return torch.stack([b, x1, y1, x1 + w, y1 + h], 1)


def kernel_bytes(plan, B, T, H, W, C, Hr, Wr):
    """Bytes the frame kernels must move for one batch: every source row they read (each output row reads one row
    of a pure window, two of a resize; rows of neighbouring output rows come from L2 at best) and every output
    element they write (16-bit packed rows or FP32)."""
    resize = (Hr, Wr) != (H, W)
    read = write = 0
    for own in plan.inputs:
        t = own.shape[2]
        read += B * t * Hr * (2 if resize else 1) * W * C
        route = plan.stem_routes.get(own.data_ptr())
        write += B * t * Hr * (route[1] * 2 if route is not None else Wr * C * 4)
    return read, write


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--kernel-steps", type=int, default=50)
    ap.add_argument("--boxes-per-clip", type=int, default=4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_detection_frames needs a CUDA device")
    cfg = esf.ava_slowfast_32x2_r50_cfg()
    cfg.NUM_GPUS = 1
    torch.manual_seed(0)
    model = esf.build_model(cfg)
    bn = {k[3:]: v for k, v in workloads.load_golden("slowfast_r50").items() if k.startswith("bn/")}
    model.load_state_dict(workloads.seeded_state_dict(model.state_dict(), seed=0, bn_stats=bn), strict=True)
    model = model.cuda().eval()
    B, T, S, alpha = a.batch, int(cfg.DATA.NUM_FRAMES), int(cfg.DATA.TEST_CROP_SIZE), cfg.SLOWFAST.ALPHA
    res = {"model": "AVA SLOWFAST_32x2_R50 (SlowFast R50 + ResNetRoIHead)", "precision": cfg.ESF.PRECISION,
           "batch": B, "frames": T, "crop_size": S, "boxes_per_clip": a.boxes_per_clip, "steps": a.steps,
           "warmup": a.warmup, "kernel_steps": a.kernel_steps, "card": card(), "runs": "each number from one run",
           "workloads": []}
    for H, W in ((256, 340), (240, 320)):
        g = torch.Generator().manual_seed(H)
        fr_h = torch.randint(0, 256, (B, T, H, W, 3), generator=g, dtype=torch.uint8).pin_memory()
        fr_d = fr_h.cuda()
        boxes = loader_boxes(B, a.boxes_per_clip, seed=H)
        t0 = time.perf_counter()
        xs_cpu, px_h = AO.prepare(fr_h, boxes, S, cfg.DATA.MEAN, cfg.DATA.STD, alpha)
        host_prep_ms = (time.perf_counter() - t0) * 1e3
        xs_h = [t.pin_memory() for t in xs_cpu]
        xs_d = [t.cuda() for t in xs_h]
        stage = [torch.empty_like(t) for t in xs_d]
        fr_stage = torch.empty_like(fr_d)

        def u8_device():
            return model.forward_ava_frames(fr_d, boxes)

        def u8_h2d():
            fr_stage.copy_(fr_h, non_blocking=True)
            return model.forward_ava_frames(fr_stage, boxes)

        def fp32_device():
            return model(xs_d, px_h)

        def fp32_h2d():
            for d, h in zip(stage, xs_h):
                d.copy_(h, non_blocking=True)
            return model(stage, px_h)

        w = {"decode": "%dx%d" % (H, W), "resized": "%dx%d" % FR.resized_size(H, W, S),
             "host_prep_ms_once": round(host_prep_ms, 1),
             "h2d_bytes": {"u8": fr_h.numel(), "fp32": sum(t.numel() * 4 for t in xs_h)}}
        with torch.no_grad():
            for name, fn in (("u8_device", u8_device), ("u8_h2d", u8_h2d), ("fp32_device", fp32_device),
                             ("fp32_h2d", fp32_h2d)):
                for _ in range(a.warmup):
                    fn()
                torch.cuda.synchronize()
                w[name + "_ms"] = round(timed(fn, a.steps), 3)
            y_u8, px = model.forward_ava_frames(fr_d, boxes, return_boxes=True)
            y_fp = model(xs_d, px_h)
            w["scores_equal"] = bool(torch.equal(y_u8, y_fp))
            w["boxes_equal"] = bool(torch.equal(px.cpu(), px_h))
            plan, fin = model._frame_plan(model.frame_shapes((B, T) + FR.resized_size(H, W, S) + (3,)), fr_d.device, 3)
            state, tabs = fin.ava(cfg), fin.crop(H, W, S, ())
            fill = lambda: FR.launch_ava(plan, fin, state, fr_d, tabs, alpha)  # noqa: E731
            for _ in range(3):
                fill()
            torch.cuda.synchronize()
            k_ms = timed(fill, a.kernel_steps)
        rd, wr = kernel_bytes(plan, B, T, H, W, 3, tabs.Hr, tabs.Wr)
        w.update(kernel_ms=round(k_ms, 4), kernel_read_gb=round(rd / 1e9, 4), kernel_write_gb=round(wr / 1e9, 4),
                 kernel_gb_per_s=round((rd + wr) / k_ms / 1e6, 1),
                 kernel_share_of_hbm=round((rd + wr) / k_ms / 1e6 / (HBM_TBS * 1e3), 4),
                 packed_stem_rows=[own.data_ptr() in plan.stem_routes for own in plan.inputs])
        res["workloads"].append(w)
        print(json.dumps(w), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
