"""JPEG frames decoded on the device (decode_jpeg) against cv2.imdecode on the host.

  python tools/bench_jpeg.py --out profiles/r12_jpeg.json

Workloads: 32 and 256 files of 640 x 360 and 1920 x 1080, quality 75 and 95, 4:2:0, restart interval 0 and one MCU
row.  The frames are a smooth moving pattern plus uniform noise of +-20 (synthetic: the ratio of compressed bytes to
pixels of real footage has not been measured here), every file distinct.  Per workload:
- `call_ms`: host clock over --iters calls of decode_jpeg(files, out) ending in a device synchronise (parse, pack, one
  H2D copy, three kernels), after --warmup calls; frames/s and megapixels/s from it; `events_ms`: CUDA events around the
  same calls (the stream also waits while the host parses).
- `host_cpu_us_per_file`: time.process_time() around each call (parse, pack and enqueue), the device idle before it,
  per file.
- `stages_ms`: device time per call of each kernel (Huffman, IDCT, colour), the memsets and the H2D copy, from
  torch.profiler in a separate pass, and the Huffman share of the kernel time.
- `h2d_bytes`: the uploaded blob (files, descriptors and tables) against the decoded pixels.
- `cv2_1thread_ms` / `cv2_pool_ms`: the same files through cv2.imdecode on one thread and on a thread pool of every
  host core (cv2 releases the GIL), per call of all files.
End to end, one AVA line: JPEG bytes -> scores of AVA SlowFast 32x2 R50 detection at batch 16 (16 clips x 32 frames of
256 x 340, quality 90, 4:2:0): decode_jpeg + forward_ava_frames against cv2.imdecode on the thread pool into pinned
memory + one H2D copy + forward_ava_frames; host clock to a device synchronise, median of --e2e-iters; both routes'
scores are compared.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import cv2
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import efficient_slowfast_b200 as esf  # noqa: E402
from bench_detection import card  # noqa: E402
from bench_detection_frames import loader_boxes  # noqa: E402
from efficient_slowfast_b200 import jpeg as J  # noqa: E402
from efficient_slowfast_b200 import workloads  # noqa: E402


def make_files(n, H, W, quality, restart, seed):
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[:H, :W]
    files = []
    for t in range(n):
        base = np.stack([(x + 3 * t) % 256, (y * 2 + t) % 256, (x + y + 5 * t) % 256], -1)
        img = np.clip(base + rng.integers(-20, 21, (H, W, 3)), 0, 255).astype(np.uint8)
        ok, buf = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, quality, cv2.IMWRITE_JPEG_RST_INTERVAL, restart,
                                             cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420])
        files.append(buf.reshape(-1))
    return files


def stage_times(fn, iters):
    """Device ms per call of each decode kernel, the memsets and the H2D copy, from torch.profiler (one profiling
    session per call)."""
    from torch.profiler import ProfilerActivity, profile

    fn()
    torch.cuda.synchronize()
    out = {}
    for _ in range(iters):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        for e in prof.key_averages():
            k = e.key
            name = ("huffman" if "jpeg_huffman" in k else "idct" if "jpeg_idct" in k else "color" if "jpeg_color" in k
                    else "memset" if "Memset" in k else "h2d" if "HtoD" in k else None)
            if name:
                t = getattr(e, "device_time_total", None)
                if t is None:
                    t = e.cuda_time_total
                out[name] = out.get(name, 0.0) + t / 1e3 / iters
    kern = sum(out.get(k, 0.0) for k in ("huffman", "idct", "color"))
    res = {k: round(v, 4) for k, v in out.items()}
    res["huffman_share_of_kernels"] = round(out.get("huffman", 0.0) / kern, 3) if kern else None
    return res


def bench_case(n, H, W, q, rst_rows, a, pool):
    mcux = -(-W // 16)
    files = make_files(n, H, W, q, mcux if rst_rows else 0, seed=n + q + W)
    out = torch.empty(n, H, W, 3, dtype=torch.uint8, device="cuda")
    hdrs = [J.parse(f) for f in files]
    parts, offs, head, data, *_ = J.pack(hdrs, files)

    def dev():
        return J.decode_jpeg(files, out)

    for _ in range(a.warmup):
        dev()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(a.iters):
        dev()
    e1.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / a.iters
    ev = e0.elapsed_time(e1) / a.iters
    cpu = 0.0
    for _ in range(a.iters):      # host CPU of the call itself, on an idle device (no wait for an earlier call)
        torch.cuda.synchronize()
        c0 = time.process_time()
        dev()
        cpu += (time.process_time() - c0) / a.iters
    torch.cuda.synchronize()
    ref = np.stack([cv2.imdecode(f, cv2.IMREAD_COLOR) for f in files[:4]])
    exact = bool(np.array_equal(out[:4].cpu().numpy(), ref))
    t0 = time.perf_counter()
    for f in files:
        cv2.imdecode(f, cv2.IMREAD_COLOR)
    one = time.perf_counter() - t0
    list(pool.map(lambda f: cv2.imdecode(f, cv2.IMREAD_COLOR), files))
    t0 = time.perf_counter()
    list(pool.map(lambda f: cv2.imdecode(f, cv2.IMREAD_COLOR), files))
    many = time.perf_counter() - t0
    return {"files": n, "size": "%dx%d" % (W, H), "quality": q, "sampling": "4:2:0",
            "restart": "one MCU row (%d MCUs)" % mcux if rst_rows else 0,
            "segments": sum(len(h.segments) for h in hdrs),
            "call_ms": round(wall * 1e3, 3), "events_ms": round(ev, 3),
            "frames_per_s": round(n / wall, 1), "megapixels_per_s": round(n * H * W / wall / 1e6, 1),
            "host_cpu_us_per_file": round(cpu / n * 1e6, 1),
            "stages_ms": stage_times(dev, 3),
            "h2d_bytes": head + data, "pixel_bytes": n * H * W * 3,
            "cv2_1thread_ms": round(one * 1e3, 3), "cv2_pool_ms": round(many * 1e3, 3),
            "device_vs_cv2_pool": round(many / wall, 3), "first_4_frames_equal_cv2": exact}


def e2e(a, pool):
    cfg = esf.ava_slowfast_32x2_r50_cfg()
    cfg.NUM_GPUS = 1
    torch.manual_seed(0)
    model = esf.build_model(cfg)
    bn = {k[3:]: v for k, v in workloads.load_golden("slowfast_r50").items() if k.startswith("bn/")}
    model.load_state_dict(workloads.seeded_state_dict(model.state_dict(), seed=0, bn_stats=bn), strict=True)
    model = model.cuda().eval()
    B, T, H, W = 16, int(cfg.DATA.NUM_FRAMES), 256, 340
    files = make_files(B * T, H, W, 90, 0, seed=7)
    boxes = loader_boxes(B, 4, seed=1)
    frames = torch.empty(B, T, H, W, 3, dtype=torch.uint8, device="cuda")
    host = torch.empty(B, T, H, W, 3, dtype=torch.uint8).pin_memory()
    hv = host.numpy().reshape(B * T, H, W, 3)

    def device_route():
        J.decode_jpeg(files, frames)
        return model.forward_ava_frames(frames, boxes)

    def host_route():
        def dec(i):
            hv[i] = cv2.imdecode(files[i], cv2.IMREAD_COLOR)
        list(pool.map(dec, range(B * T)))
        frames.copy_(host, non_blocking=True)
        return model.forward_ava_frames(frames, boxes)

    res = {"model": "AVA SLOWFAST_32x2_R50", "batch": B, "frames": T, "size": "%dx%d" % (W, H), "quality": 90}
    with torch.no_grad():
        outs = {}
        for name, fn in (("device_jpeg", device_route), ("host_cv2_pool", host_route)):
            for _ in range(a.warmup):
                fn()
            torch.cuda.synchronize()
            ts = []
            for _ in range(a.e2e_iters):
                t0 = time.perf_counter()
                y = fn()
                torch.cuda.synchronize()
                ts.append((time.perf_counter() - t0) * 1e3)
            outs[name] = y.cpu()
            res[name + "_ms"] = round(statistics.median(ts), 2)
        res["scores_equal"] = bool(torch.equal(outs["device_jpeg"], outs["host_cv2_pool"]))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--e2e-iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_jpeg needs a CUDA device")
    pool = ThreadPoolExecutor(os.cpu_count())
    res = {"card": card(), "host_cores": os.cpu_count(), "iters": a.iters, "warmup": a.warmup,
           "runs": "each number from one run", "workloads": []}
    for n in (32, 256):
        for H, W in ((360, 640), (1080, 1920)):
            for q in (75, 95):
                for rst in (0, 1):
                    res["workloads"].append(bench_case(n, H, W, q, rst, a, pool))
                    print(json.dumps(res["workloads"][-1]), file=sys.stderr)
    res["end_to_end"] = e2e(a, pool)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
