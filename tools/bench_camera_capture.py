"""The demo loop over N cameras from raw captures: the caller's host preprocessing against the device's.

  python tools/bench_camera_capture.py --out profiles/r11_camera_capture.json

Host route (what a caller does without scale_to): for every frame cv2.cvtColor(BGR2RGB) and cv2.resize(INTER_LINEAR)
to short side 224 into pinned buffers on the host, then one CameraWindows per scaled size, the frames split between them
by hand.  Device route: the raw pinned BGR captures into one CameraWindows(scale_to=224, bgr=True), which stages them on
the device and resizes them with esf_resize_u8_cv2.  Banks: every camera 1280 x 720, every camera 1920 x 1080 (both
scale to 224 x 398), and half 640 x 480 (224 x 298) / half 1280 x 720.  Models: those of tools/bench_camera_windows.py
(SlowFast 8x8 R50 with a 64-frame window, SlowFast-ShuffleNetV2 1.0x), FP16, seeded weights, cfg.ESF.MAX_BATCH = 32.

Method: both routes' windows are filled, then the routes are warmed up, alternating, for at least `--warmup-s` seconds
(the SM clock read after the warm-up is recorded); then each is timed in windows of at least `--window-s` seconds and
`--min-ticks` ticks, alternated `--repeats` times, on the host clock from the first push to a device synchronise after
the last forward, with time.process_time() over the same window (the host CPU time of the whole process: the cv2 calls
and every push).  H2D bytes per tick are counted from the shapes.  The resize kernel is timed on its own with CUDA
events over `--kernel-iters` launches of one tick's frames (all cameras, already staged); its bytes are the two source
rows it loads per output row plus the bytes it writes.  The first tick's scores of both routes are compared.  The
card's name, power limit and clocks are read in the same run.
"""
import argparse
import json
import math
import os
import statistics
import sys
import time

import cv2
import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import efficient_slowfast_b200 as esf  # noqa: E402
from bench_camera_windows import build  # noqa: E402
from bench_frames_spatial import gpu_info  # noqa: E402
from efficient_slowfast_b200 import frames as F  # noqa: E402

S = 224
BANKS = {"720p": lambda n: [(720, 1280)] * n, "1080p": lambda n: [(1080, 1920)] * n,
         "mixed": lambda n: [(480, 640) if c % 2 == 0 else (720, 1280) for c in range(n)]}


def kernel_time(bank, sizes, pool, iters):
    """(ms per launch, bytes per launch) of esf_resize_u8_cv2 on one tick of every camera's frame, staged."""
    staged = [pool[(H, W)][0].cuda() for H, W in sizes]
    dst = [b.bank[b.ring[c], 0].data_ptr() for c, b in enumerate(bank._bank_of)]
    args = ([f.data_ptr() for f in staged], dst, bank._resize, 3)
    for _ in range(5):
        F.launch_resize_cv2(*args)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        F.launch_resize_cv2(*args)
    b.record()
    torch.cuda.synchronize()
    nbytes = sum(r.Hs * (2 * r.W * 3 + r.Ws * 3) for r in bank._resize)
    return a.elapsed_time(b) / iters, nbytes


def run(model, cfg, n, bank_name, a):
    sizes = BANKS[bank_name](n)
    scaled = [F.resized_size(H, W, S) for H, W in sizes]
    L = int(cfg.DATA.NUM_FRAMES) * int(cfg.DATA.SAMPLING_RATE)
    rng = np.random.default_rng(n)
    pool = {hw: [torch.from_numpy(rng.integers(0, 256, hw + (3,), dtype=np.uint8)).pin_memory() for _ in range(5)]
            for hw in dict.fromkeys(sizes)}
    device = esf.CameraWindows(model, cfg, n, [h for h, _ in sizes], [w for _, w in sizes], scale_to=S, bgr=True)
    groups = list(dict.fromkeys(scaled))
    members = [[c for c in range(n) if scaled[c] == g] for g in groups]
    host = [esf.CameraWindows(model, cfg, len(m), g[0], g[1]) for g, m in zip(groups, members)]
    # pinned destinations of the host resize, two per camera so that a frame is not overwritten while its copy may
    # still be queued
    out = [[torch.empty(scaled[c] + (3,), dtype=torch.uint8).pin_memory() for _ in range(2)] for c in range(n)]
    rgb = {hw: np.empty(hw + (3,), np.uint8) for hw in pool}
    state = dict(frame=0, host=0)

    def frames():
        state["frame"] += 1
        return {c: pool[sizes[c]][(state["frame"] + 3 * c) % 5] for c in range(n)}

    def tick_host(fr):
        state["host"] += 1
        k = state["host"] % 2
        parts = [{} for _ in host]
        for c, f in fr.items():
            cv2.cvtColor(f.numpy(), cv2.COLOR_BGR2RGB, dst=rgb[sizes[c]])
            h, w = scaled[c]
            cv2.resize(rgb[sizes[c]], (w, h), dst=out[c][k].numpy(), interpolation=cv2.INTER_LINEAR)
            g = groups.index(scaled[c])
            parts[g][members[g].index(c)] = out[c][k]
        res = [b.push(p) for b, p in zip(host, parts)]
        if res[0] is None:
            return None
        ids = [members[g][i] for g, r in enumerate(res) for i in r[0]]
        scores = torch.cat([r[1] for r in res])
        return sorted(ids), scores[torch.tensor([ids.index(c) for c in sorted(ids)], device=scores.device)]

    def tick_device(fr):
        return device.push(fr)

    with torch.no_grad():
        for _ in range(L - 1):
            fr = frames()
            tick_host(fr)
            tick_device(fr)
        fr = frames()
        ref, got = tick_host(fr), tick_device(fr)
        same = dict(bit_identical=bool(ref[0] == got[0] and torch.equal(ref[1], got[1])),
                    argmax_equal=bool(torch.equal(ref[1].argmax(1), got[1].argmax(1))))
        routes = (("host_resize", tick_host), ("device_resize", tick_device))
        spent = {key: [0.0, 0] for key, _ in routes}
        t_end = time.perf_counter() + a.warmup_s
        while time.perf_counter() < t_end:
            for key, fn in routes:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn(frames())
                torch.cuda.synchronize()
                spent[key][0] += time.perf_counter() - t0
                spent[key][1] += 1
        clock = gpu_info().get("clocks.sm")
        ticks = {key: max(a.min_ticks, math.ceil(a.window_s / (sec / cnt))) for key, (sec, cnt) in spent.items()}
        times = {key: [] for key, _ in routes}
        cpu = {key: [] for key, _ in routes}
        for _ in range(a.repeats):
            for key, fn in routes:
                batch = [frames() for _ in range(ticks[key])]
                torch.cuda.synchronize()
                t0, c0 = time.perf_counter(), time.process_time()
                for fr in batch:
                    fn(fr)
                torch.cuda.synchronize()
                times[key].append((time.perf_counter() - t0) / ticks[key])
                cpu[key].append((time.process_time() - c0) / ticks[key])
        k_ms, k_bytes = kernel_time(device, sizes, pool, a.kernel_iters)
    h2d = dict(host_resize=sum(h * w * 3 for h, w in scaled), device_resize=sum(h * w * 3 for h, w in sizes))
    res = dict(cameras=n, bank=bank_name, capture=[list(hw) for hw in dict.fromkeys(sizes)],
               scaled=[list(g) for g in groups], window_frames=L, outputs=same, sm_clock_after_warmup=clock,
               resize_kernel=dict(ms=k_ms, bytes=k_bytes, gb_per_s=k_bytes / k_ms / 1e6))
    for key, ts in times.items():
        res[key] = dict(ticks_per_window=ticks[key], spread=(max(ts) - min(ts)) / min(ts),
                        ms_per_tick=dict(best=1e3 * min(ts), median=1e3 * statistics.median(ts)),
                        camera_frames_per_s=dict(best=n / min(ts), median=n / statistics.median(ts)),
                        host_cpu_s_per_tick=statistics.median(cpu[key]), h2d_bytes_per_tick=h2d[key],
                        all_ms=[1e3 * t for t in ts])
    res["speedup_median"] = statistics.median(times["host_resize"]) / statistics.median(times["device_resize"])
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--models", default="slowfast_8x8_r50,shufflenetv2")
    ap.add_argument("--cameras", default="1,8,32")
    ap.add_argument("--banks", default="720p,1080p,mixed")
    ap.add_argument("--window-s", type=float, default=1.0)
    ap.add_argument("--min-ticks", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--warmup-s", type=float, default=2.0)
    ap.add_argument("--kernel-iters", type=int, default=200)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: nothing here is measured on the CPU")
    cams = [int(v) for v in a.cameras.split(",")]
    res = dict(gpu=gpu_info(), window_s=a.window_s, min_ticks=a.min_ticks, warmup_s=a.warmup_s, repeats=a.repeats,
               precision="fp16", scale_to=S, cv2=cv2.__version__, cv2_threads=cv2.getNumThreads(), results=[])
    for name in a.models.split(","):
        label, cfg, model = build(name, max(cams))
        for bank in a.banks.split(","):
            for n in cams:
                r = run(model, cfg, n, bank, a)
                r.update(model=label)
                res["results"].append(r)
                h, d = r["host_resize"], r["device_resize"]
                print("%s %s N=%d: %.1f -> %.1f camera-frames/s (x%.2f), host CPU %.2f -> %.2f ms/tick, H2D %.2f -> "
                      "%.2f MB/tick, resize kernel %.3f ms (%.0f GB/s), spread %.1f%% / %.1f%%, SM clock %s, %s" % (
                          label, bank, n, h["camera_frames_per_s"]["median"], d["camera_frames_per_s"]["median"],
                          r["speedup_median"], 1e3 * h["host_cpu_s_per_tick"], 1e3 * d["host_cpu_s_per_tick"],
                          h["h2d_bytes_per_tick"] / 1e6, d["h2d_bytes_per_tick"] / 1e6, r["resize_kernel"]["ms"],
                          r["resize_kernel"]["gb_per_s"], 100 * h["spread"], 100 * d["spread"],
                          r["sm_clock_after_warmup"], r["outputs"]), flush=True)
        del model
        torch.cuda.empty_cache()
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
