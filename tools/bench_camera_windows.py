"""The demo loop over N cameras: N SlidingWindows (one batch-1 forward per camera per frame tick) against one
CameraWindows (one forward of N rows per tick, gathered from the per-camera rings on the device).

  python tools/bench_camera_windows.py --out profiles/r10_camera_windows.json

Models: SlowFast 8x8 R50 (32 frames, ALPHA 4, SAMPLING_RATE 2: a 64-frame window) and SlowFast-ShuffleNetV2 1.0x
(16 frames, ALPHA 4, SAMPLING_RATE 4), FP16, seeded weights.  Frames: a square and a 16:9 demo size (the caller's
cv2.resize output), uint8 in pinned host memory, one new frame per camera per tick.  Every model runs with
cfg.ESF.MAX_BATCH = max(N), so the batch-1 forwards of the SlidingWindows and the N-row forward of the bank come from
one plan family per frame size.  For each (model, size, N): both routes are warmed up, alternating, for at least
`--warmup-s` seconds (which also brings the SM clock up from idle; the clock read after the warm-up is recorded), then
timed in windows of at least `--window-s` seconds and `--min-ticks` ticks each (the tick count comes from the warm-up's
time per tick), the two routes alternated `--repeats` times; a window is timed on the host clock from its first push to
a device synchronise after its last forward.  Reported: camera-frames per second (N * ticks / time) and milliseconds per tick,
best and median window; which stem route the frame size took (packed 16-bit rows or the FP32 clip of the CUDA-core
stem fallback); and whether the bank's rows were bit-identical to the SlidingWindows' outputs, with their argmax.
The card's name, power limit and clocks are read in the same run.
"""
import argparse
import json
import math
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


def build(name, capacity):
    """(label, cfg, model on the GPU with MAX_BATCH = capacity, seeded weights)."""
    if name == "slowfast_8x8_r50":
        cfg = esf.slowfast_4x16_r50_cfg()
        cfg.DATA.NUM_FRAMES, cfg.DATA.SAMPLING_RATE, cfg.SLOWFAST.ALPHA = 32, 2, 4
        cfg.MULTIGRID.SHORT_CYCLE = True          # global average pool: the head takes any frame size
        label = "SlowFast 8x8 R50"
    else:
        cfg = esf.slowfast_shufflenetv2_cfg(1.0)
        cfg.DATA.SAMPLING_RATE = 4
        label = "SlowFast-ShuffleNetV2 1.0x"
    cfg.NUM_GPUS = 0
    cfg.ESF.MAX_BATCH = capacity
    torch.manual_seed(0)
    model = esf.build_model(cfg)
    model.load_state_dict(W.seeded_state_dict(model.state_dict(), seed=0), strict=True)
    return label, cfg, model.cuda().eval()


def route_of(model, rows):
    cap = next(reversed(model._plans.values()))[1]
    plan = cap.variants.get(rows, cap)
    return ["packed16" if own.data_ptr() in plan.stem_routes else "fp32_clip" for own in plan.inputs]


def run(model, cfg, n, H, Wd, a):
    L = int(cfg.DATA.NUM_FRAMES) * int(cfg.DATA.SAMPLING_RATE)
    g = torch.Generator().manual_seed(n)
    pool = [torch.randint(0, 256, (H, Wd, 3), generator=g, dtype=torch.uint8).pin_memory() for _ in range(7)]
    singles = [esf.SlidingWindow(model, cfg, H, Wd) for _ in range(n)]
    bank = esf.CameraWindows(model, cfg, n, H, Wd)
    state = dict(frame=0)

    def frames():
        state["frame"] += 1
        return {c: pool[(state["frame"] + 3 * c) % len(pool)] for c in range(n)}

    def tick_singles(fr):
        return [singles[c].push(fr[c]) for c in range(n)]

    def tick_bank(fr):
        return bank.push(fr)

    with torch.no_grad():
        for _ in range(L - 1):                       # fill every window, no forward yet
            fr = frames()
            tick_singles(fr)
            tick_bank(fr)
        fr = frames()
        ys = tick_singles(fr)
        ids, scores = tick_bank(fr)
        ref = torch.cat(ys)
        same = dict(bit_identical=bool(torch.equal(ref, scores)),
                    argmax_equal=bool(torch.equal(ref.argmax(1), scores.argmax(1))),
                    max_abs_diff=float((ref - scores).abs().max()))
        routes = (("sliding_windows", tick_singles), ("camera_windows", tick_bank))
        spent = {key: [0.0, 0] for key, _ in routes}        # warm-up seconds and ticks per route
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
        for _ in range(a.repeats):
            for key, fn in routes:
                batch = [frames() for _ in range(ticks[key])]
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for fr in batch:
                    fn(fr)
                torch.cuda.synchronize()
                times[key].append((time.perf_counter() - t0) / ticks[key])
    out = dict(cameras=n, window_frames=L, route=route_of(model, n), outputs=same, sm_clock_after_warmup=clock)
    for key, ts in times.items():
        out[key] = dict(ticks_per_window=ticks[key], spread=(max(ts) - min(ts)) / min(ts),
                        ms_per_tick=dict(best=1e3 * min(ts), median=1e3 * statistics.median(ts)),
                        camera_frames_per_s=dict(best=n / min(ts), median=n / statistics.median(ts)),
                        all_ms=[1e3 * t for t in ts])
    out["speedup_median"] = statistics.median(times["sliding_windows"]) / statistics.median(times["camera_windows"])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--models", default="slowfast_8x8_r50,shufflenetv2")
    ap.add_argument("--cameras", default="1,4,16,32")
    ap.add_argument("--sizes", default="224x224,224x398")
    ap.add_argument("--window-s", type=float, default=1.0)
    ap.add_argument("--min-ticks", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--warmup-s", type=float, default=2.0)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: nothing here is measured on the CPU")
    cams = [int(v) for v in a.cameras.split(",")]
    sizes = [tuple(int(v) for v in s.split("x")) for s in a.sizes.split(",")]
    res = dict(gpu=gpu_info(), window_s=a.window_s, min_ticks=a.min_ticks, warmup_s=a.warmup_s, repeats=a.repeats,
               precision="fp16", results=[])
    for name in a.models.split(","):
        label, cfg, model = build(name, max(cams))
        for H, Wd in sizes:
            for n in cams:
                r = run(model, cfg, n, H, Wd, a)
                r.update(model=label, frame=[H, Wd])
                res["results"].append(r)
                sw, cw = r["sliding_windows"], r["camera_windows"]
                print("%s %dx%d N=%d route %s: %.1f -> %.1f camera-frames/s (x%.2f), %.2f -> %.2f ms/tick, spread "
                      "%.1f%% / %.1f%%, SM clock %s, %s" % (
                          label, H, Wd, n, r["route"], sw["camera_frames_per_s"]["median"],
                          cw["camera_frames_per_s"]["median"], r["speedup_median"], sw["ms_per_tick"]["median"],
                          cw["ms_per_tick"]["median"], 100 * sw["spread"], 100 * cw["spread"],
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
