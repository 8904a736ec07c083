"""The reference's test protocol from whole decoded videos (csrc/esf_crop.cu esf_*_crop_videos behind
model.forward_videos and ClipStream video mode) against the best route before it.

  python tools/bench_frames_videos.py --out profiles/r7_frames_videos.json

Models: SlowFast 4x16 R50 (32 frames at SAMPLING_RATE 2, the YAML's) and Slow 8x8 R50 (8 frames at rate 8), FP16,
random weights.  Videos: 10 s of 256 x 340 uint8 frames, alternately at 30 fps (300 frames) and 25 fps (250 frames),
tested as TEST.NUM_ENSEMBLE_VIEWS 10 x NUM_SPATIAL_CROPS 3 views at TEST_CROP_SIZE 256: 30 rows per video.
  (a) per-view clips: the host samples every temporal view (frames.temporal_index, the reference decoder's
      expressions) into its own pinned uint8 clip (T, 256, 340, 3) and ClipStream runs the list of clips
      (forward_frames on a list, device crops);
  (b) ClipStream video mode: the pinned videos go to the device as they are, one copy each, and forward_videos samples
      the views on the device.
Both stream the same batches of `--videos` videos with the H2D copy overlapped with the forward.  Reported per route:
videos/s from CUDA events over a window of at least `--seconds` (>= 1) seconds, H2D bytes per video, and host
milliseconds per video spent on the host's side of the loader (the temporal sampling copies of (a); (b) has none), and
the host time of the submit calls.  A whole-video upload can be LARGER than the sampled frames: Slow 8x8 reads 80 of
300 frames per video.  The card's name, power limit and clocks are read in the same run.
"""
import argparse
import json
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import efficient_slowfast_b200 as esf  # noqa: E402
from bench_frames_spatial import gpu_info  # noqa: E402
from efficient_slowfast_b200 import frames as FR  # noqa: E402

H, W, C, S = 256, 340, 3, 256
NUM_CLIPS, VIEWS = 10, (0, 1, 2)
SECONDS = 10


def models():
    sf = esf.slowfast_4x16_r50_cfg()
    sf.DATA.SAMPLING_RATE = 2       # SLOWFAST_4x16_R50.yaml
    slow = esf.resnet_cfg("slow")   # SLOW_8x8_R50.yaml: 8 frames at rate 8
    for cfg in (sf, slow):
        cfg.DATA.TEST_CROP_SIZE = S
        cfg.TEST.NUM_ENSEMBLE_VIEWS, cfg.TEST.NUM_SPATIAL_CROPS = NUM_CLIPS, len(VIEWS)
    return {"slowfast_4x16_r50": sf, "slow_8x8_r50": slow}


def video_pool(n, seed):
    """n pinned videos, alternately 10 s at 30 and at 25 fps, and their rates."""
    g = torch.Generator().manual_seed(seed)
    rates = [30.0 if i % 2 == 0 else 25.0 for i in range(n)]
    vids = [torch.randint(0, 256, (int(SECONDS * f), H, W, C), generator=g, dtype=torch.uint8).pin_memory()
            for f in rates]
    return vids, rates


def window(step, seconds):
    """Run step(i) for i = 0, 1, ... until the CUDA-event window on the current stream covers `seconds` seconds (checked
    after every 4 steps); returns (steps, start event, end event) -- the caller records the end after the last batch."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    t0, i = time.perf_counter(), 0
    while True:
        step(i)
        i += 1
        if i % 4 == 0 and time.perf_counter() - t0 >= seconds:
            break
    return i, a, b


def per_view_route(model, cfg, vids, rates, n, seconds):
    T, rate, tfps = int(cfg.DATA.NUM_FRAMES), int(cfg.DATA.SAMPLING_RATE), float(cfg.DATA.TARGET_FPS)
    B = n * NUM_CLIPS
    st = esf.ClipStream(model, [(B, T, H, W, C)], frames=True, crop_size=S, spatial_idx=VIEWS)
    # 3 sets of pinned clips: set i % 3 is refilled only after batch i - 3's copy is known to be done (submit of
    # batch i - 1 waited for it with the stream's depth of 2)
    sets = [[torch.empty((T, H, W, C), dtype=torch.uint8).pin_memory() for _ in range(B)] for _ in range(3)]
    host = {"prep": 0.0, "submit": 0.0}

    def step(i):
        t0 = time.perf_counter()
        clips = sets[i % 3]
        for k in range(n):
            v, f = vids[(i * n + k) % len(vids)], rates[(i * n + k) % len(vids)]
            for j in range(NUM_CLIPS):
                torch.index_select(v, 0, FR.temporal_index(v.shape[0], f, T, rate, tfps, j, NUM_CLIPS),
                                   out=clips[k * NUM_CLIPS + j])
        t1 = time.perf_counter()
        st.submit(clips)
        host["prep"] += t1 - t0
        host["submit"] += time.perf_counter() - t1
    for i in range(3):
        step(i)
    st.flush()
    host.update(prep=0.0, submit=0.0)
    steps, a, b = window(step, seconds)
    st.flush()
    b.record()
    torch.cuda.synchronize()
    sec = a.elapsed_time(b) / 1e3
    return dict(videos_per_s=steps * n / sec, window_s=sec, batches=steps,
                h2d_bytes_per_video=NUM_CLIPS * T * H * W * C,
                host_sampling_ms_per_video=host["prep"] * 1e3 / (steps * n),
                host_submit_ms_per_video=host["submit"] * 1e3 / (steps * n))


def video_route(model, cfg, vids, rates, n, seconds):
    N = max(v.shape[0] for v in vids)
    st = esf.ClipStream(model, [(n, N, H, W, C)], frames=True, num_clips=NUM_CLIPS, crop_size=S, spatial_idx=VIEWS)
    host = {"submit": 0.0}
    uploaded = []

    def step(i):
        batch = [vids[(i * n + k) % len(vids)] for k in range(n)]
        fps = [rates[(i * n + k) % len(vids)] for k in range(n)]
        t0 = time.perf_counter()
        st.submit(batch, fps=fps)
        host["submit"] += time.perf_counter() - t0
        uploaded.append(sum(v.numel() for v in batch))
    for i in range(3):
        step(i)
    st.flush()
    host["submit"], uploaded[:] = 0.0, []
    steps, a, b = window(step, seconds)
    st.flush()
    b.record()
    torch.cuda.synchronize()
    sec = a.elapsed_time(b) / 1e3
    return dict(videos_per_s=steps * n / sec, window_s=sec, batches=steps,
                h2d_bytes_per_video=sum(uploaded) / (steps * n), host_sampling_ms_per_video=0.0,
                host_submit_ms_per_video=host["submit"] * 1e3 / (steps * n))


def check_equal(model, vids, rates, n):
    """Both routes' rows for one batch, compared bit for bit (the same plan runs both)."""
    cfg = model._cfg
    T, rate = int(cfg.DATA.NUM_FRAMES), int(cfg.DATA.SAMPLING_RATE)
    dev = [v.cuda() for v in vids[:n]]
    clips = [v[FR.temporal_index(v.shape[0], f, T, rate, 30.0, j, NUM_CLIPS).cuda()].contiguous()
             for v, f in zip(dev, rates[:n]) for j in range(NUM_CLIPS)]
    a = model.forward_frames(clips, crop_size=S, spatial_idx=VIEWS)
    b = model.forward_videos(dev, fps=rates[:n], crop_size=S)
    return bool(torch.equal(a, b))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--videos", type=int, default=2, help="videos per batch (x 30 rows)")
    ap.add_argument("--seconds", type=float, default=2.0, help="least length of every timed window")
    ap.add_argument("--models", default=None, help="comma-separated subset of the model names")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: nothing here is measured on the CPU")
    if a.seconds < 1:
        raise SystemExit("--seconds: a window under 1 s measures the clock and the scheduler")
    res = dict(gpu=gpu_info(), videos=dict(size=[H, W, C], seconds=SECONDS, fps=[30, 25], num_clips=NUM_CLIPS,
                                           views=list(VIEWS), crop=S, videos_per_batch=a.videos,
                                           rows_per_batch=a.videos * NUM_CLIPS * len(VIEWS)))
    vids, rates = video_pool(4, 7)
    for name, cfg in models().items():
        if a.models and name not in a.models.split(","):
            continue
        model = esf.build_model(cfg).cuda().eval()
        with torch.no_grad():
            r = dict(frames=int(cfg.DATA.NUM_FRAMES), sampling_rate=int(cfg.DATA.SAMPLING_RATE),
                     bit_identical=check_equal(model, vids, rates, a.videos))
            r["a_per_view_clips"] = per_view_route(model, cfg, vids, rates, a.videos, a.seconds)
            r["b_video_mode"] = video_route(model, cfg, vids, rates, a.videos, a.seconds)
        r["h2d_ratio_b_over_a"] = r["b_video_mode"]["h2d_bytes_per_video"] / r["a_per_view_clips"]["h2d_bytes_per_video"]
        res[name] = r
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
