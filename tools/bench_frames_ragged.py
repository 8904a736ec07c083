"""Test-time crops of clips of mixed decode sizes (csrc/esf_crop.cu esf_*_crop_ragged): kernel time against the uniform
entry points, and the end-to-end stream.

  python tools/bench_frames_ragged.py --out profiles/r6_frames_ragged.json

1. Regression check on a uniform batch (the geometry of bench_frames_spatial: 64 clips x 32 native 256 x 340 frames ->
   3 crops of 224^2, fast pathway): the ragged entry point on the list of the 64 clips against the uniform entry point
   on the stacked batch, packed FP16 rows and FP32 clip, alternating the two, CUDA events over many launches per round.
2. A mixed batch of 64 clips cycling 256 x 340, 256 x 454, 340 x 256, 240 x 320, 360 x 480 and 720 x 1280: one ragged
   call against one uniform call per geometry group (what bucketing by resolution launches), packed FP16 rows.
3. End to end through ClipStream (SlowFast 4x16 R50, 8 windows x 3 crops of 224^2 per batch, H2D overlapped with the
   forward) on a stream of such mixed batches: lists of native uint8 clips cropped on the device, against the host-cropped
   FP32 [slow, fast] clips such a stream has to ship today (the host's resize and crop time is not included), and the
   uniform 256 x 340 stream of bench_frames_spatial for reference.
Every working set is larger than the 126 MB L2.  The card's name, power limit and clocks are read in the same run.
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
from bench_frames_spatial import gpu_info, time_launches  # noqa: E402
from efficient_slowfast_b200 import frames as FR  # noqa: E402
from efficient_slowfast_b200 import runtime as rt  # noqa: E402
from efficient_slowfast_b200.workloads import case_model_and_weights  # noqa: E402

MIXED = [(256, 340), (256, 454), (340, 256), (240, 320), (360, 480), (720, 1280)]
VIEWS = (0, 1, 2)


def frame_input():
    cfg, _, _ = case_model_and_weights("slowfast_r50")
    return FR.FrameInput(cfg, torch.device("cuda"), torch.float16)


def ragged_call(L, fin, clips, S, out, pitch=None, lpad=None):
    """A closure of one esf_*_crop_ragged call over `clips` (device (T, H, W, C) tensors) into `out`."""
    batch = FR.ClipList(clips, [fin.crop(c.shape[1], c.shape[2], S, VIEWS) for c in clips])
    T = batch.T
    args = (batch.frames, batch.B, T, 3, None, T, fin.chan_src, fin.lut32.data_ptr(), batch.geom, batch.tables,
            batch.crop_yx, batch.V, S)
    s = rt.current_stream_ptr()
    if pitch is None:
        return lambda: rt.check(L.esf_frames_to_clip_crop_ragged(*args, out.data_ptr(), s))
    return lambda: rt.check(L.esf_stem_pack_u8_crop_ragged(*args, rt.F16, pitch, lpad, out.data_ptr(), s))


def uniform_call(L, fin, frames, S, out, pitch=None, lpad=None):
    """A closure of one esf_*_crop call over the stacked `frames` (B, T, H, W, C) into `out`."""
    B, T, H0, W0, _ = frames.shape
    tabs = fin.crop(H0, W0, S, VIEWS)
    geo = tabs.pointers() + (tabs.crop_yx, len(VIEWS), S)
    s = rt.current_stream_ptr()
    if pitch is None:
        return lambda: rt.check(L.esf_frames_to_clip_crop(frames.data_ptr(), B, T, H0, W0, 3, None, T, fin.chan_src,
                                                          fin.lut32.data_ptr(), *geo, out.data_ptr(), s))
    return lambda: rt.check(L.esf_stem_pack_u8_crop(frames.data_ptr(), B, T, H0, W0, 3, None, T, fin.chan_src,
                                                    fin.lut32.data_ptr(), *geo, rt.F16, pitch, lpad, out.data_ptr(), s))


def alternate(fns, iters, rounds):
    """{name: per-round ms} of the closures in `fns`, timed one after the other in every round."""
    ms = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            ms[k].append(time_launches(fn, iters))
    return {k: dict(ms_rounds=v, ms_min=min(v), ms_median=statistics.median(v), spread=(max(v) - min(v)) / min(v))
            for k, v in ms.items()}


def bench_uniform(B, T, S, iters, rounds):
    L, fin = rt.lib(), frame_input()
    frames = torch.randint(0, 256, (B, T, 256, 340, 3), dtype=torch.uint8, device="cuda")
    pitch, lpad, _ = rt.stem_geometry(S, 3, 7, 2, 3)
    xp = torch.empty((B * 3, T, S, pitch), dtype=torch.float16, device="cuda")
    clip = torch.empty((B * 3, 3, T, S, S), dtype=torch.float32, device="cuda")
    fns = {"uniform_fp16": uniform_call(L, fin, frames, S, xp, pitch, lpad),
           "ragged_fp16": ragged_call(L, fin, list(frames), S, xp, pitch, lpad),
           "uniform_fp32": uniform_call(L, fin, frames, S, clip),
           "ragged_fp32": ragged_call(L, fin, list(frames), S, clip)}
    # the two routes write the same bytes
    fns["uniform_fp16"]()
    ref = xp.clone()
    fns["ragged_fp16"]()
    torch.cuda.synchronize()
    out = alternate(fns, iters, rounds)
    out["bit_identical_fp16"] = bool(torch.equal(ref.view(torch.int16), xp.view(torch.int16)))
    out["geometry"] = dict(B=B, T=T, native=[256, 340], crop=S, views=list(VIEWS), read_mb=frames.numel() / 2 ** 20)
    return out


def bench_mixed(B, T, S, iters, rounds):
    L, fin = rt.lib(), frame_input()
    sizes = [MIXED[i % len(MIXED)] for i in range(B)]
    groups = {hw: torch.randint(0, 256, (sizes.count(hw), T) + hw + (3,), dtype=torch.uint8, device="cuda")
              for hw in MIXED}
    clips = [c for hw in MIXED for c in groups[hw]]
    pitch, lpad, _ = rt.stem_geometry(S, 3, 7, 2, 3)
    xp = torch.empty((B * 3, T, S, pitch), dtype=torch.float16, device="cuda")
    calls, row = [], 0
    for hw in MIXED:
        n = groups[hw].shape[0]
        calls.append(uniform_call(L, fin, groups[hw], S, xp[row:row + 3 * n], pitch, lpad))
        row += 3 * n

    def per_group():
        for c in calls:
            c()
    out = alternate({"ragged_one_call_fp16": ragged_call(L, fin, clips, S, xp, pitch, lpad),
                     "uniform_call_per_group_fp16": per_group}, iters, rounds)
    out["geometry"] = dict(B=B, T=T, native=[list(hw) for hw in MIXED], clips_per_geometry=[sizes.count(hw) for hw in MIXED],
                           crop=S, views=list(VIEWS), read_mb=sum(c.numel() for c in clips) / 2 ** 20,
                           uniform_launches=len(MIXED))
    return out


def run_stream(st, data, batches, rows):
    for i in range(4):                                     # warm-up: plan, graph, staging
        st.submit(data[i % len(data)])
    st.flush()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(batches):
        st.submit(data[i % len(data)])
    st.flush()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return dict(clips_per_s=batches * rows / dt, ms_per_batch=dt * 1e3 / batches)


def bench_stream(B, T, S, batches):
    cfg, model, _ = case_model_and_weights("slowfast_r50")
    model = model.cuda().eval()
    alpha = cfg.SLOWFAST.ALPHA
    g = torch.Generator().manual_seed(6)
    mixed = []
    for k in range(len(MIXED)):        # batch k starts the geometry cycle at k: every batch holds another mix
        sizes = [MIXED[(k + i) % len(MIXED)] for i in range(B)]
        mixed.append([torch.randint(0, 256, (T,) + hw + (3,), generator=g, dtype=torch.uint8).pin_memory()
                      for hw in sizes])
    cap = max(FR.arena_layout([tuple(c.shape) for c in b])[1] for b in mixed)
    H = -(-cap // (B * T * 1280 * 3))                      # staging (B, T, H, 1280, 3) of at least `cap` bytes
    uniform = [torch.randint(0, 256, (B, T, 256, 340, 3), generator=g, dtype=torch.uint8).pin_memory() for _ in range(2)]
    clips = []
    for _ in range(2):
        x = torch.randn(B * 3, 3, T, S, S, generator=g)
        clips.append([x[:, :, torch.linspace(0, T - 1, T // alpha).long()].contiguous().pin_memory(), x.pin_memory()])
    crop = dict(frames=True, crop_size=S, spatial_idx=VIEWS)
    out = {}
    with torch.no_grad():
        st = esf.ClipStream(model, [(B, T, H, 1280, 3)], **crop)
        out["mixed_native_uint8_crop_on_device"] = run_stream(st, mixed, batches, B * 3)
        out["mixed_native_uint8_crop_on_device"]["h2d_bytes_per_batch_mean"] = \
            statistics.mean(sum(c.numel() for c in b) for b in mixed)
        del st
        st = esf.ClipStream(model, [tuple(t.shape) for t in clips[0]])
        out["host_cropped_fp32"] = run_stream(st, clips, batches, B * 3)
        out["host_cropped_fp32"]["h2d_bytes_per_batch"] = st.h2d_bytes
        del st
        st = esf.ClipStream(model, [tuple(uniform[0].shape)], **crop)
        out["uniform_256x340_native_uint8_crop_on_device"] = run_stream(st, [[u] for u in uniform], batches, B * 3)
    out["geometry"] = dict(B=B, T=T, native=[list(hw) for hw in MIXED], crop=S, views=list(VIEWS), rows_per_batch=B * 3,
                           staging_shape=[B, T, H, 1280, 3], model="slowfast_r50 (4x16 R50)", precision="fp16")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--kernel-batch", type=int, default=64)
    ap.add_argument("--stream-batch", type=int, default=8)
    ap.add_argument("--batches", type=int, default=30)
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: nothing here is measured on the CPU")
    res = dict(gpu=gpu_info())
    res["uniform_batch"] = bench_uniform(a.kernel_batch, 32, 224, a.iters, a.rounds)
    res["mixed_batch"] = bench_mixed(a.kernel_batch, 32, 224, a.iters, a.rounds)
    torch.cuda.empty_cache()
    res["stream"] = bench_stream(a.stream_batch, 32, 224, a.batches)
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
