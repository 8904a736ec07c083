"""Test-time spatial sampling on the device (csrc/esf_crop.cu): kernel time and bandwidth, and the end-to-end stream.

  python tools/bench_frames_spatial.py --out profiles/r4_frames_spatial.json

1. Kernel: esf_stem_pack_u8_crop (packed FP16 stem rows) and esf_frames_to_clip_crop (FP32 clip) of the fast pathway,
   B clips of T native 256 x 340 frames -> 3 crops of 224^2, CUDA events over many launches.  Bytes = uint8 frames read
   + output written; GB/s and the share of the 7.7 TB/s HBM3e data-sheet bandwidth of one B200.
2. End to end through ClipStream (H2D copy overlapped with the forward) for the same clips, three inputs:
   native uint8 frames with crop_size / spatial_idx, pre-cropped uint8 frames (B * 3 rows), host-cropped FP32 [slow,
   fast] clips (B * 3 rows, the reference loader's output).
The card's name, power limit and clocks are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import efficient_slowfast_b200 as esf  # noqa: E402
from efficient_slowfast_b200 import frames as FR  # noqa: E402
from efficient_slowfast_b200 import runtime as rt  # noqa: E402
from efficient_slowfast_b200.workloads import case_model_and_weights  # noqa: E402

HBM_PEAK = 7.7e12


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        return dict(zip(q.split(","), [v.strip() for v in r.stdout.splitlines()[0].split(",")]))
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)}


def time_launches(fn, iters):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def bench_kernels(B, T, H0, W0, S, iters):
    cfg, _, _ = case_model_and_weights("slowfast_r50")
    L = rt.lib()
    views = (0, 1, 2)
    fin = FR.FrameInput(cfg, torch.device("cuda"), torch.float16)
    tabs = fin.crop(H0, W0, S, views)
    geo = tabs.pointers() + (tabs.crop_yx, len(views), S)
    frames = torch.randint(0, 256, (B, T, H0, W0, 3), dtype=torch.uint8, device="cuda")
    pitch, lpad, _ = rt.stem_geometry(S, 3, 7, 2, 3)
    xp = torch.empty((B * 3, T, S, pitch), dtype=torch.float16, device="cuda")
    clip = torch.empty((B * 3, 3, T, S, S), dtype=torch.float32, device="cuda")
    s = rt.current_stream_ptr()
    packed = lambda: rt.check(L.esf_stem_pack_u8_crop(  # noqa: E731
        frames.data_ptr(), B, T, H0, W0, 3, None, T, fin.chan_src, fin.lut32.data_ptr(), *geo, rt.F16, pitch, lpad,
        xp.data_ptr(), s))
    fp32 = lambda: rt.check(L.esf_frames_to_clip_crop(  # noqa: E731
        frames.data_ptr(), B, T, H0, W0, 3, None, T, fin.chan_src, fin.lut32.data_ptr(), *geo, clip.data_ptr(), s))
    out = {}
    for name, fn, wbytes in (("stem_pack_u8_crop_fp16", packed, xp.numel() * 2),
                             ("frames_to_clip_crop_fp32", fp32, clip.numel() * 4)):
        ms = time_launches(fn, iters)
        nbytes = frames.numel() + wbytes
        out[name] = dict(ms=ms, read_bytes=frames.numel(), write_bytes=wbytes, gb_per_s=nbytes / ms / 1e6,
                         share_of_hbm_peak=nbytes / (ms * 1e-3) / HBM_PEAK)
    out["geometry"] = dict(B=B, T=T, native=[H0, W0], resized=[tabs.Hr, tabs.Wr], crop=S, views=list(views),
                           working_set_mb=(frames.numel() + xp.numel() * 2) / 2 ** 20)
    return out


def bench_stream(B, T, H0, W0, S, batches):
    cfg, model, _ = case_model_and_weights("slowfast_r50")
    model = model.cuda().eval()
    alpha = cfg.SLOWFAST.ALPHA
    views = (0, 1, 2)
    g = torch.Generator().manual_seed(5)
    native = [torch.randint(0, 256, (B, T, H0, W0, 3), generator=g, dtype=torch.uint8).pin_memory() for _ in range(2)]
    Hr, Wr = FR.resized_size(H0, W0, S)
    offs = [FR.crop_offset(Hr, Wr, S, v) for v in views]
    # pre-cropped uint8: the same geometry cut out of resized frames (the byte values differ from the bilinear result;
    # only the shape matters for the timing)
    small = [n[:, :, :S, :S].repeat_interleave(3, 0).contiguous().pin_memory() for n in native]
    clips = []
    for n in native:
        x = torch.randn(B * 3, 3, T, S, S, generator=g)
        clips.append([x[:, :, torch.linspace(0, T - 1, T // alpha).long()].contiguous().pin_memory(), x.pin_memory()])
    runs = {
        "native_uint8_crop_on_device": (dict(frames=True, crop_size=S, spatial_idx=views), [[n] for n in native],
                                        [tuple(native[0].shape)]),
        "precropped_uint8": (dict(frames=True), [[c] for c in small], [tuple(small[0].shape)]),
        "host_cropped_fp32": (dict(), clips, [tuple(t.shape) for t in clips[0]]),
    }
    out = {}
    with torch.no_grad():
        for name, (kw, data, shapes) in runs.items():
            st = esf.ClipStream(model, shapes, **kw)
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
            out[name] = dict(clips_per_s=batches * B * 3 / dt, ms_per_batch=dt * 1e3 / batches,
                             h2d_bytes_per_batch=st.h2d_bytes)
    out["geometry"] = dict(B=B, T=T, native=[H0, W0], crop=S, views=list(views), rows_per_batch=B * 3,
                           crop_offsets=offs, model="slowfast_r50 (4x16 R50)", precision="fp16")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--kernel-batch", type=int, default=64)
    ap.add_argument("--stream-batch", type=int, default=8)
    ap.add_argument("--batches", type=int, default=30)
    ap.add_argument("--iters", type=int, default=50)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: nothing here is measured on the CPU")
    res = dict(gpu=gpu_info())
    res["kernel"] = bench_kernels(a.kernel_batch, 32, 256, 340, 224, a.iters)
    res["stream"] = bench_stream(a.stream_batch, 32, 256, 340, 224, a.batches)
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
