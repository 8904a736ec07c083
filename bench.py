#!/usr/bin/env python
"""Headline benchmark: clips/sec of the SlowFastDualAttention (CMDA) 8x8 R50 forward, batch 64 per GPU, 224^2
synthetic clips (BASELINE.json configs[2]), one process per GPU, no collective inside the forward and one NCCL
all-gather of the logits per step.

    python bench.py --gpus 1 --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host CPU (oracle port)
    python bench.py ... --dump-outputs DIR                   # + DIR/probs.npy: what the last timed step returned
    torchrun ... bench.py --gpus N ...                       # N > 1, weak scaling (64 clips per GPU)

Prints ONE JSON line (contract in the task statement): value = whole-job clips/s with inputs resident in HBM,
e2e = the same through model.forward() with pinned-host inputs (H2D of the step's clips and D2H of its
probabilities inside the timed region), roofline = the dominant kernel against the measured B200 peaks,
cpu_baseline = the oracle timed on this box's host cores on a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "clips/sec SlowFast-DA 8x8 R50 fwd"
UNIT = "clips/s"
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "sm_max_mhz": 1965.0}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        d["_source"] = "measured"
        return d
    d = dict(FALLBACK_PEAKS)
    d["_source"] = "fallback"
    return d


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms",
                 "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.proc.wait()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# --model -> golden case that carries its calibrated BN statistics (tests/golden/recipe.py CASES).  The default is the
# headline workload; the others are BASELINE.json's remaining configs, benchmarked with explicit --batch/--frames/--crop.
MODEL_CASES = {
    "SlowFastDualAttention": "dual_r50", "SlowFast": "slowfast_r50", "SlowFastShuffleNetV2": "shufflenetv2_w05",
    "SlowFastShuffleNet": "shufflenet_w2g3", "SlowFastMoibleNetV2": "mobilenetv2_w1", "SlowFastGhostNet": "ghostnet_w1",
}


def case_of(args_or_cfg):
    return getattr(args_or_cfg, "case", None) or MODEL_CASES[args_or_cfg.model]


def bench_cfg(args):
    from efficient_slowfast_b200 import workloads as helpers

    cfg = helpers.case_cfg(case_of(args))
    cfg.ESF.BENCH_CASE = case_of(args)
    cfg.NUM_GPUS = 1
    cfg.DATA.CROP_SIZE = args.crop
    cfg.DATA.NUM_FRAMES = args.frames
    cfg.ESF.PRECISION = args.precision
    return cfg


def build_weights(cfg):
    """Random-init weights of the named architecture, made non-degenerate with the parity recipe (gamma != 0, final
    BN != 0; BN statistics calibrated offline by the reference and shipped as a test fixture)."""
    import efficient_slowfast_b200 as esf
    from efficient_slowfast_b200 import workloads as helpers
    from efficient_slowfast_b200 import workloads as recipe

    name = cfg.ESF.get("BENCH_CASE") or MODEL_CASES[cfg.MODEL.MODEL_NAME]
    c = cfg.clone()
    c.NUM_GPUS = 0
    torch.manual_seed(0)
    model = esf.build_model(c)
    gold = helpers.load_golden(name)
    bn = {k[3:]: v for k, v in gold.items() if k.startswith("bn/")}
    model.load_state_dict(recipe.seeded_state_dict(model.state_dict(), seed=0, bn_stats=bn), strict=True)
    return model.eval()


def metric_name(args):
    if args.case:
        return "clips/sec %s fwd" % args.case
    return METRIC if args.model == "SlowFastDualAttention" else "clips/sec %s fwd" % args.model


def workload_name(args):
    if args.alpha == 0:
        return "%s (single pathway) %dx%dx%dx%d fwd, batch %d per GPU, synthetic N(0,1) clips" % (
            args.case, args.batch, args.frames, args.crop, args.crop, args.batch)
    return "%s %dx(%d|%d)x%dx%d fwd, batch %d per GPU, synthetic N(0,1) clips" % (
        args.model + (" R50" if args.model in ("SlowFast", "SlowFastDualAttention") else ""), args.batch, args.frames // args.alpha, args.frames, args.crop, args.crop, args.batch)


# ------------------------------------------------------------------------------------------------ CPU arms
def cpu_forward_timed(cfg, model, clips, frames, crop, alpha, steps, warmup):
    """Times the CPU oracle (restatement of the reference forward) on `clips` clips per step, all host threads."""
    from efficient_slowfast_b200 import workloads as recipe
    from oracle import slowfast_oracle as O

    torch.set_num_threads(os.cpu_count() or 1)
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    xs = recipe.pack_pathway_output(recipe.seeded_clip(clips, frames, crop, seed=1), alpha)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        y = O.forward(cfg, sd, xs)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return clips * len(times) / sum(times), sum(times) / len(times), y


def dump_outputs(dirname, probs):
    """Writes the class probabilities of the last timed step as dirname/probs.npy (float32), so that two builds run
    with the same arguments (hence the same seeded weights and clips) can be compared output for output.  Above 64 MB
    only a fixed, seeded sample of the rows is written."""
    import numpy as np

    a = probs.detach().float().cpu()
    limit = 64 << 20
    if a.numel() * 4 > limit:
        keep = limit // (4 * a[0].numel())
        a = a[torch.randperm(a.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values]
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "probs.npy"), a.numpy())


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = bench_cfg(args)
    model = build_weights(cfg)
    clips = args.cpu_clips
    t_start = time.time()
    value, sec, probs = cpu_forward_timed(cfg, model, clips, args.frames, args.crop, args.alpha, args.steps, args.warmup)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, probs)
    cores = torch.get_num_threads()
    sample = "%d clip(s) of the workload per step (same shape, CPU FP32 oracle port of the reference forward)" % clips
    line = {
        "impl": "reference", "metric": metric_name(args), "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args), "cpu_sample_clips_per_step": clips},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.time() - t_start,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ GPU arm
# BASELINE.json's other configs, run for a few steps each after the headline when N = 1 (`configs` in the JSON line):
# (key, model, batch, frames, crop).  configs[0] is the reference's CPU-runnable case; it is run here on the GPU at a
# batch that fills it.  GhostNet at batch 128 falls back to a smaller batch only if the arena does not fit (reason kept).
EXTRA_CONFIGS = [
    ("cfg1_shufflenetv2_w0.5", "SlowFastShuffleNetV2", 64, 32, 224),
    ("cfg2_slowfast_4x16_r50", "SlowFast", 32, 32, 224),
    ("cfg4a_ghostnet_w1.0", "SlowFastGhostNet", 128, 32, 224),
    ("cfg4b_mobilenetv2_w1.0", "SlowFastMoibleNetV2", 128, 32, 224),
    ("cfg5_shufflenet_w2.0_g3", "SlowFastShuffleNet", 256, 16, 112),
]


def golden_for(case, frames, crop):
    """(tag, batch) of the reference-generated golden of `case` whose clip has this shape, or None."""
    from efficient_slowfast_b200 import workloads as W

    for tag, b, f, c in W.CASES[case]["inputs"]:
        if f == frames and c == crop:
            return tag, b
    return None


def fill_inputs(ins, alpha, rank, dev):
    """Synthetic N(0,1) clips into the plan's static inputs: the fast clip is drawn, the slow one is its frame subset."""
    from efficient_slowfast_b200 import workloads as W

    g = torch.Generator(device=dev).manual_seed(1 + rank)
    ins[-1].normal_(generator=g)
    if alpha:
        ins[0].copy_(W.pack_pathway_output(ins[1], alpha)[0])


def parity_check(model, ins, case, frames, crop, alpha, tol=2e-2):
    """OUTSIDE the timed region: the golden clip of this shape (made by the reference, tests/golden) goes into the
    first and the last batch slots of the benched static input; both output rows must match the golden (<= 2e-2, the
    north star's 16-bit tolerance) and each other bit-exactly -- the benched batch size, plan and index paths are the
    ones being checked.  The slots are refilled with the synthetic clips afterwards."""
    from efficient_slowfast_b200 import workloads as W

    g = golden_for(case, frames, crop)
    if g is None:
        return {"skipped": "no reference golden of shape %dx%d^2 for %s" % (frames, crop, case)}
    tag, gb = g
    B = ins[0].shape[0]
    if B < gb:
        return {"skipped": "batch %d smaller than the golden's %d" % (B, gb)}
    gold = W.load_golden(case)
    xs = W.pack_pathway_output(W.seeded_clip(gb, frames, crop, seed=1), alpha)
    saved = [(t[:gb].clone(), t[B - gb:].clone()) for t in ins]
    for t, x in zip(ins, xs):
        t[:gb].copy_(x)
        t[B - gb:].copy_(x)
    with torch.no_grad():
        y = model(ins).float().cpu()
    torch.cuda.synchronize()
    for t, (a, b) in zip(ins, saved):
        t[:gb].copy_(a)
        t[B - gb:].copy_(b)
    ref = torch.as_tensor(gold[tag + "/probs"])
    first, last = y[:gb], y[B - gb:]
    err = max(W.rel_err(first, ref), W.rel_err(last, ref))
    same = bool(torch.equal(first, last))
    argmax_ok = bool(torch.equal(first.argmax(1), ref.argmax(1)) and torch.equal(last.argmax(1), ref.argmax(1)))
    ok = err <= tol and same
    return {"golden": "%s/%s" % (case, tag), "rows": [0, B - gb] if gb == 1 else [[0, gb - 1], [B - gb, B - 1]],
            "batch": B, "rel_err": err, "tol": tol, "first_equals_last_bitwise": same, "argmax_equal": argmax_ok,
            "ok": ok}


def ncu_traffic(label, batch):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the dominant kernel, from the committed
    summaries of `ncu --set full` captures (profiles/ncu_traffic.json, written by tools/ncu_summary.py --traffic)."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return None, None
    for e in json.load(open(p)):
        if e.get("label") == label and e.get("batch") == batch:
            return e["dram_bytes_read"] + e["dram_bytes_write"], e.get("source")
    return None, None


class Harness:
    def __init__(self, args):
        import torch.distributed as dist

        from efficient_slowfast_b200 import distributed as esf_dist

        self.dist, self.esf_dist = dist, esf_dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.affinity0 = os.sched_getaffinity(0)
        # pinned clip buffers must live on the GPU's own NUMA node (efficient_slowfast_b200/distributed.py)
        self.numa = esf_dist.bind_to_gpu_numa_node(self.local_rank) if not args.no_numa_bind else {"skipped": "flag"}
        if self.world > 1:
            # NCCL writes its version banner to stdout, next to the ONE JSON line of the contract: send it to stderr
            os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
            dist.init_process_group("nccl", device_id=self.dev)
        assert self.world == args.gpus or self.world == 1, "launch with torchrun --nproc-per-node %d" % args.gpus

    def barrier(self):
        torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def timed(self, fn, steps):
        """ms for `steps` calls of fn: barrier + synchronize on both sides, CUDA events, max over ranks."""
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(ms, op=self.dist.ReduceOp.MAX)
        return float(ms.item())


def setup_workload(h, args):
    from efficient_slowfast_b200 import runtime as rt

    rt.lib()  # fails loudly when the CUDA extension is missing
    cfg = bench_cfg(args)
    if args.profile_mode:
        cfg.ESF.CUDA_GRAPH = False
    model = build_weights(cfg).to(h.dev)
    B, T, S, alpha = args.batch, args.frames, args.crop, args.alpha
    shapes = [(B, 3, T // alpha, S, S), (B, 3, T, S, S)] if alpha else [(B, 3, T, S, S)]
    ins = model.input_buffers(shapes, h.dev)          # plan-owned static inputs (the CUDA graph reads these)
    plan = model._get_plan(shapes, h.dev)
    fill_inputs(ins, alpha, h.rank, h.dev)
    return cfg, model, shapes, ins, plan


def run_extra_config(h, base_args, key, model_name, batch, frames, crop):
    """One of BASELINE.json's other configs: parity check at the benched batch, >= 1 s of timed steps with clocks."""
    a = argparse.Namespace(**vars(base_args))
    a.model, a.case, a.batch, a.frames, a.crop = model_name, "", batch, frames, crop
    a.alpha = 8 if model_name == "SlowFast" else 4
    a.profile_mode = False
    note = None
    while True:
        try:
            cfg, model, shapes, ins, plan = setup_workload(h, a)
            break
        except torch.cuda.OutOfMemoryError:
            note = "batch %d does not fit 180 GB (activation arena of one plan); halved" % a.batch
            model = plan = ins = None
            torch.cuda.empty_cache()
            if a.batch <= 8:
                return {"error": note}
            a.batch //= 2
    step = lambda: model(ins)
    par = parity_check(model, ins, case_of(a), frames, crop, a.alpha)
    for _ in range(3):
        step()
    est = h.timed(step, 2) / 2
    steps = max(5, int(1000.0 / max(est, 1e-3)) + 1)
    sampler = ClockSampler(h.local_rank)
    sampler.start()
    try:
        ms = h.timed(step, steps)
    finally:
        clocks = sampler.stop()
    out = {"workload": workload_name(a), "value": a.batch * steps / (ms * 1e-3), "unit": UNIT, "steps": steps, "warmup": 5,
           "ms_per_step": ms / steps, "batch": a.batch, "launches_per_step": plan.launches_per_run,
           "arena_gb": round(plan.arena_bytes() / 1e9, 2), "clocks": clocks, "parity_check": par}
    if note:
        out["note"] = note
    del model, plan, ins
    torch.cuda.empty_cache()
    return out


def h2d_ceiling(h, nbytes, iters=6):
    """What the box's host-to-device path gives THIS job layout: every rank copies `nbytes` from pinned host memory to
    its GPU `iters` times, all ranks at once; aggregate GB/s over the slowest rank."""
    host = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    dst = torch.empty(nbytes, dtype=torch.uint8, device=h.dev)
    dst.copy_(host, non_blocking=True)
    ms = h.timed(lambda: dst.copy_(host, non_blocking=True), iters)
    return h.world * nbytes * iters / (ms * 1e-3) / 1e9


def run_gpu(args):
    from efficient_slowfast_b200 import ClipStream
    from efficient_slowfast_b200 import workloads as recipe

    h = Harness(args)
    world, rank, dev, dist = h.world, h.rank, h.dev, h.dist
    cfg, model, shapes, ins, plan = setup_workload(h, args)
    B, T, S, alpha = args.batch, args.frames, args.crop, args.alpha
    K = cfg.MODEL.NUM_CLASSES

    last = {}                                       # what the latest step returned, for --dump-outputs

    def step():
        out = model(ins)                            # graph replay; no staging copy (inputs are the static buffers)
        if world > 1:
            out = h.esf_dist.all_gather([out])[0]   # the only collective on the path (tools/test_net.py:95-98)
        last["probs"] = out
        return out

    if args.profile_mode:
        step()
        torch.cuda.synchronize()
        for _ in range(args.steps):
            step()
        torch.cuda.synchronize()
        print(json.dumps({"profile_mode": True, "launches_per_step": plan.launches_per_run}))
        return
    # north star: <= 2e-2 on the 16-bit path, <= 1e-4 on the FP32 path (2e-4 written for 224^2 clips, DESIGN.md 3.8)
    parity = parity_check(model, ins, case_of(args), T, S, alpha,
                          tol=2e-4 if args.precision == "fp32" else 2e-2) if rank == 0 else None
    for _ in range(max(args.warmup, 3)):
        step()
    sampler = ClockSampler(h.local_rank)
    if rank == 0:
        sampler.start()
    try:
        ms_total = h.timed(step, args.steps)
    finally:                                        # the sampler's nvidia-smi must not outlive a failed step
        clocks = sampler.stop() if rank == 0 else None
    value = world * B * args.steps / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last["probs"])

    # ---- end-to-end through the public API with pinned host inputs (H2D + forward + D2H per step)
    # ClipStream = the package's public host-side loop: per batch H2D from pinned memory -> model.forward ->
    # (all_gather) -> D2H, with the copy of batch i+1 overlapping the forward of batch i.  The caller hands over the
    # reference loader's [slow, fast] pair; slow_from_fast=True (verified on the first batch) uploads the fast clip only
    # and the slow pathway reads its frames out of it -- `e2e_both_pathways_uploaded` is the same loop without that.
    host = [torch.empty(s, dtype=torch.float32).pin_memory() for s in shapes]
    host[-1].normal_()
    if alpha:
        host[0].copy_(recipe.pack_pathway_output(host[1], alpha)[0])
    # the loop is a pipeline: its fill (first copy) and drain (last forward) cost one extra step in total, so it is
    # timed over at least 30 batches -- a test run streams thousands
    e2e_steps = max(2, args.e2e_steps if args.e2e_steps > 0 else max(args.steps, 30))

    def e2e_measure(**kw):
        stream = ClipStream(model, shapes, dev, depth=args.e2e_depth, gather=world > 1, **kw)

        def run():
            got = 0
            for _ in range(e2e_steps):
                got += stream.submit(host) is not None
            got += len(stream.flush())
            assert got == e2e_steps

        stream.submit(host)
        stream.flush()
        ms = h.timed(run, 1)
        return {"value": world * B * e2e_steps / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": stream.h2d_bytes,
                "d2h_bytes_per_step": B * K * 4 * world, "steps": e2e_steps, "ms_per_step": ms / e2e_steps}

    e2e = e2e_measure(slow_from_fast=bool(alpha) and hasattr(model, "forward_fast"))
    e2e["input"] = "pinned FP32 [slow, fast] host clips; the fast clip is copied, slow = its frame subset (verified)" \
        if alpha else "pinned FP32 host clip"
    e2e_both = e2e_measure() if alpha else None
    ceiling = h2d_ceiling(h, e2e["h2d_bytes_per_step"])
    e2e["h2d_ceiling_gbs"] = ceiling
    e2e["h2d_achieved_gbs"] = world * e2e["h2d_bytes_per_step"] / (e2e["ms_per_step"] * 1e-3) / 1e9
    e2e["h2d_frac_of_ceiling"] = e2e["h2d_achieved_gbs"] / ceiling
    e2e["bound"] = "host-to-device copies (all ranks share the host's PCIe / memory path)" \
        if e2e["h2d_frac_of_ceiling"] > 0.85 else "forward"
    e2e["numa_bind"] = h.numa

    # ---- the same loop fed with the decoder's uint8 frames (SURVEY 8-f4): model.forward_frames does the reference
    # loader's normalisation + pathway packing on the device; extra information, `e2e` above stays the FP32 contract
    e2e_u8 = None
    if hasattr(model, "forward_frames"):
        fshape = (B, T, S, S, 3)
        hostf = torch.randint(0, 256, fshape, dtype=torch.uint8).pin_memory()
        fstream = ClipStream(model, [fshape], dev, depth=2, gather=world > 1, frames=True)

        def e2e_frames_run():
            got = 0
            for _ in range(e2e_steps):
                got += fstream.submit([hostf]) is not None
            got += len(fstream.flush())
            assert got == e2e_steps

        fstream.submit([hostf])
        fstream.flush()
        ms_u8 = h.timed(e2e_frames_run, 1)
        e2e_u8 = {"value": world * B * e2e_steps / (ms_u8 * 1e-3), "unit": UNIT, "h2d_bytes_per_step": fstream.h2d_bytes,
                  "d2h_bytes_per_step": B * K * 4 * world, "steps": e2e_steps, "ms_per_step": ms_u8 / e2e_steps,
                  "input": "uint8 frames (B,T,H,W,C) through model.forward_frames"}
        del fstream, hostf
    del host

    # ---- per-kernel device times (CUDA events, eager launches of the same plan) and the roofline of the top kernel
    pk = peaks()
    times = plan.profile_ops(repeats=2)
    total_ms = sum(times)
    kinds = {}
    for t, m in zip(times, plan.meta):
        k = kinds.setdefault(m["kind"], dict(ms=0.0, flops=0.0, bytes=0.0, exps=0.0, launches=0))
        k["ms"] += t
        k["flops"] += m["flops"]
        k["bytes"] += m["bytes"]
        k["exps"] += m["exps"]
        k["launches"] += m["launches"]
    if args.dump_ops and rank == 0:
        with open(args.dump_ops, "w") as fh:
            for t, m in zip(times, plan.meta):
                fh.write(json.dumps(dict(ms=round(t, 4), **m)) + "\n")
    top_i = max(range(len(times)), key=lambda i: times[i])
    top, top_ms = plan.meta[top_i], times[top_i]
    tensor_peak = pk.get("bf16_tflops", FALLBACK_PEAKS["bf16_tflops"])       # burst figure: kernel timed alone
    if top["kind"] in ("conv_igemm", "attention", "stem_igemm"):
        ach = top["flops"] / (top_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "achieved": ach, "peak": tensor_peak, "unit": "TFLOP/s", "frac": ach / tensor_peak}
    else:
        ach = top["bytes"] / (top_ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"]}
    traffic, traffic_src = ncu_traffic("%s %s" % (top["kind"], top["label"]), B)
    roof.update({"traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes": top["bytes"],
                 "kernel": "%s %s" % (top["kind"], top["label"]), "ms": top_ms,
                 "share_of_step": top_ms / total_ms, "peak_source": pk["_source"]})
    if top["exps"]:
        sm_mhz = (clocks or {}).get("sm_mhz") or pk.get("sm_max_mhz", 1965.0)
        exp_peak = 148 * 16 * sm_mhz * 1e6 / 1e12   # T exp/s: 16 MUFU lanes per SM per clock at the observed clock
        roof["exp"] = {"achieved_texp_s": top["exps"] / (top_ms * 1e-3) / 1e12, "peak_texp_s": exp_peak,
                       "frac": top["exps"] / (top_ms * 1e-3) / 1e12 / exp_peak, "sm_mhz_used": sm_mhz}
    breakdown = {}
    for k, v in sorted(kinds.items(), key=lambda kv: -kv[1]["ms"]):
        e = {"ms": round(v["ms"], 3), "share": round(v["ms"] / total_ms, 4), "launches": v["launches"]}
        if v["flops"]:
            e["tflops"] = round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 2)
        if v["bytes"]:
            e["gbs"] = round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1)
        breakdown[k] = e

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- CPU baseline: the oracle on this box's host cores, bounded sample (rank 0, N = 1 only)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, h.affinity0)      # all host cores again (the NUMA binding was for the pinned buffers)
        cv, csec, _ = cpu_forward_timed(cfg, model, args.cpu_clips, T, S, alpha, steps=1, warmup=1)
        cpu = {"value": cv, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
               "sample": "%d clip(s) of the same workload, 1 warm-up + 1 timed oracle forward (%.1f s)" % (
                   args.cpu_clips, csec)}
    line = {
        "metric": metric_name(args), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": str(cfg.ESF.PRECISION), "data": "synthetic",
        "config": {"workload": workload_name(args), "global_batch": world * B, "parallelism": "dp%d" % world,
                   "l2": "inputs (1.54 GB per step) and activations (>20 GB) exceed the 126 MB L2",
                   "cuda_graph": True, "arena_gb": round(plan.arena_bytes() / 1e9, 2),
                   "weights": "random init + parity recipe (efficient_slowfast_b200/workloads.py); no trained "
                              "checkpoint is available offline"},
        "e2e": e2e,
        "gpu_launches": plan.launches_per_run * args.steps,
        "launches_per_step": plan.launches_per_run,
        "clocks": clocks, "parity_check": parity, "roofline": roof, "kernel_breakdown": breakdown,
        "eager_sum_ms": round(total_ms, 3),
    }
    if e2e_both:
        line["e2e_both_pathways_uploaded"] = e2e_both
    if e2e_u8:
        line["e2e_uint8_frames"] = e2e_u8
    if cpu:
        line["cpu_baseline"] = cpu
    if world == 1 and not args.no_extra_configs and not args.case and args.model == "SlowFastDualAttention":
        del model, plan, ins
        torch.cuda.empty_cache()
        line["configs"] = {}
        for key, name, b, f, c in EXTRA_CONFIGS:
            try:
                line["configs"][key] = run_extra_config(h, args, key, name, b, f, c)
            except Exception as e:  # noqa: BLE001 -- the headline line must still be printed
                line["configs"][key] = {"error": "%s: %s" % (type(e).__name__, e)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="SlowFastDualAttention", choices=sorted(MODEL_CASES))
    ap.add_argument("--case", default="", help="golden case (tests/golden/recipe.py CASES) instead of --model, e.g. "
                    "slow_nln_r50 / i3d_nln_r50 / i3d_r50 / slow_r50 (single-pathway ResNet, section 8-f3)")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--frames", type=int, default=32)
    ap.add_argument("--crop", type=int, default=224)
    ap.add_argument("--cpu-clips", type=int, default=1)
    ap.add_argument("--e2e-steps", type=int, default=0, help="end-to-end steps (0: --steps, at least 30)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-ops", default="", help="write per-op device times (JSON lines) to this file")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the probabilities of the last timed step to DIR/probs.npy (float32)")
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16", "fp32"],
                    help="16-bit storage / tensor-core operand format (FP32 accumulation in both)")
    ap.add_argument("--e2e-depth", type=int, default=3, help="staging slots of the end-to-end ClipStream")
    ap.add_argument("--no-extra-configs", action="store_true",
                    help="skip the short runs of BASELINE.json's other configs (`configs` in the JSON line)")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin the rank to its GPU's NUMA node")
    ap.add_argument("--profile-mode", action="store_true",
                    help="for ncu: eager launches (no CUDA graph), 1 warm-up + --steps steps, nothing else")
    args = ap.parse_args(argv)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.profile_mode and args.dump_outputs:
        ap.error("--dump-outputs writes the last timed step, and --profile-mode times none")
    args.alpha = 8 if args.model == "SlowFast" else 4
    if args.case:
        from efficient_slowfast_b200 import workloads as recipe
        spec = recipe.CASES[args.case]
        args.model = spec["model"]
        if spec.get("single"):
            args.alpha = 0
        elif args.model == "SlowFast":
            args.alpha = 8
    return args


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
