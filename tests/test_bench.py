"""bench.py: --steps sets the number of timed forwards, and --dump-outputs writes what the last of them returned."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
import helpers
import recipe
from oracle import slowfast_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ["--frames", "32", "--crop", "64", "--steps", "2", "--warmup", "1"]
GPU_SMALL = SMALL + ["--batch", "2", "--no-extra-configs", "--no-cpu-baseline", "--no-numa-bind", "--e2e-steps", "2"]


def _model_and_cfg():
    args = argparse.Namespace(case="", model="SlowFastDualAttention", crop=64, frames=32, precision="fp16")
    cfg = bench.bench_cfg(args)
    return cfg, bench.build_weights(cfg)


def _json_line(text):
    return json.loads(text.strip().splitlines()[-1])


def test_argument_checks():
    for argv in (["--steps", "0"], ["--profile-mode", "--dump-outputs", "x"]):
        with pytest.raises(SystemExit):
            bench.parse_args(argv)


def test_reference_arm_runs_steps_forwards_and_dumps_the_last(tmp_path, monkeypatch, capsys):
    forward, calls = O.forward, []

    def counting_forward(*a, **k):
        calls.append(1)
        return forward(*a, **k)

    monkeypatch.setattr(O, "forward", counting_forward)
    threads = torch.get_num_threads()
    try:
        bench.run_reference(bench.parse_args(["--impl", "reference", "--dump-outputs", str(tmp_path)] + SMALL))
    finally:
        torch.set_num_threads(threads)
    assert len(calls) == 1 + 2                                 # --warmup 1, then --steps 2 timed
    assert _json_line(capsys.readouterr().out)["steps"] == 2
    got = np.load(str(tmp_path / "probs.npy"))
    assert got.dtype == np.float32 and got.shape == (1, 400)
    cfg, model = _model_and_cfg()
    want = forward(cfg, model.state_dict(), recipe.pack_pathway_output(recipe.seeded_clip(1, 32, 64, seed=1), 4))
    assert helpers.rel_err(got, want) <= 1e-5


@pytest.mark.gpu
def test_gpu_arm_runs_steps_forwards_and_dumps_the_last(esf_lib, tmp_path, monkeypatch, capsys):
    forwards, per_window = [], []
    setup, timed = bench.setup_workload, bench.Harness.timed

    def counting_setup(h, a):
        cfg, model, shapes, ins, plan = setup(h, a)
        forward = model.forward

        def counting_forward(*x, **k):
            forwards.append(1)
            return forward(*x, **k)

        model.forward = counting_forward
        return cfg, model, shapes, ins, plan

    def counting_timed(self, fn, steps):
        n = len(forwards)
        ms = timed(self, fn, steps)
        per_window.append(len(forwards) - n)
        return ms

    monkeypatch.setattr(bench, "setup_workload", counting_setup)
    monkeypatch.setattr(bench.Harness, "timed", counting_timed)
    bench.run_gpu(bench.parse_args(GPU_SMALL + ["--dump-outputs", str(tmp_path / "a")]))
    line = _json_line(capsys.readouterr().out)
    assert per_window[0] == 2 and line["steps"] == 2          # the headline window holds exactly --steps forwards
    assert line["e2e"]["steps"] == 2
    got = np.load(str(tmp_path / "a" / "probs.npy"))
    assert got.dtype == np.float32 and got.shape == (2, 400)

    # the command line, in a process of its own, dumps the same outputs: same arguments, same inputs
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", str(tmp_path / "b")] +
                       GPU_SMALL, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    assert _json_line(r.stdout)["steps"] == 2
    assert np.array_equal(got, np.load(str(tmp_path / "b" / "probs.npy")))

    # and they are what model.forward returns for the benchmark's seeded clips
    cfg, model = _model_and_cfg()
    model = model.cuda()
    ins = [torch.empty(s, device="cuda") for s in [(2, 3, 8, 64, 64), (2, 3, 32, 64, 64)]]
    bench.fill_inputs(ins, 4, 0, ins[0].device)
    with torch.no_grad():
        want = model(ins).cpu()
    assert np.array_equal(got, want.numpy())
