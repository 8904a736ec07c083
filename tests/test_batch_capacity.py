"""Batch capacity (cfg.ESF.MAX_BATCH) on the host: how a variant's allocations and weight preparation resolve to its
capacity plan's (engine.Plan.alloc / Plan.once), and the plan key and refusals of _get_plan."""
import pytest
import torch

import helpers
from efficient_slowfast_b200 import build_model, config
from efficient_slowfast_b200 import runtime as rt
from efficient_slowfast_b200.engine import Family, Plan


def _family(n_rows=4):
    fam = Family()
    cap = Plan("cpu", "fp16", family=fam)
    a = cap.act(n_rows, 2, 3, 3, 12)                                 # rows: padded to 16 channels
    w = cap.alloc((5, 7), torch.float32, zero=True)                  # does not depend on the batch
    s = cap.alloc((n_rows * 10,), torch.uint8, flat=True)            # write-before-read scratch
    z = cap.scratch((n_rows, 6), torch.float16, zero=True)           # zero-filled state
    folded = cap.once(lambda x: (x * 2, x.sum().item(), torch.ones(2)), torch.arange(3.0))
    cap.end_compile()
    return fam, cap, (a, w, s, z, folded)


def test_variant_resolves_to_capacity_tensors():
    fam, cap, (a, w, s, z, folded) = _family()
    assert fam.built and not cap.variant and [t.data_ptr() for t, _, _ in fam.allocs] == \
        [a.data_ptr(), w.data_ptr(), s.data_ptr(), z.data_ptr()]
    assert torch.equal(folded[0], torch.tensor([0.0, 2, 4])) and folded[1] == 3.0
    v = Plan("cpu", "fp16", family=fam)
    assert v.variant
    a2 = v.act(2, 2, 3, 3, 12)
    assert a2.shape == (2, 2, 3, 3, 12) and a2.data_ptr() == a.data_ptr() and a2.stride() == a.stride()
    assert v.padded[a2.data_ptr()] == (12, 16)
    assert v.alloc((5, 7), torch.float32, zero=True) is fam.allocs[1][0]
    s2 = v.alloc((30,), torch.uint8, flat=True)
    assert s2.shape == (30,) and s2.data_ptr() == s.data_ptr()
    z2 = v.scratch((2, 6), torch.float16, zero=True)
    assert z2.shape == (2, 6) and z2.data_ptr() == z.data_ptr()
    calls = []
    out = v.once(lambda x: calls.append(x), None)     # a variant does not run the preparation
    assert not calls and out[0].device.type == "meta" and out[0].shape == (3,) and out[1] == 3.0
    v.end_compile()


@pytest.mark.parametrize("shape,dtype,zero,flat", [
    ((6, 2, 3, 3, 16), torch.float16, False, False),    # more rows than the capacity
    ((2, 2, 3, 3, 24), torch.float16, False, False),    # a per-clip dimension differs
    ((2, 2, 3, 3, 16), torch.float32, False, False),    # dtype
    ((2, 2, 3, 3, 16), torch.float16, True, False),     # zero-filled where the capacity's is not
])
def test_variant_rejects_allocations_that_do_not_fit(shape, dtype, zero, flat):
    fam, _, _ = _family()
    v = Plan("cpu", "fp16", family=fam)
    with pytest.raises(AssertionError):
        v.alloc(shape, dtype, zero=zero, flat=flat)


def test_variant_rejects_growing_1d_tensor_that_is_not_flat_scratch():
    fam = Family()
    cap = Plan("cpu", "fp16", family=fam)
    cap.alloc((40,), torch.float32)
    cap.end_compile()
    with pytest.raises(AssertionError):
        Plan("cpu", "fp16", family=fam).alloc((20,), torch.float32)
    with pytest.raises(AssertionError):
        Plan("cpu", "fp16", family=fam).alloc((20,), torch.float32, zero=True, flat=True)


def test_variant_must_replay_the_whole_capacity_plan():
    fam, _, _ = _family()
    v = Plan("cpu", "fp16", family=fam)
    v.act(1, 2, 3, 3, 12)
    with pytest.raises(AssertionError):
        v.end_compile()                                  # allocations left over: the compiles diverged
    v = Plan("cpu", "fp16", family=fam)
    for shape, dtype, zero, flat in [((1, 2, 3, 3, 16), torch.float16, False, False), ((5, 7), torch.float32, True, False),
                                     ((10,), torch.uint8, False, True), ((1, 6), torch.float16, True, False)]:
        v.alloc(shape, dtype, zero, flat)
    with pytest.raises(AssertionError):
        v.once(len, ())                                  # another function at this position
    with pytest.raises(AssertionError):
        v.alloc((1,), torch.float32)                     # more allocations than the capacity plan made


def test_standalone_plan_records_nothing():
    p = Plan("cpu", "fp16")
    p.act(2, 1, 1, 1, 8)
    assert p.once(lambda: 5) == 5 and p.family is None and p.shared is p and not p.variant


def test_max_batch_is_opt_in():
    cfg = config.get_cfg()
    assert "MAX_BATCH" not in cfg.ESF
    cfg = helpers.case_cfg("slow_r50")
    assert build_model(cfg)._max_batch == 0
    cfg.ESF.MAX_BATCH = -1
    with pytest.raises(ValueError):
        build_model(cfg)


def test_batch_over_capacity_is_refused_before_any_compile():
    cfg = helpers.case_cfg("slow_r50")
    cfg.ESF.MAX_BATCH = 4
    model = build_model(cfg).eval()
    assert model._max_batch == 4
    with pytest.raises(rt.EsfError, match="MAX_BATCH"):
        model._get_plan([(5, 3, 8, 64, 64)], torch.device("cuda", 0))
    assert len(model._plans) == 0
