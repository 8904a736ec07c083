"""AVA detection without a GPU: the RoI-align restatement of the detection oracle against torchvision, the detection
configs and their module / state_dict schema, host-side box validation, the detection branch of perform_test, and (where
the reference tree is available) the AVA YAMLs and the oracle's detection forward against the reference itself."""
import os
import sys
import types

import pytest
import torch

import detection_oracle as DO
import efficient_slowfast_b200 as esf
from efficient_slowfast_b200 import runtime as rt
from efficient_slowfast_b200 import testing as esf_testing
from efficient_slowfast_b200.workloads import seeded_state_dict
from oracle import ref_shim

# border: the whole 13 x 9 map (208 x 144 px at stride 16); zero-size; larger than the map; fractional corners
ROI_BOXES = torch.tensor([[0, 10.0, 12.0, 90.0, 100.0],
                          [1, 0.0, 0.0, 208.0, 144.0],
                          [0, -30.0, -20.0, 40.0, 50.0],
                          [1, 50.0, 50.0, 50.0, 50.0],
                          [0, -100.0, -80.0, 400.0, 300.0],
                          [1, 13.3, 7.7, 61.9, 99.1]])


def _cpu(cfg):
    cfg.NUM_GPUS = 0
    return cfg


def _cfgs():
    return {"slowfast": _cpu(esf.ava_slowfast_32x2_r50_cfg()), "slow": _cpu(esf.ava_slow_8x8_r50_cfg())}


@pytest.mark.parametrize("aligned", [True, False])
def test_oracle_roi_align_matches_torchvision(aligned):
    tv = pytest.importorskip("torchvision.ops")
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 16, 9, 13, generator=g)
    got = DO.roi_align(x, ROI_BOXES, 7, 1.0 / 16, 0, aligned)
    want = tv.roi_align(x, ROI_BOXES, 7, 1.0 / 16, 0, aligned)
    assert ((got - want).abs().max() / want.abs().max()).item() <= 1e-6
    # same order of operations as torchvision's CPU kernel: bit-identical, so the reference-gated forward test below can
    # compare the detection oracle with the reference (which runs torchvision's roi_align) bit for bit
    assert torch.equal(got, want)
    assert got[3].abs().max() == 0 if aligned else got[3].abs().max() > 0     # zero-size: empty grid vs 1 x 1 minimum


def test_default_cfg_has_reference_detection_keys():
    d = esf.get_cfg().DETECTION
    assert dict(d) == dict(ENABLE=False, ALIGNED=True, ROI_XFORM_RESOLUTION=7, SPATIAL_SCALE_FACTOR=16)


def test_ava_cfgs_restate_the_upstream_yamls():
    for name, cfg in _cfgs().items():
        npw = 2 if name == "slowfast" else 1
        assert cfg.DETECTION.ENABLE and cfg.MODEL.NUM_CLASSES == 80 and cfg.MODEL.HEAD_ACT == "sigmoid"
        assert cfg.RESNET.SPATIAL_STRIDES == [[1] * npw, [2] * npw, [2] * npw, [1] * npw]
        assert cfg.RESNET.SPATIAL_DILATIONS == [[1] * npw, [1] * npw, [1] * npw, [2] * npw]
    sf = _cfgs()["slowfast"]
    assert (sf.SLOWFAST.ALPHA, sf.SLOWFAST.FUSION_KERNEL_SZ, sf.DATA.NUM_FRAMES) == (4, 7, 32)


@pytest.mark.parametrize("name", ["slowfast", "slow"])
def test_detection_model_schema(name):
    cfg = _cfgs()[name]
    det = esf.build_model(cfg)
    cls_cfg = cfg.clone()
    cls_cfg.DETECTION.ENABLE = False
    cls = esf.build_model(cls_cfg)
    sd, sd_cls = det.state_dict(), cls.state_dict()
    assert [k for k in sd if not k.startswith("head.")] == [k for k in sd_cls if not k.startswith("head.")]
    head = {k: tuple(v.shape) for k, v in sd.items() if k.startswith("head.")}
    cin = 2304 if name == "slowfast" else 2048
    assert head == {"head.projection.weight": (80, cin), "head.projection.bias": (80,)}
    npw = det.num_pathways
    want = [n % p for p in range(npw) for n in ("s%d_tpool", "s%d_roi", "s%d_spool")] + ["dropout", "projection", "act"]
    assert [n for n, _ in det.head.named_children()] == want
    assert isinstance(det.head.act, torch.nn.Sigmoid)
    assert det.head.s0_tpool.kernel_size == [8, 1, 1]
    if npw == 2:
        assert det.head.s1_tpool.kernel_size == [32, 1, 1]
    assert det.head.s0_roi.spatial_scale == 1.0 / 16 and det.head.s0_roi.aligned and det.head.s0_roi.sampling_ratio == 0
    det.load_state_dict(seeded_state_dict(sd), strict=True)        # a reference-schema checkpoint loads strictly


def test_detection_is_refused_where_it_is_not_implemented():
    cfg = _cpu(esf.slowfast_dual_8x8_r50_cfg())
    cfg.DETECTION.ENABLE = True
    with pytest.raises(NotImplementedError):
        esf.build_model(cfg)
    cfg = _cpu(esf.slowfast_shufflenetv2_cfg(0.5))
    cfg.DETECTION.ENABLE = True
    with pytest.raises(NotImplementedError):
        esf.build_model(cfg)
    cfg = _cfgs()["slow"]
    cfg.ESF.PRECISION = "fp32"
    m = esf.build_model(cfg).eval()
    with pytest.raises(NotImplementedError):
        m._get_plan([(1, 3, 8, 64, 64)], "cpu")
    with pytest.raises(NotImplementedError):
        esf.ClipStream(m, [(1, 3, 8, 64, 64)], device="cpu")
    cls = esf.build_model(_cpu(esf.resnet_cfg("slow"))).eval()
    with pytest.raises(NotImplementedError):                     # classification models keep refusing boxes
        cls([torch.zeros(1, 3, 8, 32, 32)], torch.zeros(1, 5))


@pytest.mark.parametrize("name", ["slowfast", "slow"])
def test_head_time_axis_is_checked_before_any_plan_is_built(name):
    """The reference's ResNetRoIHead asserts that its temporal pool leaves one frame; the check runs on the clip shape,
    before a plan is evicted or compiled."""
    m = esf.build_model(_cfgs()[name]).eval()
    sentinel = object()
    m._plans["other shape"] = (m._weights_stamp(), sentinel)
    shapes = [(1, 3, 16, 64, 64), (1, 3, 64, 64, 64)][: m.num_pathways] if name == "slowfast" else [(1, 3, 16, 64, 64)]
    with pytest.raises(AssertionError):
        m._get_plan(shapes, "cpu")                                # twice the frames the head pools over
    with pytest.raises(RuntimeError):
        m._get_plan([(1, 3, 4, 64, 64), (1, 3, 16, 64, 64)] if name == "slowfast" else [(1, 3, 4, 64, 64)], "cpu")
    assert m._plans["other shape"][1] is sentinel


def test_bad_host_boxes_raise_before_launch_and_cpu_forward_raises():
    cfg = _cfgs()["slowfast"]
    m = esf.build_model(cfg).eval()
    xs = [torch.zeros(2, 3, 8, 64, 64), torch.zeros(2, 3, 32, 64, 64)]
    for bad in (torch.zeros(3, 4), torch.zeros(5), torch.zeros(2, 5, dtype=torch.long),
                torch.tensor([[2.0, 0, 0, 8, 8]]), torch.tensor([[-1.0, 0, 0, 8, 8]]),
                torch.tensor([[float("nan"), 0, 0, 8, 8]]), [[0, 0, 0, 8, 8]]):
        with pytest.raises(ValueError):
            m(xs, bad)
        with pytest.raises(ValueError):
            m.forward_fast(xs[1], bad)
    with pytest.raises(ValueError):
        m(xs)                                                    # detection without boxes
    with pytest.raises(rt.EsfError):                             # valid boxes: no CPU fallback
        m(xs, torch.tensor([[1.0, 0, 0, 8, 8]], dtype=torch.float64))


def test_roi_kernels_use_no_local_memory(esf_lib):
    """The RoI-head kernels are built for sm_100a without spills (no local memory)."""
    import shutil
    import subprocess

    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-res-usage", rt.lib_path()], stdout=subprocess.PIPE, text=True).stdout
    usage, name = {}, None
    for line in out.splitlines():
        line = line.strip()
        if line.startswith("Function "):
            name = line[len("Function "):].rstrip(":")
        elif line.startswith("REG:") and name:
            usage[name] = dict(kv.split(":") for kv in line.split() if ":" in kv and not kv.startswith("CONSTANT"))
    roi = {n: u for n, u in usage.items() if "roi_align_max_kernel" in n or "temporal_mean" in n}
    assert len(roi) == 3, sorted(roi)
    assert all(int(u["LOCAL"]) == 0 for u in roi.values()), roi


class _FakeAVAMeter:
    def __init__(self):
        self.calls = []

    def iter_tic(self):
        self.calls.append("tic")

    def iter_toc(self):
        self.calls.append("toc")

    def update_stats(self, preds, ori_boxes, metadata):
        self.calls.append(("update", preds.clone(), ori_boxes, metadata))

    def log_iter_stats(self, cur_epoch, cur_iter):
        self.calls.append(("log", cur_epoch, cur_iter))

    def finalize_metrics(self):
        self.calls.append("final")
        return "mAP"


class _FakeDetector(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.w = torch.nn.Parameter(torch.ones(1))
        self.seen = []

    def forward(self, inputs, bboxes):
        self.seen.append(([t.shape for t in inputs], bboxes))
        return bboxes[:, 1:3] * 2


def test_perform_test_detection_branch():
    cfg = _cfgs()["slowfast"]
    cfg.NUM_GPUS = 1
    boxes = [torch.tensor([[0.0, 1, 2, 3, 4], [1, 5, 6, 7, 8]]), torch.tensor([[0.0, 9, 10, 11, 12]])]
    loader = [([torch.zeros(2, 3, 8, 4, 4), torch.zeros(2, 3, 32, 4, 4)], torch.zeros(2), torch.arange(2),
               dict(boxes=b, ori_boxes=b[:, 1:] / 10, metadata=torch.full((b.shape[0], 2), i)))
              for i, b in enumerate(boxes)]
    model, meter = _FakeDetector(), _FakeAVAMeter()
    assert esf_testing.perform_test(loader, model, meter, cfg) == "mAP"
    assert [b for _, b in model.seen] == boxes
    updates = [c for c in meter.calls if isinstance(c, tuple) and c[0] == "update"]
    assert len(updates) == 2
    for (_, preds, ori, meta), b, i in zip(updates, boxes, range(2)):
        assert torch.equal(preds, b[:, 1:3] * 2) and torch.equal(ori, b[:, 1:] / 10)
        assert torch.equal(meta, torch.full((b.shape[0], 2), i))
    assert [c for c in meter.calls if isinstance(c, tuple) and c[0] == "log"] == [("log", None, 0), ("log", None, 1)]
    assert meter.calls[0] == "tic" and meter.calls[-1] == "final"
    cfg.NUM_GPUS = 2
    with pytest.raises(NotImplementedError):
        esf_testing.perform_test(loader, model, meter, cfg)


# ------------------------------------------------------------------------------------------------ reference-gated
AVA_YAMLS = ["configs/AVA/SLOWFAST_32x2_R50_SHORT.yaml", "configs/AVA/SLOW_8x8_R50_SHORT.yaml",
             "configs/AVA/c2/SLOWFAST_32x2_R101_50_50.yaml", "configs/AVA/c2/SLOWFAST_32x2_R101_50_50_v2.1.yaml",
             "configs/AVA/c2/SLOWFAST_32x2_R50.yaml", "configs/AVA/c2/SLOWFAST_64x2_R101_50_50.yaml",
             "configs/AVA/c2/SLOW_8x8_R50.yaml"]

needs_reference = pytest.mark.skipif(not ref_shim.available(), reason="reference tree not mounted")


def _reference_with_roialign():
    """ref_shim.install(), with detectron2.layers.ROIAlign backed by torchvision's roi_align so that the reference can
    build and run its ResNetRoIHead."""
    tv = pytest.importorskip("torchvision.ops")
    ref_shim.install()

    class ROIAlign(torch.nn.Module):
        def __init__(self, output_size, spatial_scale, sampling_ratio, aligned=True):
            super().__init__()
            self.output_size, self.spatial_scale = output_size, spatial_scale
            self.sampling_ratio, self.aligned = sampling_ratio, aligned

        def forward(self, x, rois):
            return tv.roi_align(x, rois, self.output_size, self.spatial_scale, self.sampling_ratio, self.aligned)

    sys.modules["detectron2.layers"].ROIAlign = ROIAlign
    for name, mod in list(sys.modules.items()):
        if name.startswith("slowfast.models") and isinstance(mod, types.ModuleType) and hasattr(mod, "ROIAlign"):
            mod.ROIAlign = ROIAlign


def _ours(rcfg):
    cfg = esf.get_cfg()
    for sec in ("RESNET", "NONLOCAL", "MODEL", "SLOWFAST", "DATA", "DETECTION", "MULTIGRID", "BN"):
        for k in cfg[sec]:
            if k in rcfg[sec]:
                cfg[sec][k] = rcfg[sec][k]
    cfg.NUM_GPUS = 0
    return cfg


@needs_reference
@pytest.mark.parametrize("yaml_rel", AVA_YAMLS)
def test_ava_yamls_build_like_reference(yaml_rel):
    _reference_with_roialign()
    if not os.path.exists(os.path.join(ref_shim.REF_ROOT, "SlowFast", yaml_rel)):
        pytest.skip("%s not in the reference tree" % yaml_rel)
    rcfg = ref_shim.get_cfg(yaml_rel)
    torch.manual_seed(0)
    ref = ref_shim.build_reference_model(rcfg)
    torch.manual_seed(0)
    ours = esf.build_model(_ours(rcfg))
    a, b = ref.state_dict(), ours.state_dict()
    assert list(a) == list(b)
    for k in a:
        assert a[k].shape == b[k].shape, k
        assert torch.equal(a[k], b[k]), k


@needs_reference
def test_ava_yamls_match_reference():
    """The restated AVA cfgs carry the values of the reference's YAMLs for every key the model builders read."""
    for fn, rel in ((esf.ava_slowfast_32x2_r50_cfg, AVA_YAMLS[0]), (esf.ava_slow_8x8_r50_cfg, AVA_YAMLS[1])):
        ours, ref = fn(), _ours(ref_shim.get_cfg(rel))
        for sec in ("RESNET", "MODEL", "SLOWFAST", "DETECTION"):
            for k in ("SPATIAL_STRIDES", "SPATIAL_DILATIONS", "NUM_CLASSES", "HEAD_ACT", "ALPHA", "FUSION_KERNEL_SZ",
                      "ENABLE", "ALIGNED", "ROI_XFORM_RESOLUTION", "SPATIAL_SCALE_FACTOR"):
                if k in ours[sec]:
                    assert ours[sec][k] == ref[sec][k], (rel, sec, k)
        assert ours.DATA.NUM_FRAMES == ref.DATA.NUM_FRAMES, rel


@needs_reference
@pytest.mark.parametrize("yaml_rel", AVA_YAMLS[:2])
def test_oracle_detection_forward_equals_reference(yaml_rel):
    _reference_with_roialign()
    rcfg = ref_shim.get_cfg(yaml_rel)
    torch.manual_seed(0)
    ref = ref_shim.build_reference_model(rcfg).eval()
    sd = seeded_state_dict(ref.state_dict())
    ref.load_state_dict(sd)
    cfg = _ours(rcfg)
    g = torch.Generator().manual_seed(1)
    fast = torch.randn(2, 3, cfg.DATA.NUM_FRAMES, 64, 96, generator=g)
    if cfg.MODEL.MODEL_NAME == "SlowFast":
        idx = torch.linspace(0, fast.shape[2] - 1, fast.shape[2] // cfg.SLOWFAST.ALPHA).long()
        xs = [fast.index_select(2, idx), fast]
    else:
        xs = [fast]
    boxes = torch.tensor([[1.0, 3, 4, 50, 60], [0, 10, 2, 90, 63], [1, 0, 0, 96, 64]])
    with torch.no_grad():
        want = ref([t.clone() for t in xs], boxes.clone())
    got = DO.forward(cfg, sd, xs, boxes)
    assert torch.equal(got, want)
