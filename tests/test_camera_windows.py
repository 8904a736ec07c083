"""demo.CameraWindows without a GPU: the per-camera ring arithmetic against the reference demo's list buffer
(tools/demo_net.py: append, then pop(0) once full), the ring-bank gather of esf_*_rings emulated with torch indexing
against oracle/input_oracle.demo_window_inputs, argument validation before anything is copied, and the C ABI's
exports and host-side range checks."""
import ctypes

import pytest
import torch

import helpers
from oracle import input_oracle as IO


def _schedule(cameras, ticks, seed):
    """Which cameras push on every tick: each camera joins at its own tick, then pushes on most later ticks."""
    g = torch.Generator().manual_seed(seed)
    join = [int(j) for j in torch.randint(0, ticks // 2, (cameras,), generator=g)]
    out = []
    for k in range(ticks):
        ids = [c for c in range(cameras) if k >= join[c] and bool(torch.rand(1, generator=g) < 0.8)]
        out.append(ids)
    return out


@pytest.mark.parametrize("stride", [1, 3])
def test_clock_matches_reference_list_buffer(stride):
    """Per camera: the slot of every frame, the rows a push makes and their oldest slot agree with the reference's
    buffer (append; full: run the model on it -- every `stride`-th time here -- then pop(0))."""
    from efficient_slowfast_b200 import demo

    N, L, nf, alpha = 5, 12, 6, 3
    pos = demo.window_indices(L, nf, alpha)
    clock = demo.CameraClock(N, L, stride)
    ring = [[None] * L for _ in range(N)]
    bufs = [[] for _ in range(N)]
    full_pushes = [0] * N
    frame = 0
    for ids in _schedule(N, 60, seed=stride):
        expect = []
        for c in ids:
            ring[c][clock.slot(c)] = frame
            bufs[c].append(frame)
            frame += 1
            if len(bufs[c]) == L:
                if full_pushes[c] % stride == 0:
                    expect.append((c, list(bufs[c])))
                full_pushes[c] += 1
                bufs[c].pop(0)
        assert [clock.ready_after_push(c) for c in ids] == [c in [e[0] for e in expect] for c in ids]
        rows = clock.advance(ids)
        assert [c for c, _ in rows] == [c for c, _ in expect]
        for (c, oldest), (_, window) in zip(rows, expect):
            for p in pos:
                assert [ring[c][(int(i) + oldest) % L] for i in p] == [window[int(i)] for i in p]
    assert sum(full_pushes) > 3 * N


def _emulate_rings(fin, bank, rows, positions):
    """What esf_frames_to_clip_rings computes (csrc/esf_simt.cu frames_to_clip_kernel<RingFrames>): clip[r, c, t, h, w] =
    lut32[c][bank[camera_r, (pos[t] + oldest_r) % L, h, w, chan_src[c]]]."""
    L = bank.shape[1]
    cam = torch.tensor([c for c, _ in rows])
    oldest = torch.tensor([o for _, o in rows])
    src = torch.tensor(list(fin.chan_src))
    out = []
    for p in positions:
        slot = (p.long().reshape(1, -1) + oldest.reshape(-1, 1)) % L              # (R, T)
        g = bank[cam.reshape(-1, 1), slot][..., src].long()                      # (R, T, H, W, C)
        out.append(torch.stack([fin.lut32[c][g[..., c]] for c in range(bank.shape[4])], dim=1).contiguous())
    return out


@pytest.mark.parametrize("name", ["dual_r50", "slow_r50"])
def test_ring_gather_reproduces_demo_inputs(name):
    """Every row of every tick, gathered from the bank as the kernel does, equals the reference demo's inputs for that
    camera's last L frames bit for bit (one and two pathways)."""
    from efficient_slowfast_b200 import demo
    from efficient_slowfast_b200 import frames as F

    cfg = helpers.case_cfg(name)
    cfg.DATA.SAMPLING_RATE = 2
    cfg.DATA.MEAN, cfg.DATA.STD = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
    nf = int(cfg.DATA.NUM_FRAMES)
    L = nf * 2
    alpha = None if name == "slow_r50" else int(cfg.SLOWFAST.ALPHA)
    N, H, W, C = 4, 5, 7, 3
    fin = F.FrameInput(cfg, torch.device("cpu"), torch.float16)
    positions = demo.window_indices(L, nf, alpha)
    clock = demo.CameraClock(N, L, 1)
    bank = torch.zeros((N, L, H, W, C), dtype=torch.uint8)
    history = [[] for _ in range(N)]
    g = torch.Generator().manual_seed(3)
    checked = 0
    for ids in _schedule(N, 3 * L, seed=11):
        for c in ids:
            f = torch.randint(0, 256, (H, W, C), generator=g, dtype=torch.uint8)
            bank[c, clock.slot(c)] = f
            history[c].append(f)
        rows = clock.advance(ids)
        if not rows:
            continue
        got = _emulate_rings(fin, bank, rows, positions)
        for r, (c, _) in enumerate(rows):
            ref = IO.demo_window_inputs(torch.stack(history[c][-L:]), cfg.DATA.MEAN, cfg.DATA.STD, nf, alpha)
            assert len(ref) == len(got)
            for x, y in zip(ref, got):
                assert torch.equal(y[r:r + 1], x.contiguous())
            checked += 1
    assert checked > 2 * N


def _check(frames, boxes=None, detection=False, clock=None, shape=(4, 6, 3)):
    from efficient_slowfast_b200 import demo

    clock = clock or demo.CameraClock(3, 4, 1)
    return demo.check_push(frames, boxes, clock, shape, torch.device("cuda", 0), detection)


def test_push_validation_before_any_copy():
    """Every refusal is a ValueError raised by check_push, which CameraWindows.push runs before it copies a frame or
    counts a push: the clock is unchanged after each one."""
    from efficient_slowfast_b200 import demo

    clock = demo.CameraClock(3, 4, 1)
    ok = torch.zeros((4, 6, 3), dtype=torch.uint8)
    bad = [
        ([ok], None),                                                    # not a dict
        ({3: ok}, None),                                                 # unknown id
        ({-1: ok}, None),
        ({True: ok}, None),
        ({"0": ok}, None),
        ({0: torch.zeros((4, 6, 4), dtype=torch.uint8)}, None),          # wrong shape
        ({0: torch.zeros((4, 6, 3), dtype=torch.float32)}, None),        # wrong dtype
        ({0: torch.zeros((6, 4, 3), dtype=torch.uint8).transpose(0, 1)}, None),      # not contiguous
        ({0: torch.zeros((4, 6, 3), dtype=torch.uint8, device="meta")}, None),       # another device
        ({0: ok}, {0: torch.zeros((1, 4))}),                             # boxes for a classification model
    ]
    for frames, boxes in bad:
        with pytest.raises(ValueError):
            demo.check_push(frames, boxes, clock, (4, 6, 3), torch.device("cuda", 0), False)
        assert clock.count == [0, 0, 0]
    ids, ready, b, counts = _check({2: ok, 0: ok}, clock=clock)
    assert ids == [0, 2] and ready == [] and b is None and clock.count == [0, 0, 0]


def test_detection_boxes_validation_and_rows():
    from efficient_slowfast_b200 import demo

    clock = demo.CameraClock(3, 2, 1)
    ok = torch.zeros((4, 6, 3), dtype=torch.uint8)
    clock.advance([0, 1, 2])                 # one frame in every ring: the next push fills the windows
    with pytest.raises(ValueError):          # a ready camera without boxes
        _check({0: ok, 1: ok}, {0: torch.zeros((1, 4))}, True, clock)
    with pytest.raises(ValueError):          # boxes for a camera without a frame in this push
        _check({0: ok}, {0: torch.zeros((1, 4)), 2: torch.zeros((1, 4))}, True, clock)
    with pytest.raises(ValueError):          # wrong box shape
        _check({0: ok}, {0: torch.zeros((1, 5))}, True, clock)
    with pytest.raises(ValueError):          # integer boxes
        _check({0: ok}, {0: torch.zeros((1, 4), dtype=torch.int64)}, True, clock)
    with pytest.raises(ValueError):          # no boxes at all
        _check({0: ok}, None, True, clock)
    assert clock.count == [1, 1, 1]
    b0 = torch.tensor([[1.0, 2.0, 3.0, 4.0], [5.0, 6.0, 7.0, 8.0]])
    b2 = torch.tensor([[0.5, 1.5, 2.5, 3.5]], dtype=torch.float64)
    ids, ready, rows, counts = _check({2: ok, 0: ok}, {0: b0, 2: b2}, True, clock)
    assert ids == ready == [0, 2] and counts == [2, 1]
    assert rows.dtype == torch.float32 and torch.equal(rows[:, 0], torch.tensor([0.0, 0.0, 1.0]))
    assert torch.equal(rows[:, 1:], torch.cat([b0, b2.float()]))


def test_library_exports_ring_entry_points_and_checks_ranges(esf_lib):
    """Both ring entry points are exported, and every range the kernel's slot arithmetic relies on is checked on the
    host copies before a launch.  Every call below passes a null output, so none of them can reach a launch even if a
    check were missing; the error message shows which check refused it (the range checks come first)."""
    P = ctypes.POINTER(ctypes.c_int32)
    for name in ("esf_stem_pack_u8_rings", "esf_frames_to_clip_rings"):
        assert hasattr(esf_lib, name)
    fake = ctypes.c_void_p(256)          # never dereferenced: every call is refused on the host
    N, L, H, W, C = 2, 8, 4, 4, 3

    def refused(rows, pos, R=None, n=N, c=C, pitch=16, clip=True):
        """(rc, error message) of esf_stem_pack_u8_rings and, with `clip`, of esf_frames_to_clip_rings."""
        rows_a = (ctypes.c_int32 * len(rows))(*rows)
        pos_a = (ctypes.c_int32 * len(pos))(*pos)
        R = len(rows) // 2 if R is None else R
        out = [(esf_lib.esf_stem_pack_u8_rings(fake, n, L, H, W, c, fake, ctypes.cast(rows_a, P), R, fake,
                                               ctypes.cast(pos_a, P), len(pos), None, fake, pitch, 0, None, None),
                esf_lib.esf_last_error())]
        if clip:
            out.append((esf_lib.esf_frames_to_clip_rings(fake, n, L, H, W, c, fake, ctypes.cast(rows_a, P), R, fake,
                                                         ctypes.cast(pos_a, P), len(pos), None, fake, None, None),
                        esf_lib.esf_last_error()))
        return out

    good_pos = [0, 2, 5, 7]
    cases = [
        (dict(rows=[0, 0], pos=good_pos, R=0), b"R 0"),                          # R >= 1
        (dict(rows=[2, 0], pos=good_pos), b"camera 2 not in [0, 2)"),            # camera out of range
        (dict(rows=[-1, 0], pos=good_pos), b"camera -1 not in"),
        (dict(rows=[1, 8], pos=good_pos), b"oldest slot 8 not in [0, 8)"),       # oldest slot out of range
        (dict(rows=[1, 0], pos=[0, 2, 5, 8]), b"pos[3] = 8 not in [0, 8)"),      # pos out of range
        (dict(rows=[1, 0], pos=[-1, 2, 5, 7]), b"pos[0] = -1"),
        (dict(rows=[1, 0], pos=good_pos, c=5), b"null/bad argument"),            # C <= 4
        (dict(rows=[1, 0], pos=good_pos, n=0), b"N 0"),
        (dict(rows=[1, 0], pos=good_pos, pitch=8, clip=False), b"bad pitch 8"),  # W * C = 12 > pitch
        (dict(rows=[1, 0], pos=good_pos), b"null argument"),                     # valid ranges, null output
    ]
    for kw, msg in cases:
        for rc, err in refused(**kw):
            assert rc < 0 and msg in err and b"launch" not in err, (kw, rc, err)
