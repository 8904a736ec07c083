"""JPEG decoding on the GPU: decode_jpeg equals cv2.imdecode bit for bit (IMREAD_COLOR and IMREAD_GRAYSCALE) on the
CPU tier's matrix, on 360p / 720p / 1080p frames and on one call mixing qualities, table sets, restart intervals and
sampling across many files; it writes nothing next to its output and nothing at all on a refused argument; an invalid
Huffman code sets only its own file's status; and the decoded frames feed forward_ava_frames / forward_frames on the
same stream with the same scores as cv2-decoded frames."""
import shutil
import subprocess

import numpy as np
import pytest
import torch

import helpers
from efficient_slowfast_b200 import decode_jpeg, runtime
from test_gpu_frames_ava import _boxes, _model
from test_jpeg import QUALITIES, SAMPLING, SIZES, encode, image, matrix_files

cv2 = pytest.importorskip("cv2")
pytestmark = pytest.mark.gpu

GUARD = 4096
SENTINEL = 0xA5


def _guarded(n, H, W, C):
    """(buffer, out): out is a contiguous (n, H, W, C) view with GUARD sentinel bytes on both sides."""
    buf = torch.full((2 * GUARD + n * H * W * C,), SENTINEL, dtype=torch.uint8, device="cuda")
    return buf, buf[GUARD:GUARD + n * H * W * C].view(n, H, W, C)


def _guards_intact(buf):
    return bool((buf[:GUARD] == SENTINEL).all()) and bool((buf[-GUARD:] == SENTINEL).all())


def _check(files, gray):
    ref = np.stack([cv2.imdecode(np.asarray(f).reshape(-1), cv2.IMREAD_GRAYSCALE if gray else cv2.IMREAD_COLOR)
                    for f in files])
    if gray:
        ref = ref[..., None]
    buf, out = _guarded(len(files), ref.shape[1], ref.shape[2], ref.shape[3])
    status = decode_jpeg(files, out, gray=gray)
    got = out.cpu().numpy()
    bad = [i for i in range(len(files)) if not np.array_equal(got[i], ref[i])]
    assert not bad, "frames %s differ from cv2.imdecode" % bad[:10]
    assert not status.any().item()
    assert _guards_intact(buf)


@pytest.mark.parametrize("size", SIZES, ids=["%dx%d" % s for s in SIZES])
def test_matrix_matches_cv2(esf_lib, size):
    """One call per size over the whole matrix: 4 qualities x 6 samplings x 3 restart intervals x 2 table kinds x 2
    contents = 288 files, in both modes."""
    files = [f for _, _, f in matrix_files([size])]
    assert len(files) == 288
    for gray in (False, True):
        _check(files, gray)


@pytest.mark.parametrize("H,W", [(360, 640), (720, 1280), (1080, 1920)])
def test_video_frames_match_cv2(esf_lib, H, W):
    """Frames at video sizes, each sampling, with and without one restart interval per MCU row."""
    files = []
    for noisy in (0, 1):
        img = image(H, W, noisy)
        for s in SAMPLING:
            mcu_w = 32 if s == "411" else (16 if s in ("422", "420") else 8)
            for r in (0, -(-W // mcu_w)):
                files.append(encode(img, 95 if noisy else 75, s, r))
    for gray in (False, True):
        _check(files, gray)


def test_mixed_call_of_many_files(esf_lib):
    """300 files of one size mixing qualities (so quantisation tables), optimised and standard Huffman tables,
    restart intervals and samplings in one call."""
    rng = np.random.default_rng(1)
    files = []
    for i in range(300):
        img = image(48, 72, i % 2, seed=i)
        files.append(encode(img, QUALITIES[i % 4], SAMPLING[(i // 4) % 6], int(rng.integers(0, 4)), int(rng.integers(0, 2))))
    for gray in (False, True):
        _check(files, gray)


def test_refused_argument_writes_nothing(esf_lib):
    files = [encode(image(32, 48, 1), 80, "420") for _ in range(3)]
    buf, out = _guarded(3, 32, 48, 3)
    torch.cuda.synchronize()
    with pytest.raises(ValueError, match="progressive"):
        decode_jpeg(files[:2] + [encode(image(32, 48, 1), 80, "420", progressive=1)], out)
    with pytest.raises(ValueError, match="file 2 is 32 x 40"):
        decode_jpeg(files[:2] + [encode(image(32, 40, 1), 80, "420")], out)
    with pytest.raises(ValueError, match="channels"):
        decode_jpeg(files, out, gray=True)
    torch.cuda.synchronize()
    assert bool((buf == SENTINEL).all())


def test_invalid_huffman_code_sets_only_its_status(esf_lib):
    """File 6's scan gets a run of 64 one-bits (FF 00 pairs: no marker, the framing is unchanged), which no Huffman
    table may code: its status is set, every other file is exact and nothing is written outside the output."""
    from efficient_slowfast_b200 import jpeg as J

    files = [encode(image(64, 96, i % 2, seed=i), 85, SAMPLING[i % 5], 2 if i % 3 else 0) for i in range(12)]
    b = bytearray(bytes(files[6]))
    begin, end = J.parse(b).segments[0]
    k = (begin + end) // 2
    while b[k - 1] == 0xFF:
        k += 1
    b[k:k + 16] = b"\xFF\x00" * 8
    files[6] = np.frombuffer(bytes(b), np.uint8)
    ref = np.stack([cv2.imdecode(f, cv2.IMREAD_COLOR) for f in files])
    buf, out = _guarded(12, 64, 96, 3)
    status = decode_jpeg(files, out).cpu()
    assert status[6] != 0 and int(status.ne(0).sum()) == 1
    got = out.cpu().numpy()
    assert all(np.array_equal(got[i], ref[i]) for i in range(12) if i != 6)
    assert _guards_intact(buf)


def _jpeg_clip(T, H, W, seed, sampling="420", quality=90):
    """T JPEG files of a smooth moving pattern plus noise."""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[:H, :W]
    files = []
    for t in range(T):
        base = np.stack([(x + 3 * t) % 256, (y * 2 + t) % 256, (x + y + 5 * t) % 256], -1)
        img = np.clip(base + rng.integers(-20, 21, (H, W, 3)), 0, 255).astype(np.uint8)
        files.append(encode(img, quality, sampling, restart=t % 3))
    return files


@pytest.mark.parametrize("name", ["slowfast_r50", "slow_r50"])
def test_ava_frames_from_jpeg(esf_lib, name):
    """decode_jpeg into the (B, T, H, W, 3) frames tensor, then forward_ava_frames on the same stream with no
    synchronisation in between: the scores equal those from cv2-decoded frames bit for bit."""
    cfg, model = _model(name)
    B, T, H, W = 2, cfg.DATA.NUM_FRAMES, 256, 340
    files = [f for b in range(B) for f in _jpeg_clip(T, H, W, seed=b)]
    boxes = _boxes(5, B, seed=3)
    host = torch.from_numpy(np.stack([cv2.imdecode(f, cv2.IMREAD_COLOR) for f in files]).reshape(B, T, H, W, 3))
    with torch.no_grad():
        want = model.forward_ava_frames(host.cuda(), boxes).cpu()
        frames = torch.empty(B, T, H, W, 3, dtype=torch.uint8, device="cuda")
        status = decode_jpeg(files, frames)
        got = model.forward_ava_frames(frames, boxes).cpu()
    assert torch.equal(frames.cpu(), host)
    assert torch.equal(got, want)
    assert not status.any().item()


def test_gray_frames_from_jpeg(esf_lib):
    """decode_jpeg(gray=True) of colour files into the (B, T, H, W, 1) frames of a grey R18 model, then forward_frames:
    equal to the same call on cv2.IMREAD_GRAYSCALE frames."""
    cfg, model, _ = helpers.case_model_and_weights("dual_r18_gray")
    model = model.cuda().eval()
    B, T, H, W = 2, cfg.DATA.NUM_FRAMES, 112, 112
    files = [f for b in range(B) for f in _jpeg_clip(T, H, W, seed=10 + b, sampling=["420", "444"][b])]
    host = torch.from_numpy(np.stack([cv2.imdecode(f, cv2.IMREAD_GRAYSCALE) for f in files]).reshape(B, T, H, W, 1))
    with torch.no_grad():
        want = model.forward_frames(host.cuda()).cpu()
        frames = torch.empty(B, T, H, W, 1, dtype=torch.uint8, device="cuda")
        status = decode_jpeg(files, frames, gray=True)
        got = model.forward_frames(frames).cpu()
    assert torch.equal(frames.cpu(), host)
    assert torch.equal(got, want)
    assert not status.any().item()


def test_jpeg_kernels_use_no_local_memory(esf_lib):
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    out = subprocess.run([cuobjdump, "-res-usage", runtime.lib_path()], stdout=subprocess.PIPE, text=True).stdout
    usage, name = {}, None
    for line in out.splitlines():
        line = line.strip()
        if line.startswith("Function "):
            name = line[len("Function "):].rstrip(":")
        elif line.startswith("REG:") and name and "jpeg" in name:
            usage[name] = dict(kv.split(":") for kv in line.split() if ":" in kv and not kv.startswith("CONSTANT"))
    assert len(usage) == 3, sorted(usage)
    assert all(int(u["LOCAL"]) == 0 for u in usage.values()), usage
