"""JPEG decoding, CPU tier: the numpy restatement of the decoder (tests/jpeg_oracle.py, on the product's header parser) is
bit-equal to cv2.imdecode in IMREAD_COLOR and IMREAD_GRAYSCALE over a matrix of sizes, qualities, sampling factors,
restart intervals, optimised tables and content; decode_jpeg refuses what it does not decode with ValueError before
anything is copied or launched; the C ABI's argument checks return error codes."""
import ctypes
import itertools
import struct

import numpy as np
import pytest
import torch

import jpeg_oracle as O
from efficient_slowfast_b200 import jpeg as J

cv2 = pytest.importorskip("cv2")

SIZES = [(1, 1), (2, 3), (7, 13), (8, 8), (16, 16), (17, 33), (37, 53), (120, 161)]
QUALITIES = [1, 50, 90, 100]
SAMPLING = ["444", "422", "420", "440", "411", "gray"]
RESTARTS = [0, 1, 3]


def image(h, w, noisy, seed=0):
    if noisy:
        return np.random.default_rng(seed + h * 1000 + w).integers(0, 256, (h, w, 3), dtype=np.uint8)
    y, x = np.mgrid[:h, :w]
    return np.stack([x * 255 // max(w - 1, 1), y * 255 // max(h - 1, 1), (x + y) * 7 % 256], -1).astype(np.uint8)


def encode(img, quality=90, sampling="420", restart=0, optimize=0, progressive=0):
    """cv2.imencode of a BGR frame; sampling "gray" writes a one-component file of its grey conversion."""
    params = [cv2.IMWRITE_JPEG_QUALITY, quality, cv2.IMWRITE_JPEG_RST_INTERVAL, restart, cv2.IMWRITE_JPEG_OPTIMIZE,
              optimize, cv2.IMWRITE_JPEG_PROGRESSIVE, progressive]
    if sampling == "gray":
        img = cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)
    else:
        params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, getattr(cv2, "IMWRITE_JPEG_SAMPLING_FACTOR_" + sampling)]
    ok, buf = cv2.imencode(".jpg", img, params)
    assert ok
    return buf.reshape(-1)


def matrix_files(sizes=SIZES):
    """((h, w), parameters, file) over the whole matrix."""
    for (h, w), noisy in itertools.product(sizes, (0, 1)):
        img = image(h, w, noisy)
        for q, s, r, o in itertools.product(QUALITIES, SAMPLING, RESTARTS, (0, 1)):
            yield (h, w), (q, s, r, o, noisy), encode(img, q, s, r, o)


@pytest.mark.parametrize("size", SIZES, ids=["%dx%d" % s for s in SIZES])
def test_oracle_is_cv2_imdecode(size):
    n = 0
    for _, params, buf in matrix_files([size]):
        for gray in (False, True):
            ref = cv2.imdecode(buf, cv2.IMREAD_GRAYSCALE if gray else cv2.IMREAD_COLOR)
            got = O.decode(buf, gray=gray)
            assert got.shape == ref.shape and np.array_equal(got, ref), (size, params, gray)
            n += 1
    assert n == 2 * len(QUALITIES) * len(SAMPLING) * len(RESTARTS) * 2 * 2


def test_parser_segments_and_tables():
    """One segment per restart interval, each ending before its RST marker; tables shared by files of one encoder
    pack once; every Huffman table's lookahead agrees with the canonical code."""
    img = image(37, 53, 1)
    for r in (0, 1, 3):
        buf = encode(img, 75, "420", r)
        h = J.parse(buf)
        mx, my, geo = h.geometry()
        assert (mx, my) == (4, 3) and geo[0][:2] == (8, 6) and geo[1][2:] == (27, 19)
        assert len(h.segments) == (1 if r == 0 else -(-mx * my // r))
        for b0, b1 in h.segments[:-1]:
            assert buf[b1] == 0xFF and 0xD0 <= buf[b1 + 1] <= 0xD7
        assert buf[h.segments[-1][1]:h.segments[-1][1] + 2].tolist() == [0xFF, 0xD9]
    files = [encode(image(16, 64, n), 75, "420", 1) for n in (0, 1)]
    parts, offs, head, data, nh, nq, fd, sd = J.pack([J.parse(f) for f in files], files)
    assert (nh, nq) == (4, 2) and data == sum(f.size for f in files)
    assert [p.size for p in parts] == [2 * 80, 8 * 24, 4 * 1424, 2 * 128]         # include/esf.h's layout
    assert offs == [0, 160, 352, 352 + 5696] and head == 352 + 5696 + 256
    assert sd["file"].tolist() == [0] * 4 + [1] * 4 and sd["first_mcu"].tolist() == [0, 1, 2, 3] * 2
    assert sd["begin"][4] >= files[0].size
    for counts, symbols in J.parse(files[1]).dc + J.parse(files[1]).ac:
        t = J.huffman_table(counts, symbols)
        canon = O._canonical(counts, symbols)
        for (ln, code), sym in canon.items():
            if ln <= J.HUFF_LOOKAHEAD:
                assert t["look"][code << (J.HUFF_LOOKAHEAD - ln)] == (ln << 8) | sym
            else:
                assert t["look"][code >> (ln - J.HUFF_LOOKAHEAD)] == 0
                assert code <= t["maxcode"][ln] and t["values"][code + t["valoffset"][ln]] == sym


def _find(buf, marker):
    b = bytes(buf)
    i = b.index(bytes([0xFF, marker]))
    return i


def _patched(buf, marker, offset, value):
    b = bytearray(bytes(buf))
    b[_find(buf, marker) + offset] = value
    return bytes(b)


def _with_exif_orientation(buf, orientation):
    tiff = b"II*\x00" + struct.pack("<I", 8) + struct.pack("<H", 1) + struct.pack("<HHIHH", 0x0112, 3, 1, orientation, 0) \
        + struct.pack("<I", 0)
    app1 = b"Exif\x00\x00" + tiff
    b = bytes(buf)
    return b[:2] + b"\xFF\xE1" + struct.pack(">H", len(app1) + 2) + app1 + b[2:]


def refusal_cases():
    img = image(16, 24, 1)
    base = encode(img, 80, "420")
    sof = 0xC0
    return {
        "progressive": (encode(img, 80, "420", progressive=1), "progressive"),
        "sof9": (_patched(base, sof, 1, 0xC9), "arithmetic"),
        "12-bit": (_patched(base, sof, 4, 12), "12-bit"),
        "4-components": (_patched(base, sof, 9, 4), "4 components"),
        "exif-orientation-6": (_with_exif_orientation(base, 6), "orientation 6"),
        "truncated": (bytes(base)[:len(base) // 2], "truncated"),
        "no-eoi": (bytes(base)[:-2], "truncated"),
    }


@pytest.mark.parametrize("case", sorted(refusal_cases()))
def test_refused_files(case):
    buf, what = refusal_cases()[case]
    with pytest.raises(ValueError, match=what):
        J.parse(buf)
    with pytest.raises(ValueError, match=what):     # before `out`'s device is looked at
        J.decode_jpeg([buf], torch.zeros(1, 16, 24, 3, dtype=torch.uint8))


def test_exif_orientation_1_and_other_markers_are_accepted():
    img = image(16, 24, 0)
    buf = _with_exif_orientation(encode(img, 80, "422"), 1)
    assert np.array_equal(O.decode(buf), cv2.imdecode(np.frombuffer(buf, np.uint8), cv2.IMREAD_COLOR))


def test_bad_out_is_refused():
    """dtype, device, contiguity, channel count, frame count: ValueError before any file is read or copied."""
    buf = encode(image(16, 24, 0), 80, "420")
    good = (1, 16, 24, 3)
    with pytest.raises(ValueError, match="uint8"):
        J.decode_jpeg([buf], torch.zeros(good, dtype=torch.float32))
    with pytest.raises(ValueError, match="CUDA"):
        J.decode_jpeg([buf], torch.zeros(good, dtype=torch.uint8))
    with pytest.raises(ValueError, match="files"):
        J.decode_jpeg([buf, buf], torch.zeros(good, dtype=torch.uint8))
    with pytest.raises(ValueError, match="bytes, bytearray"):
        J.decode_jpeg([buf, "x"], torch.zeros((2,) + good[1:], dtype=torch.uint8))
    with pytest.raises(ValueError, match="3 channels"):
        J.decode_jpeg([buf], torch.zeros(good, dtype=torch.uint8), gray=True)
    with pytest.raises(ValueError, match="contiguous"):
        J.decode_jpeg([buf], torch.zeros(1, 24, 16, 3, dtype=torch.uint8).transpose(1, 2))
    with pytest.raises(ValueError, match="at least one"):
        J.decode_jpeg([], torch.zeros(good, dtype=torch.uint8))


def test_size_mismatch_is_refused():
    buf = encode(image(16, 24, 0), 80, "420")
    with pytest.raises(ValueError, match="file 1 is 16 x 24, out's frames are 16 x 32"):
        J.decode_jpeg([encode(image(16, 32, 0)), buf], torch.zeros(2, 16, 32, 3, dtype=torch.uint8))


def _abi_args(files, gray=0):
    hdrs = [J.parse(f) for f in files]
    parts, offs, head, data, nh, nq, fd, sd = J.pack(hdrs, files)
    return fd, sd, head, head + data, nh, nq


ESF_ERR_ARG = -1


def test_cabi_argument_checks(esf_lib):
    """Every descriptor is checked on the host copies before any launch: each bad call returns ESF_ERR_ARG, which the
    library returns only before its first CUDA call (the device addresses below are fakes and are never reached)."""
    files = [encode(image(16, 24, n), 80, "420", r) for n, r in ((0, 1), (1, 0))]
    fd, sd, head, total, nh, nq = _abi_args(files)
    n = ctypes.c_int64()
    assert esf_lib.esf_jpeg_scratch_bytes(fd.ctypes.data, 2, 0, ctypes.addressof(n)) == 0
    assert n.value == 2 * ((12 * 64 * 2 + 255) // 256 * 256 + (12 * 64 + 255) // 256 * 256)
    assert esf_lib.esf_jpeg_scratch_bytes(None, 2, 0, ctypes.addressof(n)) == ESF_ERR_ARG
    assert esf_lib.esf_jpeg_scratch_bytes(fd.ctypes.data, 0, 0, ctypes.addressof(n)) == ESF_ERR_ARG
    fake = 1 << 40     # 16-byte aligned

    def call(fd=fd, sd=sd, nseg=len(sd), total=total, scratch=n.value, H=16, W=24, C=3, gray=0, nh=nh, blob=fake):
        return esf_lib.esf_jpeg_decode(blob, total, fd.ctypes.data, len(fd), sd.ctypes.data, nseg, nh, nq, fake,
                                       scratch, fake, H, W, C, gray, fake, None)

    def refused(what=b"", **kw):
        rc = call(**kw)
        return rc == ESF_ERR_ARG and what in esf_lib.esf_last_error()

    assert refused(blob=None)
    assert refused(b"misaligned", blob=fake + 8)
    assert refused(b"file 0 is 16 x 24", H=17)
    assert refused(C=1) and refused(gray=1)
    assert refused(b"scratch", scratch=n.value - 1)
    assert refused(b"outside", total=head + int(sd["end"].max()) - 1)
    assert refused(nseg=len(sd) - 1)
    assert refused(b"table index", nh=1)
    for field, value in (("file", 1), ("first_mcu", 5), ("begin", -1)):
        bad = sd.copy()
        bad[1][field] = value
        assert refused(sd=bad), field
    for field, value in (("ncomp", 2), ("restart", -1)):
        bad = fd.copy()
        bad[0][field] = value
        assert refused(fd=bad), field
    bad = fd.copy()
    bad[0]["h"][0], bad[0]["v"][0] = 3, 1
    assert refused(b"sampling", fd=bad)
