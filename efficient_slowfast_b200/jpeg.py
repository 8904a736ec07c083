"""Baseline JPEG frames decoded on the device, bit-identical to cv2.imdecode (the bundled libjpeg-turbo).

The reference's frame-directory loaders (slowfast/datasets/utils.py retry_load_images, used by the AVA, Charades and SSv2
datasets) read every frame with cv2.imread.  decode_jpeg(files, out) does that decode for a batch of frames on the
device: this module walks each file's markers on the host (per-header work and numpy passes over the compressed bytes),
packs the files, their descriptors and the Huffman / quantisation tables into one pinned buffer, uploads it with one
cudaMemcpyAsync and runs esf_jpeg_decode (csrc/esf_jpeg.cu): Huffman decoding with one thread per entropy-coded
segment, libjpeg's islow IDCT, and libjpeg-turbo's fancy chroma upsampling and YCbCr -> BGR tables written into `out`.

What the decoder does not restate is refused with ValueError before anything is copied or launched: progressive,
lossless, arithmetic-coded and 12-bit files, more than one scan, 2 or 4 components, a colour transform other than
YCbCr, sampling other than 4:4:4, 4:2:2, 4:2:0, 4:4:0 and 4:1:1 with 1x1 chroma, an EXIF orientation other than 1 (cv2
would rotate the frame), and files that are truncated or not framed as their headers say.
"""
import ctypes

import numpy as np
import torch

# The layouts of include/esf.h: esf_jpeg_file (20 int32) and esf_jpeg_segment (int64 begin, end; int32 file, first_mcu)
FILE_DTYPE = np.dtype([("H", "<i4"), ("W", "<i4"), ("ncomp", "<i4"), ("restart", "<i4"), ("h", "<i4", 3),
                       ("v", "<i4", 3), ("qt", "<i4", 3), ("dc", "<i4", 3), ("ac", "<i4", 3), ("pad", "<i4")])
SEGMENT_DTYPE = np.dtype([("begin", "<i8"), ("end", "<i8"), ("file", "<i4"), ("first_mcu", "<i4")])
HUFF_LOOKAHEAD = 9
# one device Huffman table: uint16 look[512] (code length << 8 | symbol, 0: longer than 9 bits), int32 maxcode[18],
# int32 valoffset[18], uint8 values[256]
HUFF_DTYPE = np.dtype([("look", "<u2", 1 << HUFF_LOOKAHEAD), ("maxcode", "<i4", 18), ("valoffset", "<i4", 18),
                       ("values", "u1", 256)])
ALIGN = 16

# luma sampling factors (h, v) cv2.imencode writes (IMWRITE_JPEG_SAMPLING_FACTOR_444, 422, 420, 440, 411)
LUMA_SAMPLING = ((1, 1), (2, 1), (2, 2), (1, 2), (4, 1))

ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13,
                   6, 7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45,
                   38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63], dtype=np.int64)   # zig-zag index -> natural index


class JpegHeader:
    """What the decoder needs of one baseline file: size, components, the tables its scan uses and the byte ranges of
    its entropy-coded segments (one per restart interval, or the whole scan), as offsets into the file."""
    __slots__ = ("height", "width", "comps", "quant", "dc", "ac", "restart", "segments")

    def __init__(self, height, width, comps, quant, dc, ac, restart, segments):
        self.height, self.width = height, width
        self.comps = comps          # [(h, v)] per component, in scan order
        self.quant = quant          # [int16[64] natural order, as libjpeg's ISLOW_MULT_TYPE holds it] per component
        self.dc, self.ac = dc, ac   # [(counts bytes[16], symbols bytes)] per component
        self.restart = restart      # MCUs per restart interval, 0: none
        self.segments = segments    # [(begin, end)] entropy-coded bytes, markers and fill bytes excluded

    def geometry(self):
        """(MCUs per row, MCU rows, [(blocks per row, block rows, width, height) per component]) as libjpeg derives
        them.  A single-component scan is not interleaved: its MCU is one block whatever the sampling factors."""
        H, W = self.height, self.width
        if len(self.comps) == 1:
            mx, my = -(-W // 8), -(-H // 8)
            return mx, my, [(mx, my, W, H)]
        hm = max(h for h, _ in self.comps)
        vm = max(v for _, v in self.comps)
        mx, my = -(-W // (8 * hm)), -(-H // (8 * vm))
        return mx, my, [(mx * h, my * v, -(-W * h // hm), -(-H * v // vm)) for h, v in self.comps]


def _u16(b, i):
    return (b[i] << 8) | b[i + 1]


def _exif_orientation(seg):
    """Orientation (tag 0x0112) of IFD0 of an APP1 Exif payload, or None."""
    if len(seg) < 14 or bytes(seg[:6]) != b"Exif\x00\x00":
        return None
    t = bytes(seg[6:])
    if t[:2] == b"II":
        order = "little"
    elif t[:2] == b"MM":
        order = "big"
    else:
        return None
    rd = lambda o, n: int.from_bytes(t[o:o + n], order)  # noqa: E731
    ifd = rd(4, 4)
    if ifd + 2 > len(t):
        return None
    for k in range(rd(ifd, 2)):
        e = ifd + 2 + 12 * k
        if e + 12 > len(t):
            return None
        if rd(e, 2) == 0x0112:
            return rd(e + 8, 2) if rd(e + 2, 2) == 3 else rd(e + 8, 4)
    return None


_SOF_NAMES = {0xC2: "progressive (SOF2)", 0xC3: "lossless (SOF3)", 0xC5: "differential (SOF5)",
              0xC6: "differential progressive (SOF6)", 0xC7: "differential lossless (SOF7)"}


def parse(buf):
    """JpegHeader of one baseline file (bytes-like or 1-D uint8 array); ValueError for what the decoder refuses."""
    b = np.frombuffer(buf, dtype=np.uint8) if not isinstance(buf, np.ndarray) else buf
    if b.ndim != 1 or b.dtype != np.uint8:
        raise ValueError("a JPEG file is bytes, bytearray, memoryview or a 1-D uint8 array")
    n = b.size
    b = memoryview(b)               # indexing yields Python ints
    if n < 4 or b[0] != 0xFF or b[1] != 0xD8:
        raise ValueError("not a JPEG file (no SOI marker)")
    pos = 2
    qt, huff = {}, {}
    frame = None
    restart = 0
    jfif = adobe = False
    adobe_transform = None
    scan = None
    while True:
        if pos >= n:
            raise ValueError("truncated JPEG file: no EOI marker")
        if b[pos] != 0xFF:
            raise ValueError("corrupt JPEG file: expected a marker at byte %d" % pos)
        while pos < n and b[pos] == 0xFF:
            pos += 1
        if pos >= n:
            raise ValueError("truncated JPEG file: no EOI marker")
        m = int(b[pos])
        pos += 1
        if m == 0xD9:
            break
        if 0xD0 <= m <= 0xD7 or m == 0x01:
            raise ValueError("corrupt JPEG file: marker 0x%02X outside a scan" % m)
        if pos + 2 > n:
            raise ValueError("truncated JPEG file: marker 0x%02X runs past the end" % m)
        L = _u16(b, pos)
        if L < 2 or pos + L > n:
            raise ValueError("truncated JPEG file: marker 0x%02X segment runs past the end" % m)
        seg = b[pos + 2:pos + L]
        pos += L
        if m in (0xC0, 0xC1):
            if frame is not None:
                raise ValueError("corrupt JPEG file: more than one SOF marker")
            if len(seg) < 6:
                raise ValueError("corrupt JPEG file: short SOF segment")
            if seg[0] != 8:
                raise ValueError("%d-bit JPEG files are not supported (8-bit precision only)" % seg[0])
            H, W, nc = _u16(seg, 1), _u16(seg, 3), int(seg[5])
            if nc not in (1, 3):
                raise ValueError("JPEG files with %d components are not supported (1 or 3; no CMYK/YCCK)" % nc)
            if len(seg) < 6 + 3 * nc:
                raise ValueError("corrupt JPEG file: short SOF segment")
            if H == 0 or W == 0:
                raise ValueError("JPEG files whose height is set by a DNL marker are not supported")
            frame = (H, W, [(int(seg[6 + 3 * i]), int(seg[7 + 3 * i]) >> 4, int(seg[7 + 3 * i]) & 15,
                             int(seg[8 + 3 * i])) for i in range(nc)])
        elif m in _SOF_NAMES:
            raise ValueError("%s JPEG files are not supported (baseline only)" % _SOF_NAMES[m])
        elif 0xC9 <= m <= 0xCF:
            raise ValueError("arithmetic-coded JPEG files (marker 0x%02X) are not supported" % m)
        elif m == 0xC4:
            i = 0
            while i < len(seg):
                if i + 17 > len(seg):
                    raise ValueError("corrupt JPEG file: short DHT segment")
                tc, th = int(seg[i]) >> 4, int(seg[i]) & 15
                counts = bytes(seg[i + 1:i + 17])
                total = sum(counts)
                if tc > 1 or th > 3 or total > 256 or i + 17 + total > len(seg):
                    raise ValueError("corrupt JPEG file: bad DHT segment")
                huff[(tc, th)] = (counts, bytes(seg[i + 17:i + 17 + total]))
                i += 17 + total
        elif m == 0xDB:
            i = 0
            while i < len(seg):
                pq, tq = int(seg[i]) >> 4, int(seg[i]) & 15
                size = 128 if pq else 64
                if pq > 1 or tq > 3 or i + 1 + size > len(seg):
                    raise ValueError("corrupt JPEG file: bad DQT segment")
                raw = np.frombuffer(seg[i + 1:i + 1 + size], np.uint8)
                zz = (raw[0::2].astype(np.int64) << 8 | raw[1::2]) if pq else raw.astype(np.int64)
                nat = np.empty(64, np.int64)
                nat[ZIGZAG] = zz
                qt[tq] = nat.astype(np.uint16).view(np.int16)
                i += 1 + size
        elif m == 0xDD:
            if len(seg) < 2:
                raise ValueError("corrupt JPEG file: short DRI segment")
            restart = _u16(seg, 0)
        elif m == 0xE0:
            jfif = jfif or bytes(seg[:5]) == b"JFIF\x00"
        elif m == 0xE1:
            o = _exif_orientation(seg)
            if o is not None and o != 1:
                raise ValueError("EXIF orientation %d is not supported (cv2.imdecode would rotate the frame)" % o)
        elif m == 0xEE:
            if len(seg) >= 12 and bytes(seg[:5]) == b"Adobe":
                adobe, adobe_transform = True, int(seg[11])
        elif m == 0xDC:
            raise ValueError("JPEG files with a DNL marker are not supported")
        elif m == 0xDA:
            if scan is not None:
                raise ValueError("multi-scan JPEG files are not supported (one interleaved scan only)")
            if frame is None:
                raise ValueError("corrupt JPEG file: SOS before SOF")
            ns = int(seg[0]) if len(seg) else 0
            if len(seg) < 4 + 2 * ns:
                raise ValueError("corrupt JPEG file: short SOS segment")
            H, W, comps = frame
            if ns != len(comps) or [int(seg[1 + 2 * i]) for i in range(ns)] != [c[0] for c in comps]:
                raise ValueError("multi-scan JPEG files are not supported (one interleaved scan only)")
            ss, se, ahl = int(seg[1 + 2 * ns]), int(seg[2 + 2 * ns]), int(seg[3 + 2 * ns])
            if ss != 0 or se != 63 or ahl != 0:
                raise ValueError("corrupt JPEG file: spectral selection of a sequential scan")
            sel = [(int(seg[2 + 2 * i]) >> 4, int(seg[2 + 2 * i]) & 15) for i in range(ns)]
            try:
                quant = [qt[c[3]] for c in comps]
                dc = [huff[(0, td)] for td, _ in sel]
                ac = [huff[(1, ta)] for _, ta in sel]
            except KeyError:
                raise ValueError("corrupt JPEG file: the scan uses an undefined table") from None
            segments, pos = _scan_segments(b.obj, pos)
            scan = (quant, dc, ac, segments)
    if frame is None or scan is None:
        raise ValueError("corrupt JPEG file: no frame or no scan")
    H, W, comps = frame
    if len(comps) == 3:
        if jfif:
            rgb = False
        elif adobe:
            rgb = adobe_transform == 0
            if adobe_transform not in (0, 1):
                raise ValueError("Adobe colour transform %d is not supported (YCbCr only)" % adobe_transform)
        else:
            rgb = [c[0] for c in comps] == [82, 71, 66]
        if rgb:
            raise ValueError("RGB JPEG files are not supported (YCbCr only)")
        samp = [(c[1], c[2]) for c in comps]
        if samp[1] != (1, 1) or samp[2] != (1, 1) or samp[0] not in LUMA_SAMPLING:
            raise ValueError("JPEG sampling %s is not supported (luma 1x1, 2x1, 2x2, 1x2 or 4x1 with 1x1 chroma)"
                             % "/".join("%dx%d" % s for s in samp))
    else:
        samp = [(1, 1)]
    quant, dc, ac, segments = scan
    for t in dc:
        if max(t[1], default=0) > 15:
            raise ValueError("corrupt JPEG file: bad DC Huffman table")
    hdr = JpegHeader(H, W, samp, quant, dc, ac, restart, segments)
    mx, my, _ = hdr.geometry()
    want = -(-mx * my // restart) if restart else 1
    if len(segments) != want:
        raise ValueError("corrupt JPEG file: %d entropy-coded segments where the header implies %d"
                         % (len(segments), want))
    for t in dc + ac:
        huffman_table(*t)            # refuses a table libjpeg refuses
    return hdr


def _scan_segments(b, start):
    """Entropy-coded segments of the scan starting at `start` and the position of the marker that ends it.  A marker
    is 0xFF followed by neither 0x00 (a stuffed data byte) nor 0xFF (fill); fill bytes before it are not data."""
    d = b[start:]
    ff = np.flatnonzero(d[:-1] == 0xFF)
    nxt = d[ff + 1]
    marks = ff[(nxt != 0x00) & (nxt != 0xFF)]
    segments = []
    begin = start
    expect = 0
    for mk in marks.tolist():
        code = int(d[mk + 1])
        end = mk
        while end > 0 and d[end - 1] == 0xFF and start + end > begin:
            end -= 1
        segments.append((begin, start + end))
        if 0xD0 <= code <= 0xD7:
            if code != 0xD0 + expect:
                raise ValueError("corrupt JPEG file: restart marker RST%d where RST%d was due" % (code - 0xD0, expect))
            expect = (expect + 1) & 7
            begin = start + mk + 2
            continue
        return segments, start + mk
    raise ValueError("truncated JPEG file: the scan runs past the end of the file")


_HUFF_CACHE = {}


def huffman_table(counts, symbols):
    """The device table (HUFF_DTYPE) of one DHT entry, cached by its bytes: libjpeg's jpeg_make_d_derived_tbl
    (maxcode, valoffset) plus a 9-bit lookahead.  ValueError for a table libjpeg refuses (a code of all ones)."""
    key = counts + symbols
    t = _HUFF_CACHE.get(key)
    if t is not None:
        return t
    t = np.zeros((), HUFF_DTYPE)
    t["values"][:len(symbols)] = np.frombuffer(symbols, np.uint8)
    t["maxcode"][:] = -1
    code, p = 0, 0
    look = t["look"]
    for ln in range(1, 17):
        c = counts[ln - 1]
        t["valoffset"][ln] = p - code
        if c:
            if ln <= HUFF_LOOKAHEAD:
                for k in range(c):
                    lo = (code + k) << (HUFF_LOOKAHEAD - ln)
                    look[lo:lo + (1 << (HUFF_LOOKAHEAD - ln))] = (ln << 8) | symbols[p + k]
            code += c
            p += c
            t["maxcode"][ln] = code - 1
        if code >= (1 << ln):
            raise ValueError("corrupt JPEG file: bad Huffman table")
        code <<= 1
    t["maxcode"][17] = 0xFFFFF
    if len(_HUFF_CACHE) > 4096:
        _HUFF_CACHE.clear()
    _HUFF_CACHE[key] = t
    return t


def _as_array(f):
    if isinstance(f, np.ndarray):
        if f.ndim != 1 or f.dtype != np.uint8:
            raise ValueError("a JPEG file array must be 1-D uint8, got %s %s" % (f.dtype, f.shape))
        return np.ascontiguousarray(f)
    if isinstance(f, (bytes, bytearray, memoryview)):
        return np.frombuffer(f, dtype=np.uint8)
    raise ValueError("JPEG files are bytes, bytearray, memoryview or 1-D uint8 arrays, got %s" % type(f).__name__)


def _check_out(out, nfiles, gray):
    if not isinstance(out, torch.Tensor):
        raise ValueError("out must be a torch.Tensor")
    if out.dtype != torch.uint8:
        raise ValueError("out must be uint8, got %s" % out.dtype)
    if not out.is_contiguous():
        raise ValueError("out must be contiguous")
    if out.dim() < 3:
        raise ValueError("out must be (..., H, W, C), got %s" % tuple(out.shape))
    C = out.shape[-1]
    if C != (1 if gray else 3):
        raise ValueError("out has %d channels; gray=%s decodes to %d" % (C, gray, 1 if gray else 3))
    if out.numel() // max(1, out.shape[-3] * out.shape[-2] * C) != nfiles or out.numel() == 0:
        raise ValueError("out's leading dims %s hold %d frames, not the %d files"
                         % (tuple(out.shape[:-3]), out.numel() // max(1, out.shape[-3] * out.shape[-2] * C), nfiles))
    return int(out.shape[-3]), int(out.shape[-2]), int(C)


def _aligned(x):
    return (x + ALIGN - 1) // ALIGN * ALIGN


def pack(headers, arrays):
    """(blob uint8 array, n_huff, n_quant, files, segments) in the layout esf_jpeg_decode reads: file descriptors,
    segments, Huffman tables, quantisation tables, then the files' bytes (segment offsets count from there).  Tables
    that repeat across files are stored once."""
    n = len(headers)
    files = np.zeros(n, FILE_DTYPE)
    nseg = sum(len(h.segments) for h in headers)
    segs = np.zeros(nseg, SEGMENT_DTYPE)
    huff_ix, quant_ix = {}, {}
    huffs, quants = [], []
    s = 0
    data_off = 0
    for i, (h, a) in enumerate(zip(headers, arrays)):
        f = files[i]
        f["H"], f["W"], f["ncomp"], f["restart"] = h.height, h.width, len(h.comps), h.restart
        for c, (hs, vs) in enumerate(h.comps):
            f["h"][c], f["v"][c] = hs, vs
            qk = h.quant[c].tobytes()
            if qk not in quant_ix:
                quant_ix[qk] = len(quants)
                quants.append(h.quant[c])
            f["qt"][c] = quant_ix[qk]
            for field, t in (("dc", h.dc[c]), ("ac", h.ac[c])):
                k = t[0] + t[1]
                if k not in huff_ix:
                    huff_ix[k] = len(huffs)
                    huffs.append(huffman_table(*t))
                f[field][c] = huff_ix[k]
        ns = len(h.segments)
        seg = np.asarray(h.segments, np.int64).reshape(ns, 2)
        segs["begin"][s:s + ns] = seg[:, 0] + data_off
        segs["end"][s:s + ns] = seg[:, 1] + data_off
        segs["file"][s:s + ns] = i
        segs["first_mcu"][s:s + ns] = np.arange(ns) * h.restart
        s += ns
        data_off += a.size
    parts = [files.view(np.uint8), segs.view(np.uint8), np.array(huffs, HUFF_DTYPE).view(np.uint8),
             np.stack(quants).astype("<i2").view(np.uint8).reshape(-1)]
    offs = []
    size = 0
    for p in parts:
        offs.append(size)
        size = _aligned(size + p.size)
    return parts, offs, size, data_off, len(huffs), len(quants), files, segs


class _Staging:
    """Two pinned upload buffers, each rewritten only after the copy that last read it has finished."""

    def __init__(self):
        self.bufs = [None, None]
        self.events = [None, None]
        self.turn = 0

    def take(self, nbytes):
        i = self.turn
        self.turn ^= 1
        if self.events[i] is not None:
            self.events[i].synchronize()
        if self.bufs[i] is None or self.bufs[i].numel() < nbytes:
            self.bufs[i] = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, pin_memory=True)
        return i, self.bufs[i]

    def copied(self, i):
        ev = torch.cuda.Event()
        ev.record()
        self.events[i] = ev


_STAGING = _Staging()


def decode_jpeg(files, out, gray=False):
    """Decode baseline JPEG files into `out`, bit-identical to cv2.imdecode(buf, cv2.IMREAD_COLOR) (BGR) or, with
    gray=True, cv2.IMREAD_GRAYSCALE.

    files: a list of bytes, bytearray, memoryview or 1-D uint8 numpy arrays, one JPEG file per frame.  out: a
    contiguous uint8 CUDA tensor (..., H, W, C) whose leading dims flatten to len(files) in C order, C = 3 (1 with
    gray=True); every file must be H x W.  Asynchronous on the current stream, with no synchronisation.  Returns a
    device int32 tensor with one entry per file: 0, or nonzero when the file's scan holds an invalid Huffman code (that
    frame's pixels are then unspecified; the other frames are unaffected).  Raises ValueError, before anything is
    copied or launched, for a file or an `out` the decoder does not take (see the module docstring)."""
    from . import runtime as rt

    files = list(files)
    if not files:
        raise ValueError("decode_jpeg needs at least one file")
    H, W, C = _check_out(out, len(files), gray)
    arrays = [_as_array(f) for f in files]
    headers = []
    for i, a in enumerate(arrays):
        try:
            h = parse(a)
        except ValueError as e:
            raise ValueError("file %d: %s" % (i, e)) from None
        if (h.height, h.width) != (H, W):
            raise ValueError("file %d is %d x %d, out's frames are %d x %d" % (i, h.height, h.width, H, W))
        headers.append(h)
    if not out.is_cuda:
        raise ValueError("out must be a CUDA tensor")
    parts, offs, head_bytes, data_bytes, nh, nq, fdesc, sdesc = pack(headers, arrays)
    total = head_bytes + data_bytes
    L = rt.lib()
    dev_index = out.device.index
    with torch.cuda.device(dev_index):
        scratch_bytes = ctypes.c_int64()
        rt.check(L.esf_jpeg_scratch_bytes(fdesc.ctypes.data, len(files), int(gray), ctypes.addressof(scratch_bytes)),
                 "esf_jpeg_scratch_bytes")
        slot, host = _STAGING.take(total)
        hv = host.numpy()
        for p, o in zip(parts, offs):
            hv[o:o + p.size] = p
        o = head_bytes
        for a in arrays:
            hv[o:o + a.size] = a
            o += a.size
        blob = torch.empty(total, dtype=torch.uint8, device=out.device)
        blob.copy_(host[:total], non_blocking=True)
        _STAGING.copied(slot)
        scratch = torch.empty(max(1, scratch_bytes.value), dtype=torch.uint8, device=out.device)
        status = torch.empty(len(files), dtype=torch.int32, device=out.device)
        rt.check(L.esf_jpeg_decode(blob.data_ptr(), total, fdesc.ctypes.data, len(files), sdesc.ctypes.data,
                                   len(sdesc), nh, nq, scratch.data_ptr(), scratch_bytes.value, out.data_ptr(), H, W,
                                   C, int(gray), status.data_ptr(), rt.current_stream_ptr()), "esf_jpeg_decode")
    return status
