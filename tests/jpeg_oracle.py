"""A numpy restatement of the baseline decoder cv2.imdecode runs (the bundled libjpeg-turbo, default settings): Huffman
decoding (jdhuff.c), the islow IDCT (jidctint.c), fancy upsampling (jdsample.c) and the YCbCr -> BGR tables (jdcolor.c).
It shares the product's header parser (efficient_slowfast_b200.jpeg.parse) and nothing else, and is the CPU proof of the
rules the CUDA decoder follows."""
import numpy as np

from efficient_slowfast_b200 import jpeg as J

NATURAL = np.concatenate([J.ZIGZAG, np.full(16, 63)])   # libjpeg's jpeg_natural_order with its 16 guard entries


class _Bits:
    """MSB-first bit reader over one entropy-coded segment: FF 00 is a data byte FF; past the end it feeds zeros."""

    def __init__(self, data):
        out = bytearray()
        i, n = 0, len(data)
        while i < n:
            out.append(data[i])
            i += 2 if data[i] == 0xFF else 1
        self.s = "".join(format(x, "08b") for x in out)
        self.p = 0

    def get(self, k):
        if k == 0:
            return 0
        v = self.s[self.p:self.p + k]
        self.p += k
        return int(v.ljust(k, "0"), 2)


def _canonical(counts, symbols):
    """{(length, code): symbol} of one DHT entry."""
    table, code, p = {}, 0, 0
    for ln in range(1, 17):
        for _ in range(counts[ln - 1]):
            table[(ln, code)] = symbols[p]
            code += 1
            p += 1
        code <<= 1
    return table


def _decode_symbol(bits, table):
    code = 0
    for ln in range(1, 17):
        code = (code << 1) | bits.get(1)
        s = table.get((ln, code))
        if s is not None:
            return s
    raise ValueError("invalid Huffman code")


def _extend(v, s):
    return v - (1 << s) + 1 if s and v < (1 << (s - 1)) else v


def coefficients(buf, hdr=None):
    """Per component, int64 (block rows, blocks per row, 64) quantised coefficients in natural order."""
    hdr = hdr or J.parse(buf)
    mx, my, geo = hdr.geometry()
    coef = [np.zeros((bh, bw, 64), np.int64) for bw, bh, _, _ in geo]
    dcs = [_canonical(*t) for t in hdr.dc]
    acs = [_canonical(*t) for t in hdr.ac]
    total = mx * my
    per = hdr.restart or total
    single = len(hdr.comps) == 1
    for si, (b0, b1) in enumerate(hdr.segments):
        bits = _Bits(buf[b0:b1])
        pred = [0] * len(hdr.comps)
        for m in range(si * per, min(total, (si + 1) * per)):
            ry, rx = divmod(m, mx)
            for c, (h, v) in enumerate(hdr.comps):
                for by, bx in ([(ry, rx)] if single else [(ry * v + a, rx * h + e) for a in range(v) for e in range(h)]):
                    blk = coef[c][by, bx]
                    s = _decode_symbol(bits, dcs[c])
                    pred[c] += _extend(bits.get(s), s)
                    blk[0] = np.int16(pred[c])
                    k = 1
                    while k < 64:
                        rs = _decode_symbol(bits, acs[c])
                        r, s = rs >> 4, rs & 15
                        if s:
                            k += r
                            blk[NATURAL[k]] = _extend(bits.get(s), s)
                        elif r != 15:
                            break
                        else:
                            k += 15
                        k += 1
    return hdr, coef


C13 = {"0_298631336": 2446, "0_390180644": 3196, "0_541196100": 4433, "0_765366865": 6270, "0_899976223": 7373,
       "1_175875602": 9633, "1_501321110": 12299, "1_847759065": 15137, "1_961570560": 16069, "2_053119869": 16819,
       "2_562915447": 20995, "3_072711026": 25172}


def _idct_1d(x, shift):
    """jidctint.c's 8-point pass on axis 1 of x (N, 8, M), descaled by `shift` with rounding."""
    k = C13
    z1 = (x[:, 2] + x[:, 6]) * k["0_541196100"]
    tmp2 = z1 - x[:, 6] * k["1_847759065"]
    tmp3 = z1 + x[:, 2] * k["0_765366865"]
    tmp0 = (x[:, 0] + x[:, 4]) << 13
    tmp1 = (x[:, 0] - x[:, 4]) << 13
    t10, t13, t11, t12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
    a0, a1, a2, a3 = x[:, 7], x[:, 5], x[:, 3], x[:, 1]
    z1, z2, z3, z4 = a0 + a3, a1 + a2, a0 + a2, a1 + a3
    z5 = (z3 + z4) * k["1_175875602"]
    a0 = a0 * k["0_298631336"]
    a1 = a1 * k["2_053119869"]
    a2 = a2 * k["3_072711026"]
    a3 = a3 * k["1_501321110"]
    z1 = z1 * -k["0_899976223"]
    z2 = z2 * -k["2_562915447"]
    z3 = z3 * -k["1_961570560"] + z5
    z4 = z4 * -k["0_390180644"] + z5
    a0 += z1 + z3
    a1 += z2 + z4
    a2 += z2 + z3
    a3 += z1 + z4
    r = 1 << (shift - 1)
    out = [t10 + a3, t11 + a2, t12 + a1, t13 + a0, t13 - a0, t12 - a1, t11 - a2, t10 - a3]
    return np.stack([(o + r) >> shift for o in out], axis=1)


def idct_islow(coef, quant):
    """(N, 64) natural-order coefficients and int16[64] quantisation -> (N, 8, 8) uint8 samples."""
    x = (coef.astype(np.int64) * quant.astype(np.int64)).reshape(-1, 8, 8)     # [n, row (v), col (u)]
    ws = _idct_1d(x, 13 - 2)                                                     # columns: pass 1, PASS1_BITS 2
    y = _idct_1d(ws.transpose(0, 2, 1), 13 + 2 + 3).transpose(0, 2, 1)         # rows: pass 2
    y = ((y + 512) & 1023) - 512                                                 # range_limit[x & RANGE_MASK]
    return np.clip(y + 128, 0, 255).astype(np.uint8)


def planes(hdr, coef, comps):
    """Component planes (block rows * 8, blocks per row * 8) uint8 of the components in `comps`."""
    out = []
    for c in comps:
        bh, bw, _ = coef[c].shape
        s = idct_islow(coef[c].reshape(-1, 64), hdr.quant[c]).reshape(bh, bw, 8, 8)
        out.append(s.transpose(0, 2, 1, 3).reshape(bh * 8, bw * 8))
    return out


def upsample(p, cw, ch, h, v, hm, vm, H, W):
    """libjpeg-turbo's upsampling of one component plane (real size ch x cw) to H x W."""
    p = p[:ch, :cw].astype(np.int64)
    fx, fy = hm // h, vm // v
    ys, xs = np.arange(H), np.arange(W)
    if (fx, fy) == (1, 1):
        return p[:H, :W]
    if (fx, fy) == (2, 1) and cw > 2:
        j = xs >> 1
        other = np.where(xs & 1, np.minimum(j + 1, cw - 1), np.maximum(j - 1, 0))
        return (3 * p[:, j] + p[:, other] + np.where(xs & 1, 2, 1)) >> 2
    if (fx, fy) == (1, 2):
        i = ys >> 1
        other = np.where(ys & 1, np.minimum(i + 1, ch - 1), np.maximum(i - 1, 0))
        return (3 * p[i] + p[other] + np.where(ys & 1, 2, 1)[:, None]) >> 2
    if (fx, fy) == (2, 2) and cw > 2:
        i = ys >> 1
        other = np.where(ys & 1, np.minimum(i + 1, ch - 1), np.maximum(i - 1, 0))
        cs = 3 * p[i] + p[other]                                                   # (H, cw) column sums
        j = xs >> 1
        nb = np.where(xs & 1, np.minimum(j + 1, cw - 1), np.maximum(j - 1, 0))
        return (3 * cs[:, j] + cs[:, nb] + np.where(xs & 1, 7, 8)) >> 4
    return p[ys // fy][:, xs // fx]                                                 # replication (h2v1 / h2v2 narrow, h4v1)


SCALEBITS, ONE_HALF = 16, 1 << 15


def _fix(x):
    return int(x * (1 << SCALEBITS) + 0.5)


def ycc_to_bgr(y, cb, cr):
    cb, cr = cb - 128, cr - 128
    r = y + ((_fix(1.40200) * cr + ONE_HALF) >> SCALEBITS)
    g = y + ((-_fix(0.34414) * cb + ONE_HALF - _fix(0.71414) * cr) >> SCALEBITS)
    b = y + ((_fix(1.77200) * cb + ONE_HALF) >> SCALEBITS)
    return np.clip(np.stack([b, g, r], axis=-1), 0, 255).astype(np.uint8)


def decode(buf, gray=False):
    """cv2.imdecode(buf, IMREAD_GRAYSCALE if gray else IMREAD_COLOR), restated: (H, W) or (H, W, 3) uint8."""
    buf = bytes(buf)
    hdr, coef = coefficients(buf)
    H, W = hdr.height, hdr.width
    _, _, geo = hdr.geometry()
    ncomp = len(hdr.comps)
    pl = planes(hdr, coef, [0] if gray or ncomp == 1 else range(ncomp))
    y = pl[0][:H, :W].astype(np.int64)
    if gray:
        return y.astype(np.uint8)
    if ncomp == 1:
        return np.repeat(y.astype(np.uint8)[..., None], 3, axis=2)
    hm = max(h for h, _ in hdr.comps)
    vm = max(v for _, v in hdr.comps)
    ch = [upsample(pl[c], geo[c][2], geo[c][3], *hdr.comps[c], hm, vm, H, W) for c in (1, 2)]
    return ycc_to_bgr(y, *ch)
