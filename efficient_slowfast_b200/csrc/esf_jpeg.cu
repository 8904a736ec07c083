// Baseline JPEG decoding bit-identical to cv2.imdecode (OpenCV's bundled libjpeg-turbo with its default settings), for
// the frame-directory loaders of the reference (slowfast/datasets/utils.py retry_load_images: cv2.imread per frame).
//
// The host (efficient_slowfast_b200/jpeg.py) parses every file's markers and packs one blob (layout in include/esf.h):
// file descriptors, entropy-coded segments, Huffman tables, quantisation tables, then the files' bytes.  Three launches:
//
//   1. jpeg_huffman_kernel: one thread (lane 0 of its own warp) per entropy-coded segment (a restart interval, or the
//      whole scan), all segments of all files in parallel.  jdhuff.c's decode_mcu: DC prediction reset at every segment, FF 00 byte stuffing, runs
//      through the zig-zag order (with libjpeg's 16 guard entries), int16 coefficients in natural order.  An invalid code
//      sets the file's status and decodes as symbol 0, as libjpeg does; past its segment the reader feeds zero bits.
//      The coefficient area is zeroed first (cudaMemsetAsync), so only the coded coefficients are stored.
//   2. jpeg_idct_kernel: jidctint.c's jpeg_idct_islow (CONST_BITS 13, PASS1_BITS 2, range limit of x & 1023 around
//      128), eight lanes per 8x8 block: lane j runs column j (pass 1), then row j (pass 2), through shared memory.
//   3. jpeg_color_kernel: one thread per pixel.  jdsample.c's upsampling of each chroma plane -- the "fancy" triangle
//      filters for h2v1 and h2v2 when the plane is wider than 2 samples (else replication), always for h1v2, integral
//      replication for h4v1 -- with edges replicating the last real row / column, then jdcolor.c's ycc_rgb_convert
//      (FIX(1.40200), FIX(1.77200), FIX(0.71414), FIX(0.34414), SCALEBITS 16, ONE_HALF) written as BGR into `out`.
//      Grey output is the Y plane (chroma is decoded by the Huffman stage only to be skipped); a one-component file in
//      colour mode is replicated to three channels.
//
// Scratch (esf_jpeg_scratch_bytes): per file, the int16 coefficients of the components the output needs, then their
// sample planes (blocks per row * 8 wide, block rows * 8 high), at one stride per call.
#include <algorithm>

#include "esf_common.cuh"
#include "esf_host.h"

namespace esf {

constexpr int kHuffLook = 9;

struct HuffTab {                     // jpeg.py HUFF_DTYPE
  uint16_t look[1 << kHuffLook];     // code length << 8 | symbol for codes of <= 9 bits, else 0
  int32_t maxcode[18];               // libjpeg's jpeg_make_d_derived_tbl
  int32_t valoffset[18];
  uint8_t values[256];
};
static_assert(sizeof(HuffTab) == 1424, "HuffTab is jpeg.py's HUFF_DTYPE");
static_assert(sizeof(esf_jpeg_file) == 80 && sizeof(esf_jpeg_segment) == 24, "descriptor layouts of include/esf.h");

// libjpeg's jpeg_natural_order: zig-zag index -> natural index, with 16 guard entries for runs past the last coefficient
__constant__ uint8_t kNatural[80] = {
    0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13,
    6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31,
    39, 46, 53, 60, 61, 54, 47, 55, 62, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63};

inline __host__ __device__ long long align16(long long x) { return (x + 15) & ~15LL; }

// Offsets of the blob's sections (include/esf.h)
struct JpegLayout {
  long long segs, huff, quant, data;
};
inline JpegLayout jpeg_layout(int n_files, int n_segs, int n_huff, int n_quant) {
  JpegLayout L;
  L.segs = align16((long long)n_files * sizeof(esf_jpeg_file));
  L.huff = align16(L.segs + (long long)n_segs * sizeof(esf_jpeg_segment));
  L.quant = align16(L.huff + (long long)n_huff * sizeof(HuffTab));
  L.data = align16(L.quant + (long long)n_quant * 128);
  return L;
}

// libjpeg's geometry of one file (jdinput.c initial_setup / per_scan_setup), restricted to the components stored:
// all of them, or the luma plane only for grey output.
struct JpegGeom {
  int mcux, mcuy, ncomp, nstore;
  int hmax, vmax;
  int bw[3], bh[3];          // blocks per row, block rows
  int cw[3], ch[3];          // real (downsampled) width and height
  long long blk0[3];         // first block of the component in the file's coefficient area
  long long plane0[3];       // first byte of the component's plane
  long long blocks, plane_bytes;
};

inline __host__ __device__ JpegGeom jpeg_geom(const esf_jpeg_file& f, int gray) {
  JpegGeom g;
  g.ncomp = f.ncomp;
  g.nstore = gray ? 1 : f.ncomp;
  if (f.ncomp == 1) {
    g.hmax = g.vmax = 1;
    g.mcux = (f.W + 7) / 8;
    g.mcuy = (f.H + 7) / 8;
  } else {
    g.hmax = f.h[0], g.vmax = f.v[0];   // chroma is 1x1 (checked)
    g.mcux = (f.W + 8 * g.hmax - 1) / (8 * g.hmax);
    g.mcuy = (f.H + 8 * g.vmax - 1) / (8 * g.vmax);
  }
  g.blocks = 0, g.plane_bytes = 0;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const int h = f.ncomp == 1 ? 1 : f.h[c], v = f.ncomp == 1 ? 1 : f.v[c];
    g.bw[c] = g.mcux * h, g.bh[c] = g.mcuy * v;
    g.cw[c] = (f.W * h + g.hmax - 1) / g.hmax;
    g.ch[c] = (f.H * v + g.vmax - 1) / g.vmax;
    g.blk0[c] = g.blocks, g.plane0[c] = g.plane_bytes;
    if (c < g.nstore) {
      g.blocks += (long long)g.bw[c] * g.bh[c];
      g.plane_bytes += (long long)g.bw[c] * g.bh[c] * 64;
    }
  }
  return g;
}

// MSB-first bit reader over [p, e): FF 00 is the data byte FF; past the end it feeds zero bits (libjpeg's behaviour at
// a marker).  fill() leaves at least 57 bits, enough for a code (<= 16) and its extra bits (<= 15).
struct BitReader {
  const uint8_t* p;
  const uint8_t* e;
  unsigned long long buf;
  int n;
  __device__ __forceinline__ void fill() {
    while (n <= 56) {
      unsigned b = 0;
      if (p < e) {
        b = __ldg(p++);
        if (b == 0xFF && p < e) ++p;   // the stuffed 0x00
      }
      buf |= (unsigned long long)b << (56 - n);
      n += 8;
    }
  }
  __device__ __forceinline__ unsigned peek(int k) const { return (unsigned)(buf >> (64 - k)); }
  __device__ __forceinline__ void skip(int k) { buf <<= k; n -= k; }
  __device__ __forceinline__ int get(int k) {   // 1 <= k <= 16
    const unsigned v = peek(k);
    skip(k);
    return (int)v;
  }
};

__device__ __forceinline__ int huff_decode(BitReader& br, const HuffTab* t, bool& bad) {
  const unsigned e = __ldg(&t->look[br.peek(kHuffLook)]);
  if (e) {
    br.skip((int)(e >> 8));
    return (int)(e & 0xFF);
  }
  const int code = (int)br.peek(16);
  for (int l = kHuffLook + 1; l <= 16; ++l) {
    const int c = code >> (16 - l);
    if (c <= __ldg(&t->maxcode[l])) {
      br.skip(l);
      return __ldg(&t->values[(c + __ldg(&t->valoffset[l])) & 255]);
    }
  }
  bad = true;   // no code of <= 16 bits: jpeg_huff_decode's JWRN_HUFF_BAD_CODE, symbol 0
  br.skip(16);
  return 0;
}

__device__ __forceinline__ int huff_extend(int v, int s) { return v < (1 << (s - 1)) ? v - (1 << s) + 1 : v; }

// One segment per warp, decoded by its lane 0: the segments' codes diverge at every symbol, so lanes of one warp would
// take turns, while separate warps let the schedulers hide each decoder's load latency behind the others'.
constexpr int kHuffWarps = 4;

__global__ void __launch_bounds__(32 * kHuffWarps) jpeg_huffman_kernel(const uint8_t* __restrict__ blob, JpegLayout L,
                                                                   int n_segs, int16_t* __restrict__ coef,
                                                                   long long coef_stride, int gray,
                                                                   int* __restrict__ status) {
  __shared__ uint8_t nat[80];
  for (int i = threadIdx.x; i < 80; i += blockDim.x) nat[i] = kNatural[i];
  __syncthreads();
  const int s = blockIdx.x * kHuffWarps + (threadIdx.x >> 5);
  if ((threadIdx.x & 31) != 0 || s >= n_segs) return;
  const esf_jpeg_segment sg = reinterpret_cast<const esf_jpeg_segment*>(blob + L.segs)[s];
  const esf_jpeg_file f = reinterpret_cast<const esf_jpeg_file*>(blob)[sg.file];
  const JpegGeom g = jpeg_geom(f, gray);
  const HuffTab* tabs = reinterpret_cast<const HuffTab*>(blob + L.huff);
  const HuffTab *dc0 = tabs + f.dc[0], *dc1 = tabs + f.dc[1], *dc2 = tabs + f.dc[2];
  const HuffTab *ac0 = tabs + f.ac[0], *ac1 = tabs + f.ac[1], *ac2 = tabs + f.ac[2];
  int16_t* fcoef = coef + (long long)sg.file * coef_stride;
  const int total = g.mcux * g.mcuy;
  const int m1 = min(total, sg.first_mcu + (f.restart ? f.restart : total));
  const int hl = g.ncomp == 1 ? 1 : f.h[0], nl = g.ncomp == 1 ? 1 : f.h[0] * f.v[0];
  const int per_mcu = g.ncomp == 1 ? 1 : nl + 2;
  BitReader br{blob + L.data + sg.begin, blob + L.data + sg.end, 0ull, 0};
  int pred0 = 0, pred1 = 0, pred2 = 0;
  bool bad = false;
  for (int m = sg.first_mcu; m < m1; ++m) {
    const int my = m / g.mcux, mx = m - my * g.mcux;
    for (int b = 0; b < per_mcu; ++b) {
      const int c = b < nl ? 0 : b - nl + 1;
      const int by = c == 0 ? my * (nl / hl) + b / hl : my, bx = c == 0 ? mx * hl + b % hl : mx;
      const HuffTab* dct = c == 0 ? dc0 : (c == 1 ? dc1 : dc2);
      const HuffTab* act = c == 0 ? ac0 : (c == 1 ? ac1 : ac2);
      const bool store = c < g.nstore;
      int16_t* blk = fcoef + ((c == 0 ? g.blk0[0] : (c == 1 ? g.blk0[1] : g.blk0[2])) +
                              (long long)by * (c == 0 ? g.bw[0] : g.bw[1]) + bx) * 64;   // chroma: bw[1] == bw[2]
      br.fill();
      int t = huff_decode(br, dct, bad);
      const int diff = t ? huff_extend(br.get(t), t) : 0;
      const int pred = (c == 0 ? pred0 : (c == 1 ? pred1 : pred2)) + diff;
      pred0 = c == 0 ? pred : pred0;
      pred1 = c == 1 ? pred : pred1;
      pred2 = c == 2 ? pred : pred2;
      if (store) blk[0] = (int16_t)pred;
      for (int k = 1; k < 64; ++k) {
        br.fill();
        const int rs = huff_decode(br, act, bad);
        const int r = rs >> 4, sz = rs & 15;
        if (sz) {
          k += r;
          const int v = huff_extend(br.get(sz), sz);
          if (store) blk[nat[k]] = (int16_t)v;
        } else {
          if (r != 15) break;
          k += 15;
        }
      }
    }
  }
  if (bad) atomicOr(status + sg.file, 1);
}

// jidctint.c constants (CONST_BITS 13)
constexpr int F0298 = 2446, F0390 = 3196, F0541 = 4433, F0765 = 6270, F0899 = 7373, F1175 = 9633, F1501 = 12299,
              F1847 = 15137, F1961 = 16069, F2053 = 16819, F2562 = 20995, F3072 = 25172;

// One 8-point pass of jpeg_idct_islow on x[0..7], descaled by `shift` with rounding
template <int SHIFT>
__device__ __forceinline__ void idct8(const int (&x)[8], int (&o)[8]) {
  int z1 = (x[2] + x[6]) * F0541;
  const int tmp2 = z1 - x[6] * F1847, tmp3 = z1 + x[2] * F0765;
  const int tmp0 = (x[0] + x[4]) * 8192, tmp1 = (x[0] - x[4]) * 8192;
  const int t10 = tmp0 + tmp3, t13 = tmp0 - tmp3, t11 = tmp1 + tmp2, t12 = tmp1 - tmp2;
  int a0 = x[7], a1 = x[5], a2 = x[3], a3 = x[1];
  z1 = a0 + a3;
  int z2 = a1 + a2, z3 = a0 + a2, z4 = a1 + a3;
  const int z5 = (z3 + z4) * F1175;
  a0 *= F0298, a1 *= F2053, a2 *= F3072, a3 *= F1501;
  z1 *= -F0899, z2 *= -F2562;
  z3 = z3 * -F1961 + z5;
  z4 = z4 * -F0390 + z5;
  a0 += z1 + z3, a1 += z2 + z4, a2 += z2 + z3, a3 += z1 + z4;
  constexpr int r = 1 << (SHIFT - 1);
  o[0] = (t10 + a3 + r) >> SHIFT, o[7] = (t10 - a3 + r) >> SHIFT;
  o[1] = (t11 + a2 + r) >> SHIFT, o[6] = (t11 - a2 + r) >> SHIFT;
  o[2] = (t12 + a1 + r) >> SHIFT, o[5] = (t12 - a1 + r) >> SHIFT;
  o[3] = (t13 + a0 + r) >> SHIFT, o[4] = (t13 - a0 + r) >> SHIFT;
}

__device__ __forceinline__ unsigned idct_sample(int x) {   // range_limit[x & RANGE_MASK] of the post-IDCT table
  return (unsigned)min(max((((x + 512) & 1023) - 512) + 128, 0), 255);
}

constexpr int kIdctThreads = 128;   // 16 blocks of 8 lanes

__global__ void __launch_bounds__(kIdctThreads) jpeg_idct_kernel(const uint8_t* __restrict__ blob, JpegLayout L,
                                                                const int16_t* __restrict__ coef, long long coef_stride,
                                                                uint8_t* __restrict__ planes, long long plane_stride,
                                                                int gray) {
  __shared__ int ws[kIdctThreads / 8][64];
  const int file = blockIdx.y;
  const esf_jpeg_file f = reinterpret_cast<const esf_jpeg_file*>(blob)[file];
  const JpegGeom g = jpeg_geom(f, gray);
  const int slot = threadIdx.x >> 3, j = threadIdx.x & 7;
  const long long b = (long long)blockIdx.x * (kIdctThreads / 8) + slot;
  const bool valid = b < g.blocks;
  const int c = b < g.blk0[1] || g.nstore == 1 ? 0 : (b < g.blk0[2] || g.nstore == 2 ? 1 : 2);
  const long long local = b - (c == 0 ? g.blk0[0] : (c == 1 ? g.blk0[1] : g.blk0[2]));
  const int bw = c == 0 ? g.bw[0] : (c == 1 ? g.bw[1] : g.bw[2]);
  const int16_t* q = reinterpret_cast<const int16_t*>(blob + L.quant) + 64 * (c == 0 ? f.qt[0] : (c == 1 ? f.qt[1] : f.qt[2]));
  const int16_t* in = coef + (long long)file * coef_stride + b * 64;
  int x[8], o[8];
  if (valid) {
#pragma unroll
    for (int k = 0; k < 8; ++k) x[k] = (int)__ldg(in + 8 * k + j) * (int)__ldg(q + 8 * k + j);   // DEQUANTIZE
    idct8<13 - 2>(x, o);   // pass 1: column j
#pragma unroll
    for (int k = 0; k < 8; ++k) ws[slot][8 * k + j] = o[k];
  }
  __syncwarp();
  if (!valid) return;
#pragma unroll
  for (int k = 0; k < 8; ++k) x[k] = ws[slot][8 * j + k];
  idct8<13 + 2 + 3>(x, o);   // pass 2: row j
  const unsigned lo = idct_sample(o[0]) | idct_sample(o[1]) << 8 | idct_sample(o[2]) << 16 | idct_sample(o[3]) << 24;
  const unsigned hi = idct_sample(o[4]) | idct_sample(o[5]) << 8 | idct_sample(o[6]) << 16 | idct_sample(o[7]) << 24;
  const long long by = local / bw, bx = local - by * bw;
  uint8_t* dst = planes + (long long)file * plane_stride + (c == 0 ? g.plane0[0] : (c == 1 ? g.plane0[1] : g.plane0[2])) +
                 (by * 8 + j) * (bw * 8) + bx * 8;
  *reinterpret_cast<uint2*>(dst) = make_uint2(lo, hi);
}

// jdsample.c's upsampling of a chroma plane P (pitch, real size cw x ch) by (fx, fy) at output pixel (y, x)
__device__ __forceinline__ int upsample(const uint8_t* __restrict__ P, int pitch, int cw, int ch, int fx, int fy, int y,
                                        int x) {
  if (fx == 1 && fy == 1) return P[(long long)y * pitch + x];
  if (fx == 1) {   // h1v2: fancy whatever the width
    const int i = y >> 1, o = (y & 1) ? min(i + 1, ch - 1) : max(i - 1, 0);
    return (3 * P[(long long)i * pitch + x] + P[(long long)o * pitch + x] + 1 + (y & 1)) >> 2;
  }
  if (fx == 2 && cw > 2) {
    const int j = x >> 1, oj = (x & 1) ? min(j + 1, cw - 1) : max(j - 1, 0);
    if (fy == 1) {   // h2v1
      const uint8_t* r = P + (long long)y * pitch;
      return (3 * r[j] + r[oj] + 1 + (x & 1)) >> 2;
    }
    const int i = y >> 1, oi = (y & 1) ? min(i + 1, ch - 1) : max(i - 1, 0);   // h2v2
    const uint8_t* r0 = P + (long long)i * pitch;
    const uint8_t* r1 = P + (long long)oi * pitch;
    const int cs = 3 * r0[j] + r1[j], cso = 3 * r0[oj] + r1[oj];
    return (3 * cs + cso + 8 - (x & 1)) >> 4;
  }
  return P[(long long)(y / fy) * pitch + x / fx];   // replication: narrow h2v1 / h2v2, h4v1
}

constexpr int kColorThreads = 256;

__global__ void __launch_bounds__(kColorThreads) jpeg_color_kernel(const uint8_t* __restrict__ blob,
                                                                  const uint8_t* __restrict__ planes,
                                                                  long long plane_stride, uint8_t* __restrict__ out,
                                                                  int H, int W, int C, int gray) {
  const int file = blockIdx.y;
  const int p = blockIdx.x * kColorThreads + threadIdx.x;
  if (p >= H * W) return;
  const int y = p / W, x = p - y * W;
  const esf_jpeg_file f = reinterpret_cast<const esf_jpeg_file*>(blob)[file];
  const JpegGeom g = jpeg_geom(f, gray);
  const uint8_t* pl = planes + (long long)file * plane_stride;
  const int Y = pl[(long long)y * (g.bw[0] * 8) + x];
  uint8_t* o = out + ((long long)file * H * W + p) * C;
  if (C == 1) {
    o[0] = (uint8_t)Y;
    return;
  }
  if (g.ncomp == 1) {
    o[0] = o[1] = o[2] = (uint8_t)Y;
    return;
  }
  const int cb = upsample(pl + g.plane0[1], g.bw[1] * 8, g.cw[1], g.ch[1], g.hmax, g.vmax, y, x) - 128;
  const int cr = upsample(pl + g.plane0[2], g.bw[2] * 8, g.cw[2], g.ch[2], g.hmax, g.vmax, y, x) - 128;
  constexpr int kOneHalf = 1 << 15;
  const int r = Y + ((91881 * cr + kOneHalf) >> 16);                    // Cr_r_tab: FIX(1.40200)
  const int gg = Y + ((-22554 * cb + kOneHalf - 46802 * cr) >> 16);     // Cb_g_tab + Cr_g_tab: FIX(0.34414), FIX(0.71414)
  const int b = Y + ((116130 * cb + kOneHalf) >> 16);                   // Cb_b_tab: FIX(1.77200)
  o[0] = (uint8_t)min(max(b, 0), 255);
  o[1] = (uint8_t)min(max(gg, 0), 255);
  o[2] = (uint8_t)min(max(r, 0), 255);
}

// Checks one file descriptor; returns its geometry's coefficient and plane bytes through the pointers
static int jpeg_check_file(const esf_jpeg_file& f, int i, int gray, int n_huff, int n_quant, long long* coef_bytes,
                           long long* plane_bytes) {
  ESF_CHECK_ARG(f.H > 0 && f.W > 0 && f.H <= 65535 && f.W <= 65535, "esf_jpeg: file %d: bad size %d x %d", i, f.H, f.W);
  ESF_CHECK_ARG(f.ncomp == 1 || f.ncomp == 3, "esf_jpeg: file %d: %d components (1 or 3)", i, f.ncomp);
  ESF_CHECK_ARG(f.restart >= 0 && f.restart <= 65535, "esf_jpeg: file %d: restart interval %d", i, f.restart);
  if (f.ncomp == 3) {
    const int h = f.h[0], v = f.v[0];
    ESF_CHECK_ARG(f.h[1] == 1 && f.v[1] == 1 && f.h[2] == 1 && f.v[2] == 1 &&
                      ((h == 1 && v == 1) || (h == 2 && v == 1) || (h == 2 && v == 2) || (h == 1 && v == 2) ||
                       (h == 4 && v == 1)),
                  "esf_jpeg: file %d: sampling %dx%d/%dx%d/%dx%d", i, f.h[0], f.v[0], f.h[1], f.v[1], f.h[2], f.v[2]);
  }
  for (int c = 0; c < f.ncomp; ++c)
    ESF_CHECK_ARG(f.qt[c] >= 0 && f.qt[c] < n_quant && f.dc[c] >= 0 && f.dc[c] < n_huff && f.ac[c] >= 0 &&
                      f.ac[c] < n_huff,
                  "esf_jpeg: file %d: component %d: table index out of range", i, c);
  const JpegGeom g = jpeg_geom(f, gray);
  *coef_bytes = g.blocks * 128;
  *plane_bytes = g.plane_bytes;
  return ESF_OK;
}

// (coefficient stride, plane stride) in bytes of a call: the largest file, 256-byte aligned
static int jpeg_strides(const esf_jpeg_file* files, int n, int gray, int n_huff, int n_quant, long long* cs,
                        long long* ps) {
  *cs = *ps = 0;
  for (int i = 0; i < n; ++i) {
    long long c = 0, p = 0;
    const int rc = jpeg_check_file(files[i], i, gray, n_huff, n_quant, &c, &p);
    if (rc != ESF_OK) return rc;
    *cs = std::max(*cs, c), *ps = std::max(*ps, p);
  }
  *cs = (*cs + 255) & ~255LL, *ps = (*ps + 255) & ~255LL;
  return ESF_OK;
}

}  // namespace esf

using namespace esf;

extern "C" int esf_jpeg_scratch_bytes(const esf_jpeg_file* files_host, int32_t n_files, int32_t gray, int64_t* bytes) {
  ESF_CHECK_ARG(files_host && bytes && n_files >= 1 && n_files <= 65535, "esf_jpeg_scratch_bytes: null/bad argument");
  long long cs = 0, ps = 0;
  // table indices are checked by esf_jpeg_decode against the call's table counts
  const int rc = jpeg_strides(files_host, n_files, gray != 0, 1 << 30, 1 << 30, &cs, &ps);
  if (rc != ESF_OK) return rc;
  *bytes = (int64_t)n_files * (cs + ps);
  return ESF_OK;
}

extern "C" int esf_jpeg_decode(const void* blob, int64_t blob_bytes, const esf_jpeg_file* files_host, int32_t n_files,
                               const esf_jpeg_segment* segs_host, int32_t n_segs, int32_t n_huff, int32_t n_quant,
                               void* scratch, int64_t scratch_bytes, uint8_t* out, int32_t H, int32_t W, int32_t C,
                               int32_t gray, void* status, void* stream) {
  ESF_CHECK_ARG(blob && files_host && segs_host && scratch && out && status, "esf_jpeg_decode: null argument");
  ESF_CHECK_ARG((reinterpret_cast<uintptr_t>(blob) & 15) == 0 && (reinterpret_cast<uintptr_t>(scratch) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(status) & 3) == 0,
                "esf_jpeg_decode: misaligned blob, scratch or status");
  ESF_CHECK_ARG(n_files >= 1 && n_files <= 65535 && n_segs >= n_files && n_huff >= 1 && n_quant >= 1,
                "esf_jpeg_decode: bad counts (files %d, segments %d, tables %d / %d)", n_files, n_segs, n_huff, n_quant);
  ESF_CHECK_ARG(H > 0 && W > 0 && (long long)H * W * C < (1LL << 31) && (gray ? C == 1 : C == 3),
                "esf_jpeg_decode: bad output %d x %d x %d (gray %d)", H, W, C, gray);
  const JpegLayout L = jpeg_layout(n_files, n_segs, n_huff, n_quant);
  ESF_CHECK_ARG(blob_bytes >= L.data, "esf_jpeg_decode: blob of %lld bytes is smaller than its tables",
                (long long)blob_bytes);
  const long long data_bytes = blob_bytes - L.data;
  long long cs = 0, ps = 0;
  int rc = jpeg_strides(files_host, n_files, gray != 0, n_huff, n_quant, &cs, &ps);
  if (rc != ESF_OK) return rc;
  ESF_CHECK_ARG(scratch_bytes >= (long long)n_files * (cs + ps), "esf_jpeg_decode: scratch of %lld bytes, %lld needed",
                (long long)scratch_bytes, (long long)n_files * (cs + ps));
  for (int i = 0; i < n_files; ++i)
    ESF_CHECK_ARG(files_host[i].H == H && files_host[i].W == W, "esf_jpeg_decode: file %d is %d x %d, out is %d x %d",
                  i, files_host[i].H, files_host[i].W, H, W);
  // segments: grouped by file in file order, each file's restart intervals in order and all of them present
  int s = 0;
  for (int i = 0; i < n_files; ++i) {
    const esf_jpeg_file& f = files_host[i];
    const JpegGeom g = jpeg_geom(f, gray != 0);
    const long long total = (long long)g.mcux * g.mcuy;
    const long long nseg = f.restart ? (total + f.restart - 1) / f.restart : 1;
    for (long long k = 0; k < nseg; ++k, ++s) {
      ESF_CHECK_ARG(s < n_segs, "esf_jpeg_decode: file %d has fewer segments than its restart interval implies", i);
      const esf_jpeg_segment& sg = segs_host[s];
      ESF_CHECK_ARG(sg.file == i && sg.first_mcu == k * f.restart, "esf_jpeg_decode: segment %d: file %d, first MCU %d",
                    s, sg.file, sg.first_mcu);
      ESF_CHECK_ARG(sg.begin >= 0 && sg.begin <= sg.end && sg.end <= data_bytes,
                    "esf_jpeg_decode: segment %d: bytes [%lld, %lld) outside the %lld data bytes", s,
                    (long long)sg.begin, (long long)sg.end, data_bytes);
    }
  }
  ESF_CHECK_ARG(s == n_segs, "esf_jpeg_decode: %d segments, the files have %d", n_segs, s);

  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const uint8_t* b = static_cast<const uint8_t*>(blob);
  int16_t* coef = static_cast<int16_t*>(scratch);
  uint8_t* planes = static_cast<uint8_t*>(scratch) + (long long)n_files * cs;
  ESF_CUDA(cudaMemsetAsync(status, 0, sizeof(int32_t) * n_files, st));
  ESF_CUDA(cudaMemsetAsync(coef, 0, (size_t)n_files * cs, st));
  jpeg_huffman_kernel<<<cdiv(n_segs, kHuffWarps), 32 * kHuffWarps, 0, st>>>(b, L, n_segs, coef, cs / 2, gray != 0,
                                                                            static_cast<int*>(status));
  rc = check_launch("jpeg_huffman_kernel");
  if (rc != ESF_OK) return rc;
  const long long max_blocks = cs / 128;
  jpeg_idct_kernel<<<dim3((unsigned)((max_blocks + kIdctThreads / 8 - 1) / (kIdctThreads / 8)), (unsigned)n_files),
                     kIdctThreads, 0, st>>>(b, L, coef, cs / 2, planes, ps, gray != 0);
  rc = check_launch("jpeg_idct_kernel");
  if (rc != ESF_OK) return rc;
  jpeg_color_kernel<<<dim3((unsigned)cdiv(H * W, kColorThreads), (unsigned)n_files), kColorThreads, 0, st>>>(
      b, planes, ps, out, H, W, C, gray != 0);
  return check_launch("jpeg_color_kernel");
}
