// Test-time spatial sampling of uint8 frames (the reference's Kinetics test branch, SlowFast/slowfast/datasets/kinetics.py
// test mode + utils.spatial_sampling): tensor_normalize -> short-side bilinear resize (transform.random_short_side_scale_jitter
// with min = max = crop size, F.interpolate(mode="bilinear", align_corners=False)) -> uniform_crop at spatial_idx 0/1/2
// -> pack_pathway_output, fused into one pass from the decoder's native frames to the stem input.
//
// Arithmetic.  The reference runs the resize on the CPU in FP32.  Its source indices and weights are tabulated per axis on
// the host (efficient_slowfast_b200/frames.py axis_table, checked against torch's own weights), so the kernel does no
// index arithmetic.  The blend is the order and FMA use of ATen's CPU kernel (UpSampleKernel.cpp, Interpolate<2, ..., 2>
// as compiled with FMA contraction):
//   t0 = fma(x00, w0, x01 * w1);  t1 = fma(x10, w0, x11 * w1);  y = fma(t0, l0, t1 * l1)
// with explicit round-to-nearest intrinsics so that nvcc contracts nothing else.  An axis whose size does not change has
// the table (i0 = d, i1 = 0, w0 = 1, w1 = 0), which makes the blend the identity, as in ATen.  When neither axis is resized
// the crop is a pure window and the kernel is a table look-up (template RESIZE = false).
//
// Work split.  One block per (clip, output frame, output row y); it loops over the V views.  Views along the long axis of a
// landscape clip share the resized row, hence the two source rows: those are read once (16-byte loads into shared memory)
// and all V crops of the row are emitted from them.  Portrait clips crop along y, so each view reloads its own rows.
//
// Mixed decode sizes (esf_*_crop_ragged).  A test split mixes resolutions and aspect ratios, but every clip's output is
// the same V x (C, T, S, S); only the source geometry differs.  Each clip brings its own source address, (H0, W0),
// resized size, axis tables and crop offsets (CropClip), and the geometry of up to kCropChunk clips travels by value in
// the kernel parameters of one launch (CropChunk, inside the classic 4 KB parameter block): a call uploads nothing,
// allocates nothing and keeps no host array past its return.  The work split is the uniform kernel's; a block reads
// its clip's entry and takes the resize or the pure-window path for that clip (a block-uniform branch).  Both kernels
// run the same row loads and emission loop (crop_rows).
//
// Temporal views of whole videos (esf_*_crop_videos).  The reference's test loader samples NUM_ENSEMBLE_VIEWS clips out of
// every decoded video (decoder.get_start_end_idx + temporal_sampling).  There a "clip" is one (video, temporal view)
// pair: its source is the whole video (Tsrc_b, H0, W0, C), shared by the video's views, and its frames are row b of a
// device frame table t_index[B][T], each entry clamped to the clip's own Tsrc_b.  The chunk (CropVideoChunk) is the
// ragged one plus the per-clip Tsrc; the kernel body is the ragged kernel's, instantiated for that chunk.
//
// AVA detection (esf_*_ava, esf_ava_boxes).  The test split of the AVA loader (datasets/ava_dataset.py
// _images_and_boxes_preprocessing, PyTorch backend) resizes the [0, 1] values (table u / 255) to short side S with no
// crop and normalises after the resize, before its BGR -> RGB swap.  The same crop_rows body writes the whole Hr x Wr
// frame as one view at (0, 0) under the AvaEmit policy; the boxes get the loader's FP64 numpy arithmetic on the device.
#include <algorithm>
#include <type_traits>

#include "esf_common.cuh"
#include "esf_host.h"

namespace esf {

constexpr int kCropThreads = 256;
constexpr int kCropMaxViews = 8;
constexpr int kCropMaxRowBytes = 16384;  // W0 * C of one source row (two rows live in shared memory)
constexpr int kCropChunk = 32;           // clips of one ragged launch (their geometry is in the parameter block)

// Source geometry of one clip.
struct CropClip {
  const uint8_t* frames;  // (Tsrc, H0, W0, C); in a uniform batch that of clip 0, clip b following at b * Tsrc * H0 * W0 * C
  const int32_t* y_idx;   // [Hr][2] source rows (i0, i1) of every resized row
  const float* y_wt;      // [Hr][2] (l0, l1)
  const int32_t* x_idx;   // [Wr][2]
  const float* x_wt;      // [Wr][2]
  int H0, W0, Hr, Wr;
  int y0[kCropMaxViews], x0[kCropMaxViews];
};

// What every clip of a call shares.
struct CropShared {
  const int32_t* t_index;
  const float* lut;       // [C][256] normalised value of byte u in OUTPUT channel c
  int Tsrc, T, C, S, V;
  int chan_src[4];
};

struct CropParams {       // B clips of one geometry
  CropShared s;
  CropClip g;
  int B;
};

struct CropChunk {        // up to kCropChunk clips of their own geometry; g[i] is output clip clip0 + i
  CropShared s;
  int clip0;
  CropClip g[kCropChunk];
};
// + the kernel's other parameters (pitch, lpad, f16, out)
static_assert(sizeof(CropChunk) + 3 * sizeof(int) + sizeof(void*) + 8 <= 4096, "CropChunk must fit the 4 KB parameters");

struct CropVideoChunk {   // up to kCropChunk (video, temporal view) clips; clip clip0 + i reads row clip0 + i of t_index
  CropShared s;
  int clip0;
  int Tsrc[kCropChunk];   // frames of clip i's video
  CropClip g[kCropChunk];
};
static_assert(sizeof(CropVideoChunk) + 3 * sizeof(int) + sizeof(void*) + 8 <= 4096,
              "CropVideoChunk must fit the 4 KB parameters");

// Frame-table row and source length of clip b of a chunk: one shared row for a ragged chunk, one row per clip of videos.
__device__ __forceinline__ int chunk_row(const CropChunk&, int) { return 0; }
__device__ __forceinline__ int chunk_tsrc(const CropChunk& p, int) { return p.s.Tsrc; }
__device__ __forceinline__ int chunk_row(const CropVideoChunk& p, int b) { return p.clip0 + b; }
__device__ __forceinline__ int chunk_tsrc(const CropVideoChunk& p, int b) { return p.Tsrc[b]; }

// copy bytes [src, src + n) into shared memory at dst + (src & 15), i.e. with the source's 16-byte phase, so that the
// aligned body moves as 16-byte loads and stores and only the ragged ends go byte by byte; returns the row's start
__device__ __forceinline__ const uint8_t* load_row_bytes(uint8_t* dst, const uint8_t* __restrict__ src, int n) {
  const int phase = (int)(reinterpret_cast<uintptr_t>(src) & 15);
  uint8_t* row = dst + phase;
  const int head = min(n, (16 - phase) & 15);
  const int body = (n - head) >> 4;
  const uint4* s4 = reinterpret_cast<const uint4*>(src + head);
  uint4* d4 = reinterpret_cast<uint4*>(row + head);
  for (int i = threadIdx.x; i < body; i += blockDim.x) d4[i] = __ldg(s4 + i);
  for (int i = threadIdx.x; i < head; i += blockDim.x) row[i] = __ldg(src + i);
  for (int i = head + 16 * body + threadIdx.x; i < n; i += blockDim.x) row[i] = __ldg(src + i);
  return row;
}

// One output value of the view at resized column xr, output channel c (source channel cs), rows r0 / r1 in shared memory.
template <bool RESIZE>
__device__ __forceinline__ float crop_value(const CropClip& g, int C, const uint8_t* r0, const uint8_t* r1,
                                            const float* lut_s, int xr, int c, int cs, float l0, float l1) {
  const float* lc = lut_s + c * 256;
  if (!RESIZE) return lc[r0[xr * C + cs]];
  const int2 xi = __ldg(reinterpret_cast<const int2*>(g.x_idx) + xr);
  const float2 xw = __ldg(reinterpret_cast<const float2*>(g.x_wt) + xr);
  const int a = min(max(xi.x, 0), g.W0 - 1) * C + cs, b = min(max(xi.y, 0), g.W0 - 1) * C + cs;
  const float t0 = __fmaf_rn(lc[r0[a]], xw.x, __fmul_rn(lc[r0[b]], xw.y));
  const float t1 = __fmaf_rn(lc[r1[a]], xw.x, __fmul_rn(lc[r1[b]], xw.y));
  return __fmaf_rn(t0, l0, __fmul_rn(t1, l1));
}

// The block's (clip, output frame, output row) and the source frame of that output frame: entry t of row `row` of the
// frame table, clamped to the clip's Tsrc frames.
__device__ __forceinline__ void crop_block(const CropShared& s, int& b, int& t, int& y) {
  y = blockIdx.x % s.S;
  t = (blockIdx.x / s.S) % s.T;
  b = blockIdx.x / (s.S * s.T);
}

__device__ __forceinline__ int source_frame(const CropShared& s, int row, int t, int Tsrc) {
  return s.t_index ? min(max(__ldg(s.t_index + row * s.T + t), 0), Tsrc - 1) : t;
}

// What a route emits: the size of its output frames and the final value of output channel c from the resized value v.
// CropEmit: the S x S crops of the classification routes, whose table already holds normalised values.
struct CropEmit {
  __device__ __forceinline__ int height(const CropShared& s, const CropClip&) const { return s.S; }
  __device__ __forceinline__ int width(const CropShared& s, const CropClip&) const { return s.S; }
  __device__ __forceinline__ float value(float v, int) const { return v; }
};

// AvaEmit: the whole resized Hr x Wr frame of the AVA test branch, which resizes the [0, 1] values (table u / 255) and
// normalises afterwards: (v - mean[c]) / std[c] with the statistics of output channel c (those of its source channel).
struct AvaEmit {
  float mean[4], std[4];
  __device__ __forceinline__ int height(const CropShared&, const CropClip& g) const { return g.Hr; }
  __device__ __forceinline__ int width(const CropShared&, const CropClip& g) const { return g.Wr; }
  __device__ __forceinline__ float value(float v, int c) const { return __fdiv_rn(__fsub_rn(v, mean[c]), std[c]); }
};

// All V crops of output row y of frame t of output clip oc, from the source frame `frame` of geometry g.  The output
// frames are Ho x Wo = e.height x e.width (S x S for the crops).
// PACKED: rows [B*V][T][Ho][pitch] of 16-bit stem input (layout of esf_stem_pack), else FP32 NCDHW (B*V, C, T, Ho, Wo)
template <bool RESIZE, bool PACKED, class Emit = CropEmit>
__device__ __forceinline__ void crop_rows(const CropShared& s, const CropClip& g, const uint8_t* frame, int oc, int t,
                                          int y, const float* lut_s, uint8_t* rows_s, int pitch, int lpad, int f16,
                                          void* __restrict__ out, const Emit& e = Emit()) {
  const int row_bytes = g.W0 * s.C;
  const int row_pitch = ((row_bytes + 15) & ~15) + 16;   // + 16: room for the source's 16-byte phase
  const uint8_t* r0 = rows_s;
  const uint8_t* r1 = rows_s + row_pitch;
  int loaded = -1;   // resized row whose source rows are in shared memory
  for (int v = 0; v < s.V; ++v) {
    const int yr = g.y0[v] + y;
    float l0 = 1.f, l1 = 0.f;
    if (yr != loaded) {
      int s0 = yr, s1 = yr;
      if (RESIZE) {
        const int2 yi = __ldg(reinterpret_cast<const int2*>(g.y_idx) + yr);
        s0 = min(max(yi.x, 0), g.H0 - 1), s1 = min(max(yi.y, 0), g.H0 - 1);
      }
      __syncthreads();   // the previous view's reads of the rows are done
      r0 = load_row_bytes(rows_s, frame + (long long)s0 * row_bytes, row_bytes);
      if (RESIZE) r1 = load_row_bytes(rows_s + row_pitch, frame + (long long)s1 * row_bytes, row_bytes);
      __syncthreads();
      loaded = yr;
    }
    if (RESIZE) {
      const float2 yw = __ldg(reinterpret_cast<const float2*>(g.y_wt) + yr);
      l0 = yw.x, l1 = yw.y;
    }
    const long long orow = ((long long)(oc * s.V + v) * s.T + t) * e.height(s, g) + y;   // (clip row, t, y) of the output
    const int x0 = g.x0[v];
    if (PACKED) {
      uint16_t* dst = static_cast<uint16_t*>(out) + orow * pitch;
      const int SC = e.width(s, g) * s.C;
      for (int ck = threadIdx.x; ck < pitch / 8; ck += blockDim.x) {
        const int j0 = ck * 8 - lpad;
        int x = j0 >= 0 ? j0 / s.C : -1 - ((-1 - j0) / s.C);   // floor division: lpad need not be a multiple of C
        int c = j0 - x * s.C;
        float f[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int j = j0 + k;
          f[k] = (j >= 0 && j < SC) ? e.value(crop_value<RESIZE>(g, s.C, r0, r1, lut_s, x0 + x, c, s.chan_src[c], l0, l1), c)
                                     : 0.f;
          if (++c == s.C) c = 0, ++x;
        }
        uint4 o;
        o.x = pack16x2(f[0], f[1], f16);
        o.y = pack16x2(f[2], f[3], f16);
        o.z = pack16x2(f[4], f[5], f16);
        o.w = pack16x2(f[6], f[7], f16);
        *reinterpret_cast<uint4*>(dst + ck * 8) = o;
      }
    } else {
      // out[(oc*V + v), c, t, y, :]: one thread = 4 consecutive x of one channel (16-byte store when Wo % 4 == 0)
      const int S4 = (e.width(s, g) + 3) / 4;
      const bool vec = (e.width(s, g) & 3) == 0;
      for (int i = threadIdx.x; i < s.C * S4; i += blockDim.x) {
        const int c = i / S4, xs = (i - c * S4) * 4;
        float f[4];
#pragma unroll
        for (int k = 0; k < 4; ++k)
          f[k] = xs + k < e.width(s, g)
                     ? e.value(crop_value<RESIZE>(g, s.C, r0, r1, lut_s, x0 + xs + k, c, s.chan_src[c], l0, l1), c)
                     : 0.f;
        float* dst = static_cast<float*>(out) + ((((long long)(oc * s.V + v) * s.C + c) * s.T + t) * e.height(s, g) + y) * e.width(s, g) + xs;
        if (vec) {
          *reinterpret_cast<float4*>(dst) = make_float4(f[0], f[1], f[2], f[3]);
        } else {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (xs + k < e.width(s, g)) dst[k] = f[k];
        }
      }
    }
  }
}

// B clips of one geometry: clip b's frames follow clip b - 1's.
template <bool RESIZE, bool PACKED>
__global__ void __launch_bounds__(kCropThreads) crop_frames_kernel(const CropParams p, int pitch, int lpad, int f16,
                                                                   void* __restrict__ out) {
  __shared__ float lut_s[4 * 256];
  extern __shared__ __align__(16) uint8_t rows_s[];
  for (int i = threadIdx.x; i < p.s.C * 256; i += blockDim.x) lut_s[i] = p.s.lut[i];
  int b, t, y;
  crop_block(p.s, b, t, y);
  const int ts = source_frame(p.s, 0, t, p.s.Tsrc);
  const uint8_t* frame = p.g.frames + ((long long)b * p.s.Tsrc + ts) * p.g.H0 * (p.g.W0 * p.s.C);
  crop_rows<RESIZE, PACKED>(p.s, p.g, frame, b, t, y, lut_s, rows_s, pitch, lpad, f16, out);
}

// A chunk of clips, each of its own geometry; resized and pure-window clips may be mixed.  Both paths live in one
// kernel, and the clip's entry is addressed by register: at the default budget of 32 registers the packed variant
// spills, at 6 blocks per SM (<= 40 registers) neither does.  Chunk: CropChunk (clips of one frame count and one frame
// index) or CropVideoChunk (temporal views of videos: a frame-table row and a source length per clip).
template <bool PACKED, class Chunk>
__global__ void __launch_bounds__(kCropThreads, 6) crop_frames_ragged_kernel(const __grid_constant__ Chunk p, int pitch,
                                                                          int lpad, int f16, void* __restrict__ out) {
  __shared__ float lut_s[4 * 256];
  extern __shared__ __align__(16) uint8_t rows_s[];
  for (int i = threadIdx.x; i < p.s.C * 256; i += blockDim.x) lut_s[i] = p.s.lut[i];
  int b, t, y;
  crop_block(p.s, b, t, y);
  const int ts = source_frame(p.s, chunk_row(p, b), t, chunk_tsrc(p, b));
  const CropClip& g = p.g[b];
  const uint8_t* frame = g.frames + (long long)ts * g.H0 * (g.W0 * p.s.C);
  if (g.Hr != g.H0 || g.Wr != g.W0)
    crop_rows<true, PACKED>(p.s, g, frame, p.clip0 + b, t, y, lut_s, rows_s, pitch, lpad, f16, out);
  else
    crop_rows<false, PACKED>(p.s, g, frame, p.clip0 + b, t, y, lut_s, rows_s, pitch, lpad, f16, out);
}

// The AVA test branch on B clips of one geometry: every output row y < Hr of the whole resized frame, one block each;
// normalisation after the resize (AvaEmit).  Frames whose short side already is the target size take the pure window.
struct AvaParams {
  CropShared s;   // V = 1, S = min(Hr, Wr)
  CropClip g;     // one view at (0, 0)
  AvaEmit e;
  int B;
};

template <bool RESIZE, bool PACKED>
__global__ void __launch_bounds__(kCropThreads) ava_frames_kernel(const __grid_constant__ AvaParams p, int pitch,
                                                                  int lpad, int f16, void* __restrict__ out) {
  __shared__ float lut_s[4 * 256];
  extern __shared__ __align__(16) uint8_t rows_s[];
  for (int i = threadIdx.x; i < p.s.C * 256; i += blockDim.x) lut_s[i] = p.s.lut[i];
  const int y = blockIdx.x % p.g.Hr;
  const int t = (blockIdx.x / p.g.Hr) % p.s.T;
  const int b = blockIdx.x / (p.g.Hr * p.s.T);
  const int ts = source_frame(p.s, 0, t, p.s.Tsrc);
  const uint8_t* frame = p.g.frames + ((long long)b * p.s.Tsrc + ts) * p.g.H0 * (p.g.W0 * p.s.C);
  crop_rows<RESIZE, PACKED, AvaEmit>(p.s, p.g, frame, b, t, y, lut_s, rows_s, pitch, lpad, f16, out, p.e);
}

// numpy's maximum(lo, x) / minimum(hi, x) of a non-NaN bound: a NaN x stays NaN, -0.0 against 0.0 gives the bound
__device__ __forceinline__ double np_max(double lo, double x) { return lo >= x ? lo : x; }
__device__ __forceinline__ double np_min(double hi, double x) { return hi <= x ? hi : x; }

// The loader's box arithmetic of the AVA test branch (FP64, as numpy runs it on the float64 boxes of ava_helper), one
// thread per box: [0, 1] coordinates times (W0, H0), clip_boxes_to_image(H0, W0), the short-side scale factor
// new / old of random_short_side_scale_jitter (none for a pure window), clip_boxes_to_image(S, S), then FP32 as the
// detection collate makes it.  Column 0 (the batch index) is passed through.
__global__ void __launch_bounds__(128) ava_boxes_kernel(const void* __restrict__ in, int f64, int K, int H0, int W0,
                                                        int Hr, int Wr, int S, float* __restrict__ out) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  const bool resize = Hr != H0 || Wr != W0;
  const double num = W0 < H0 ? (double)Hr : (double)Wr, den = W0 < H0 ? (double)H0 : (double)W0;
  for (int j = 0; j < 5; ++j) {
    double v = f64 ? __ldg(static_cast<const double*>(in) + 5LL * k + j)
                   : (double)__ldg(static_cast<const float*>(in) + 5LL * k + j);
    if (j > 0) {
      const bool x = (j & 1) != 0;   // columns 1, 3: x1, x2; 2, 4: y1, y2
      v = __dmul_rn(v, x ? (double)W0 : (double)H0);
      v = np_min((x ? W0 : H0) - 1.0, np_max(0.0, v));
      if (resize) v = __ddiv_rn(__dmul_rn(v, num), den);
      v = np_min(S - 1.0, np_max(0.0, v));
    }
    out[5LL * k + j] = __double2float_rn(v);
  }
}

static int crop_shared(CropShared* s, const char* who, int32_t B, int32_t Tsrc, int32_t C, const int32_t* t_index,
                       int32_t T, const int32_t* chan_src, const float* lut32, int32_t V, int32_t S) {
  ESF_CHECK_ARG(lut32 && B > 0 && Tsrc > 0 && T > 0 && C >= 1 && C <= 4, "%s: null/bad argument", who);
  ESF_CHECK_ARG(t_index || T == Tsrc, "%s: T (%d) != Tsrc (%d) needs a frame index", who, T, Tsrc);
  ESF_CHECK_ARG(V >= 1 && V <= kCropMaxViews && S > 0, "%s: bad views (%d) / crop size (%d)", who, V, S);
  s->t_index = t_index, s->lut = lut32;
  s->Tsrc = Tsrc, s->T = T, s->C = C, s->S = S, s->V = V;
  for (int c = 0; c < 4; ++c) {
    s->chan_src[c] = (chan_src && c < C) ? chan_src[c] : c;
    ESF_CHECK_ARG(c >= C || (s->chan_src[c] >= 0 && s->chan_src[c] < C), "%s: chan_src[%d] out of range", who, c);
  }
  return ESF_OK;
}

// Geometry of clip `clip` (-1: the one geometry of a uniform batch); needs the checked CropShared s.
static int crop_clip(CropClip* g, const char* who, int clip, const CropShared& s, const void* frames, int32_t H0,
                     int32_t W0, const void* y_index, const void* y_weight, int32_t Hr, const void* x_index,
                     const void* x_weight, int32_t Wr, const int32_t* crop_yx) {
  ESF_CHECK_ARG(frames && crop_yx && H0 > 0 && W0 > 0, "%s: clip %d: null/bad argument", who, clip);
  ESF_CHECK_ARG((long long)W0 * s.C <= kCropMaxRowBytes, "%s: clip %d: source rows of %lld bytes exceed %d", who, clip,
                (long long)W0 * s.C, kCropMaxRowBytes);
  ESF_CHECK_ARG(Hr > 0 && Wr > 0, "%s: clip %d: bad resized size %d x %d", who, clip, Hr, Wr);
  const bool resize = Hr != H0 || Wr != W0;
  ESF_CHECK_ARG(!resize || (y_index && y_weight && x_index && x_weight), "%s: clip %d: resize tables missing", who, clip);
  g->frames = static_cast<const uint8_t*>(frames);
  g->y_idx = static_cast<const int32_t*>(y_index), g->y_wt = static_cast<const float*>(y_weight);
  g->x_idx = static_cast<const int32_t*>(x_index), g->x_wt = static_cast<const float*>(x_weight);
  g->H0 = H0, g->W0 = W0, g->Hr = Hr, g->Wr = Wr;
  const int V = s.V, S = s.S;
  for (int v = 0; v < kCropMaxViews; ++v) {
    g->y0[v] = v < V ? crop_yx[2 * v] : 0;
    g->x0[v] = v < V ? crop_yx[2 * v + 1] : 0;
    ESF_CHECK_ARG(v >= V || (g->y0[v] >= 0 && g->y0[v] + S <= Hr && g->x0[v] >= 0 && g->x0[v] + S <= Wr),
                  "%s: clip %d: crop %d at (%d, %d) of size %d leaves the %d x %d frame", who, clip, v, g->y0[v],
                  g->x0[v], S, Hr, Wr);
  }
  return ESF_OK;
}

static size_t crop_smem(int W0, int C) { return 2 * (size_t)(((W0 * C + 15) & ~15) + 16); }

static int crop_params(CropParams* p, const char* who, const uint8_t* frames, int32_t B, int32_t Tsrc, int32_t H0,
                       int32_t W0, int32_t C, const int32_t* t_index, int32_t T, const int32_t* chan_src,
                       const float* lut32, const int32_t* y_index, const float* y_weight, int32_t Hr,
                       const int32_t* x_index, const float* x_weight, int32_t Wr, const int32_t* crop_yx_host,
                       int32_t V, int32_t S) {
  int rc = crop_shared(&p->s, who, B, Tsrc, C, t_index, T, chan_src, lut32, V, S);
  if (rc != ESF_OK) return rc;
  rc = crop_clip(&p->g, who, -1, p->s, frames, H0, W0, y_index, y_weight, Hr, x_index, x_weight, Wr, crop_yx_host);
  if (rc != ESF_OK) return rc;
  ESF_CHECK_ARG((long long)B * T * S < (1LL << 31), "%s: grid too large", who);
  p->B = B;
  return ESF_OK;
}

template <bool PACKED>
static int crop_launch(const char* who, const CropParams& p, int pitch, int lpad, int f16, void* out, void* stream) {
  const bool resize = p.g.Hr != p.g.H0 || p.g.Wr != p.g.W0;
  const size_t smem = crop_smem(p.g.W0, p.s.C);
  const unsigned grid = (unsigned)((long long)p.B * p.s.T * p.s.S);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (resize)
    crop_frames_kernel<true, PACKED><<<grid, kCropThreads, smem, s>>>(p, pitch, lpad, f16, out);
  else
    crop_frames_kernel<false, PACKED><<<grid, kCropThreads, smem, s>>>(p, pitch, lpad, f16, out);
  return check_launch(who);
}

// frames_host: B device addresses; geom_host [B][4]: H0, W0, Hr, Wr (CropChunk) or [B][5]: Tsrc, H0, W0, Hr, Wr
// (CropVideoChunk, whose t_index is a [B][T] table); tables_host [B][4]: device addresses of y_index, y_weight, x_index,
// x_weight; crop_yx_host [B][V][2].  Every clip is checked before the first launch.
template <bool PACKED, class Chunk>
static int crop_ragged(const char* who, const char* kernel, const void* frames_host, int32_t B, int32_t Tsrc, int32_t C,
                       const int32_t* t_index, int32_t T, const int32_t* chan_src, const float* lut32,
                       const int32_t* geom_host, const void* tables_host, const int32_t* crop_yx_host, int32_t V,
                       int32_t S, int pitch, int lpad, int f16, void* out, void* stream) {
  constexpr bool kVideos = std::is_same<Chunk, CropVideoChunk>::value;
  constexpr int kGeom = kVideos ? 5 : 4;   // int32 entries of a clip's geom_host row
  Chunk p{};
  int rc = crop_shared(&p.s, who, B, Tsrc, C, t_index, T, chan_src, lut32, V, S);
  if (rc != ESF_OK) return rc;
  ESF_CHECK_ARG(frames_host && geom_host && tables_host && crop_yx_host, "%s: null host array", who);
  ESF_CHECK_ARG((long long)kCropChunk * T * S < (1LL << 31), "%s: grid too large", who);
  ESF_CHECK_ARG((long long)B * T < (1LL << 31), "%s: frame table too large", who);
  const void* const* fr = static_cast<const void* const*>(frames_host);
  const void* const* tb = static_cast<const void* const*>(tables_host);
  auto clip = [&](CropClip* g, int b) {
    const int32_t* gm = geom_host + kGeom * b + (kVideos ? 1 : 0);
    if constexpr (kVideos) ESF_CHECK_ARG(gm[-1] >= 1, "%s: clip %d: a video of %d frames", who, b, gm[-1]);
    return crop_clip(g, who, b, p.s, fr[b], gm[0], gm[1], tb[4 * b], tb[4 * b + 1], gm[2], tb[4 * b + 2],
                     tb[4 * b + 3], gm[3], crop_yx_host + 2 * V * b);
  };
  for (int b = 0; b < B; ++b) {   // a bad clip anywhere: nothing is written
    CropClip g;
    if ((rc = clip(&g, b)) != ESF_OK) return rc;
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  for (int b0 = 0; b0 < B; b0 += kCropChunk) {
    const int n = std::min(B - b0, kCropChunk);
    p.clip0 = b0;
    int w0 = 0;
    for (int i = 0; i < n; ++i) {
      clip(&p.g[i], b0 + i);
      w0 = std::max(w0, p.g[i].W0);
      if constexpr (kVideos) p.Tsrc[i] = geom_host[kGeom * (b0 + i)];
    }
    const unsigned grid = (unsigned)(n * T * S);
    crop_frames_ragged_kernel<PACKED, Chunk><<<grid, kCropThreads, crop_smem(w0, C), s>>>(p, pitch, lpad, f16, out);
    if ((rc = check_launch(kernel)) != ESF_OK) return rc;
  }
  return ESF_OK;
}

static int check_packed_out(const char* who, int32_t dtype, int32_t pitch, int32_t lpad, int32_t S, int32_t C,
                            const void* xp) {
  ESF_CHECK_ARG(xp && is16(dtype), "%s: null output / bad dtype", who);
  ESF_CHECK_ARG(pitch % 8 == 0 && lpad >= 0 && pitch >= lpad + S * C && (reinterpret_cast<uintptr_t>(xp) & 15) == 0,
                "%s: bad pitch %d / lpad %d", who, pitch, lpad);
  return ESF_OK;
}

static int check_clip_out(const char* who, int32_t S, const float* clip) {
  ESF_CHECK_ARG(clip && ((S & 3) != 0 || (reinterpret_cast<uintptr_t>(clip) & 15) == 0), "%s: null / misaligned clip",
                who);
  return ESF_OK;
}

// The video entry points read every clip's frames through its row of the table: there is no identity default.
static int check_frame_table(const char* who, const int32_t* t_index) {
  ESF_CHECK_ARG(t_index, "%s: null frame table (t_index [B][T])", who);
  return ESF_OK;
}

// Geometry of the AVA test branch: one view of the whole Hr x Wr frame, the statistics of every output channel.
static int ava_params(AvaParams* p, const char* who, const uint8_t* frames, int32_t B, int32_t Tsrc, int32_t H0,
                      int32_t W0, int32_t C, const int32_t* t_index, int32_t T, const int32_t* chan_src,
                      const float* lut32, const float* mean_host, const float* std_host, const int32_t* y_index,
                      const float* y_weight, int32_t Hr, const int32_t* x_index, const float* x_weight, int32_t Wr) {
  static const int32_t kWhole[2] = {0, 0};
  int rc = crop_shared(&p->s, who, B, Tsrc, C, t_index, T, chan_src, lut32, 1, std::max(1, std::min(Hr, Wr)));
  if (rc != ESF_OK) return rc;
  rc = crop_clip(&p->g, who, -1, p->s, frames, H0, W0, y_index, y_weight, Hr, x_index, x_weight, Wr, kWhole);
  if (rc != ESF_OK) return rc;
  ESF_CHECK_ARG(mean_host && std_host, "%s: null mean / std", who);
  ESF_CHECK_ARG((long long)B * T * Hr < (1LL << 31), "%s: grid too large", who);
  for (int c = 0; c < 4; ++c) {   // normalised before the channel swap: output c takes its source channel's statistics
    p->e.mean[c] = c < C ? mean_host[p->s.chan_src[c]] : 0.f;
    p->e.std[c] = c < C ? std_host[p->s.chan_src[c]] : 1.f;
  }
  p->B = B;
  return ESF_OK;
}

template <bool PACKED>
static int ava_launch(const char* who, const AvaParams& p, int pitch, int lpad, int f16, void* out, void* stream) {
  const bool resize = p.g.Hr != p.g.H0 || p.g.Wr != p.g.W0;
  const size_t smem = crop_smem(p.g.W0, p.s.C);
  const unsigned grid = (unsigned)((long long)p.B * p.s.T * p.g.Hr);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (resize)
    ava_frames_kernel<true, PACKED><<<grid, kCropThreads, smem, s>>>(p, pitch, lpad, f16, out);
  else
    ava_frames_kernel<false, PACKED><<<grid, kCropThreads, smem, s>>>(p, pitch, lpad, f16, out);
  return check_launch(who);
}

// The demo's frame resize (tools/demo_net.py -> datasets/cv2_transform.scale: cv2.resize(frame, (Ws, Hs),
// interpolation=cv2.INTER_LINEAR) on uint8), OpenCV's fixed-point arithmetic in integers only.  Every axis is a host
// table (efficient_slowfast_b200/frames.py cv2_axis_table) of (source index s, weights w0 | w1 << 16), 11-bit weights;
// the x table holds OpenCV's clamped (s, f), the y table its unclamped s.  Both read s and s + 1 clamped to the frame:
//   row_k[x] = p_k[s_x] * w0_x + p_k[s_x + 1] * w1_x                                       (k = source rows s_y, s_y + 1)
//   out = (((w0_y * (row_0 >> 4)) >> 16) + ((w1_y * (row_1 >> 4)) >> 16) + 2) >> 2,  saturated   (VResizeLinear, uint8)
// One block per output row of one frame (grid.y: the frame of the chunk): the two source rows go to shared memory with
// 16-byte loads, then one thread per output byte.  A launch takes up to kResizeChunk frames of their own geometry, source
// and destination, by value in the parameter block.
constexpr int kResizeChunk = 64;

struct ResizeFrame {
  const uint8_t* src;    // (H, W, C)
  uint8_t* dst;          // (Hs, Ws, C)
  const int2* y_tab;     // [Hs]
  const int2* x_tab;     // [Ws]
  int H, W, Hs, Ws;
};

struct ResizeChunk {
  int C;
  ResizeFrame f[kResizeChunk];
};
static_assert(sizeof(ResizeChunk) <= 4096, "ResizeChunk must fit the 4 KB parameters");

__global__ void __launch_bounds__(kCropThreads) resize_u8_cv2_kernel(const __grid_constant__ ResizeChunk p) {
  extern __shared__ __align__(16) uint8_t rows_s[];
  const ResizeFrame& f = p.f[blockIdx.y];
  const int y = blockIdx.x;
  if (y >= f.Hs) return;
  const int C = p.C;
  const int row_bytes = f.W * C;
  const int row_pitch = ((row_bytes + 15) & ~15) + 16;   // + 16: room for the source's 16-byte phase
  const int2 yt = __ldg(f.y_tab + y);
  const int s0 = min(max(yt.x, 0), f.H - 1), s1 = min(max(yt.x + 1, 0), f.H - 1);
  const uint8_t* r0 = load_row_bytes(rows_s, f.src + (long long)s0 * row_bytes, row_bytes);
  const uint8_t* r1 = load_row_bytes(rows_s + row_pitch, f.src + (long long)s1 * row_bytes, row_bytes);
  __syncthreads();
  const int b0 = yt.y & 0xffff, b1 = (int)((unsigned)yt.y >> 16);
  const int n = f.Ws * C;
  uint8_t* dst = f.dst + (long long)y * n;
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    const int x = j / C, c = j - x * C;
    const int2 xt = __ldg(f.x_tab + x);
    const int a = min(max(xt.x, 0), f.W - 1) * C + c, b = min(max(xt.x + 1, 0), f.W - 1) * C + c;
    const int a0 = xt.y & 0xffff, a1 = (int)((unsigned)xt.y >> 16);
    const int v0 = r0[a] * a0 + r0[b] * a1;
    const int v1 = r1[a] * a0 + r1[b] * a1;
    const int v = (((b0 * (v0 >> 4)) >> 16) + ((b1 * (v1 >> 4)) >> 16) + 2) >> 2;
    dst[j] = (uint8_t)min(max(v, 0), 255);
  }
}

}  // namespace esf

using namespace esf;

extern "C" int esf_resize_u8_cv2(const void* frames_host, const void* dst_host, const int32_t* geom_host,
                                 const void* tables_host, int32_t B, int32_t C, void* stream) {
  ESF_CHECK_ARG(B >= 1 && frames_host && dst_host && geom_host && tables_host, "esf_resize_u8_cv2: null/bad argument");
  // C = 2: OpenCV resizes exact 2x downscales of 2-channel frames with INTER_AREA, which this kernel does not restate
  ESF_CHECK_ARG(C == 1 || C == 3 || C == 4, "esf_resize_u8_cv2: %d channels (1, 3 or 4)", C);
  const void* const* src = static_cast<const void* const*>(frames_host);
  void* const* dst = static_cast<void* const*>(const_cast<void*>(dst_host));
  const void* const* tb = static_cast<const void* const*>(tables_host);
  for (int b = 0; b < B; ++b) {   // a bad frame anywhere: nothing is written
    const int32_t* g = geom_host + 4 * b;
    ESF_CHECK_ARG(src[b] && dst[b] && tb[2 * b] && tb[2 * b + 1], "esf_resize_u8_cv2: frame %d: null address", b);
    ESF_CHECK_ARG(((reinterpret_cast<uintptr_t>(tb[2 * b]) | reinterpret_cast<uintptr_t>(tb[2 * b + 1])) & 7) == 0,
                  "esf_resize_u8_cv2: frame %d: misaligned axis table", b);
    ESF_CHECK_ARG(g[0] > 0 && g[1] > 0 && g[2] > 0 && g[3] > 0, "esf_resize_u8_cv2: frame %d: bad size %d x %d -> %d x %d",
                  b, g[0], g[1], g[2], g[3]);
    ESF_CHECK_ARG((long long)g[1] * C <= kCropMaxRowBytes, "esf_resize_u8_cv2: frame %d: source rows of %lld bytes exceed %d",
                  b, (long long)g[1] * C, kCropMaxRowBytes);
    ESF_CHECK_ARG((long long)g[2] * g[3] * C < (1LL << 31), "esf_resize_u8_cv2: frame %d: output too large", b);
  }
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  ResizeChunk p{};
  p.C = C;
  for (int b0 = 0; b0 < B; b0 += kResizeChunk) {
    const int n = std::min(B - b0, kResizeChunk);
    int hs = 0, w0 = 0;
    for (int i = 0; i < n; ++i) {
      const int32_t* g = geom_host + 4 * (b0 + i);
      ResizeFrame& f = p.f[i];
      f.src = static_cast<const uint8_t*>(src[b0 + i]);
      f.dst = static_cast<uint8_t*>(dst[b0 + i]);
      f.y_tab = static_cast<const int2*>(tb[2 * (b0 + i)]);
      f.x_tab = static_cast<const int2*>(tb[2 * (b0 + i) + 1]);
      f.H = g[0], f.W = g[1], f.Hs = g[2], f.Ws = g[3];
      hs = std::max(hs, f.Hs), w0 = std::max(w0, f.W);
    }
    resize_u8_cv2_kernel<<<dim3((unsigned)hs, (unsigned)n), kCropThreads, crop_smem(w0, C), s>>>(p);
    const int rc = check_launch("resize_u8_cv2_kernel");
    if (rc != ESF_OK) return rc;
  }
  return ESF_OK;
}

extern "C" int esf_stem_pack_u8_crop(const uint8_t* frames, int32_t B, int32_t Tsrc, int32_t H0, int32_t W0, int32_t C,
                                     const int32_t* t_index, int32_t T, const int32_t* chan_src, const float* lut32,
                                     const int32_t* y_index, const float* y_weight, int32_t Hr, const int32_t* x_index,
                                     const float* x_weight, int32_t Wr, const int32_t* crop_yx_host, int32_t V, int32_t S,
                                     int32_t dtype, int32_t pitch, int32_t lpad, void* xp, void* stream) {
  CropParams p;
  int rc = crop_params(&p, "esf_stem_pack_u8_crop", frames, B, Tsrc, H0, W0, C, t_index, T, chan_src, lut32, y_index,
                       y_weight, Hr, x_index, x_weight, Wr, crop_yx_host, V, S);
  if (rc != ESF_OK) return rc;
  if ((rc = check_packed_out("esf_stem_pack_u8_crop", dtype, pitch, lpad, S, C, xp)) != ESF_OK) return rc;
  return crop_launch<true>("crop_frames_kernel (packed)", p, pitch, lpad, dtype == ESF_F16, xp, stream);
}

extern "C" int esf_frames_to_clip_crop(const uint8_t* frames, int32_t B, int32_t Tsrc, int32_t H0, int32_t W0, int32_t C,
                                       const int32_t* t_index, int32_t T, const int32_t* chan_src, const float* lut32,
                                       const int32_t* y_index, const float* y_weight, int32_t Hr, const int32_t* x_index,
                                       const float* x_weight, int32_t Wr, const int32_t* crop_yx_host, int32_t V,
                                       int32_t S, float* clip, void* stream) {
  CropParams p;
  int rc = crop_params(&p, "esf_frames_to_clip_crop", frames, B, Tsrc, H0, W0, C, t_index, T, chan_src, lut32, y_index,
                       y_weight, Hr, x_index, x_weight, Wr, crop_yx_host, V, S);
  if (rc != ESF_OK) return rc;
  if ((rc = check_clip_out("esf_frames_to_clip_crop", S, clip)) != ESF_OK) return rc;
  return crop_launch<false>("crop_frames_kernel (clip)", p, 0, 0, 0, clip, stream);
}

extern "C" int esf_stem_pack_u8_crop_ragged(const void* frames_host, int32_t B, int32_t Tsrc, int32_t C,
                                            const int32_t* t_index, int32_t T, const int32_t* chan_src,
                                            const float* lut32, const int32_t* geom_host, const void* tables_host,
                                            const int32_t* crop_yx_host, int32_t V, int32_t S, int32_t dtype,
                                            int32_t pitch, int32_t lpad, void* xp, void* stream) {
  const int rc = check_packed_out("esf_stem_pack_u8_crop_ragged", dtype, pitch, lpad, S, C, xp);
  if (rc != ESF_OK) return rc;
  return crop_ragged<true, CropChunk>("esf_stem_pack_u8_crop_ragged", "crop_frames_ragged_kernel (packed)", frames_host, B, Tsrc,
                           C, t_index, T, chan_src, lut32, geom_host, tables_host, crop_yx_host, V, S, pitch, lpad,
                           dtype == ESF_F16, xp, stream);
}

extern "C" int esf_frames_to_clip_crop_ragged(const void* frames_host, int32_t B, int32_t Tsrc, int32_t C,
                                              const int32_t* t_index, int32_t T, const int32_t* chan_src,
                                              const float* lut32, const int32_t* geom_host, const void* tables_host,
                                              const int32_t* crop_yx_host, int32_t V, int32_t S, float* clip,
                                              void* stream) {
  const int rc = check_clip_out("esf_frames_to_clip_crop_ragged", S, clip);
  if (rc != ESF_OK) return rc;
  return crop_ragged<false, CropChunk>("esf_frames_to_clip_crop_ragged", "crop_frames_ragged_kernel (clip)", frames_host, B, Tsrc,
                            C, t_index, T, chan_src, lut32, geom_host, tables_host, crop_yx_host, V, S, 0, 0, 0, clip,
                            stream);
}

extern "C" int esf_stem_pack_u8_crop_videos(const void* frames_host, int32_t B, int32_t C, const int32_t* t_index,
                                            int32_t T, const int32_t* chan_src, const float* lut32,
                                            const int32_t* geom_host, const void* tables_host,
                                            const int32_t* crop_yx_host, int32_t V, int32_t S, int32_t dtype,
                                            int32_t pitch, int32_t lpad, void* xp, void* stream) {
  int rc = check_packed_out("esf_stem_pack_u8_crop_videos", dtype, pitch, lpad, S, C, xp);
  if (rc != ESF_OK) return rc;
  if ((rc = check_frame_table("esf_stem_pack_u8_crop_videos", t_index)) != ESF_OK) return rc;
  return crop_ragged<true, CropVideoChunk>("esf_stem_pack_u8_crop_videos", "crop_frames_ragged_kernel (videos, packed)",
                                           frames_host, B, T, C, t_index, T, chan_src, lut32, geom_host, tables_host,
                                           crop_yx_host, V, S, pitch, lpad, dtype == ESF_F16, xp, stream);
}

extern "C" int esf_frames_to_clip_crop_videos(const void* frames_host, int32_t B, int32_t C, const int32_t* t_index,
                                              int32_t T, const int32_t* chan_src, const float* lut32,
                                              const int32_t* geom_host, const void* tables_host,
                                              const int32_t* crop_yx_host, int32_t V, int32_t S, float* clip,
                                              void* stream) {
  int rc = check_clip_out("esf_frames_to_clip_crop_videos", S, clip);
  if (rc != ESF_OK) return rc;
  if ((rc = check_frame_table("esf_frames_to_clip_crop_videos", t_index)) != ESF_OK) return rc;
  return crop_ragged<false, CropVideoChunk>("esf_frames_to_clip_crop_videos", "crop_frames_ragged_kernel (videos, clip)",
                                            frames_host, B, T, C, t_index, T, chan_src, lut32, geom_host, tables_host,
                                            crop_yx_host, V, S, 0, 0, 0, clip, stream);
}

extern "C" int esf_stem_pack_u8_ava(const uint8_t* frames, int32_t B, int32_t Tsrc, int32_t H0, int32_t W0, int32_t C,
                                    const int32_t* t_index, int32_t T, const int32_t* chan_src, const float* lut32,
                                    const float* mean_host, const float* std_host, const int32_t* y_index,
                                    const float* y_weight, int32_t Hr, const int32_t* x_index, const float* x_weight,
                                    int32_t Wr, int32_t dtype, int32_t pitch, int32_t lpad, void* xp, void* stream) {
  AvaParams p;
  int rc = ava_params(&p, "esf_stem_pack_u8_ava", frames, B, Tsrc, H0, W0, C, t_index, T, chan_src, lut32, mean_host,
                      std_host, y_index, y_weight, Hr, x_index, x_weight, Wr);
  if (rc != ESF_OK) return rc;
  if ((rc = check_packed_out("esf_stem_pack_u8_ava", dtype, pitch, lpad, Wr, C, xp)) != ESF_OK) return rc;
  return ava_launch<true>("ava_frames_kernel (packed)", p, pitch, lpad, dtype == ESF_F16, xp, stream);
}

extern "C" int esf_frames_to_clip_ava(const uint8_t* frames, int32_t B, int32_t Tsrc, int32_t H0, int32_t W0, int32_t C,
                                      const int32_t* t_index, int32_t T, const int32_t* chan_src, const float* lut32,
                                      const float* mean_host, const float* std_host, const int32_t* y_index,
                                      const float* y_weight, int32_t Hr, const int32_t* x_index, const float* x_weight,
                                      int32_t Wr, float* clip, void* stream) {
  AvaParams p;
  int rc = ava_params(&p, "esf_frames_to_clip_ava", frames, B, Tsrc, H0, W0, C, t_index, T, chan_src, lut32, mean_host,
                      std_host, y_index, y_weight, Hr, x_index, x_weight, Wr);
  if (rc != ESF_OK) return rc;
  if ((rc = check_clip_out("esf_frames_to_clip_ava", Wr, clip)) != ESF_OK) return rc;
  return ava_launch<false>("ava_frames_kernel (clip)", p, 0, 0, 0, clip, stream);
}

extern "C" int esf_ava_boxes(const void* boxes, int32_t f64, int32_t K, int32_t H0, int32_t W0, int32_t Hr, int32_t Wr,
                             int32_t S, float* out, void* stream) {
  ESF_CHECK_ARG(K >= 0 && (K == 0 || (boxes && out)), "esf_ava_boxes: null/bad argument");
  ESF_CHECK_ARG(H0 > 0 && W0 > 0 && Hr > 0 && Wr > 0 && S > 0, "esf_ava_boxes: bad geometry %d x %d -> %d x %d, size %d",
                H0, W0, Hr, Wr, S);
  if (K == 0) return ESF_OK;
  ava_boxes_kernel<<<(K + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(boxes, f64 != 0, K, H0, W0, Hr, Wr,
                                                                                   S, out);
  return check_launch("ava_boxes_kernel");
}
