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
#include <algorithm>

#include "esf_common.cuh"
#include "esf_host.h"

namespace esf {

constexpr int kCropThreads = 256;
constexpr int kCropMaxViews = 8;
constexpr int kCropMaxRowBytes = 16384;  // W0 * C of one source row (two rows live in shared memory)

struct CropParams {
  const uint8_t* frames;  // (B, Tsrc, H0, W0, C)
  const int32_t* t_index;
  int B, Tsrc, T, H0, W0, C;
  int chan_src[4];
  const float* lut;       // [C][256] normalised value of byte u in OUTPUT channel c
  const int32_t* y_idx;   // [Hr][2] source rows (i0, i1) of every resized row
  const float* y_wt;      // [Hr][2] (l0, l1)
  const int32_t* x_idx;   // [Wr][2]
  const float* x_wt;      // [Wr][2]
  int Hr, Wr, S, V;
  int y0[kCropMaxViews], x0[kCropMaxViews];
};

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
__device__ __forceinline__ float crop_value(const CropParams& p, const uint8_t* r0, const uint8_t* r1, const float* lut_s,
                                            int xr, int c, int cs, float l0, float l1) {
  const float* lc = lut_s + c * 256;
  if (!RESIZE) return lc[r0[xr * p.C + cs]];
  const int2 xi = __ldg(reinterpret_cast<const int2*>(p.x_idx) + xr);
  const float2 xw = __ldg(reinterpret_cast<const float2*>(p.x_wt) + xr);
  const int a = min(max(xi.x, 0), p.W0 - 1) * p.C + cs, b = min(max(xi.y, 0), p.W0 - 1) * p.C + cs;
  const float t0 = __fmaf_rn(lc[r0[a]], xw.x, __fmul_rn(lc[r0[b]], xw.y));
  const float t1 = __fmaf_rn(lc[r1[a]], xw.x, __fmul_rn(lc[r1[b]], xw.y));
  return __fmaf_rn(t0, l0, __fmul_rn(t1, l1));
}

// PACKED: rows [B*V][T][S][pitch] of 16-bit stem input (layout of esf_stem_pack), else FP32 NCDHW (B*V, C, T, S, S)
template <bool RESIZE, bool PACKED>
__global__ void __launch_bounds__(kCropThreads) crop_frames_kernel(const CropParams p, int pitch, int lpad, int f16,
                                                                   void* __restrict__ out) {
  __shared__ float lut_s[4 * 256];
  extern __shared__ __align__(16) uint8_t rows_s[];
  const int row_bytes = p.W0 * p.C;
  const int row_pitch = ((row_bytes + 15) & ~15) + 16;   // + 16: room for the source's 16-byte phase
  const uint8_t* r0 = rows_s;
  const uint8_t* r1 = rows_s + row_pitch;
  for (int i = threadIdx.x; i < p.C * 256; i += blockDim.x) lut_s[i] = p.lut[i];

  const int y = blockIdx.x % p.S;
  const int t = (blockIdx.x / p.S) % p.T;
  const int b = blockIdx.x / (p.S * p.T);
  const int ts = p.t_index ? min(max(__ldg(p.t_index + t), 0), p.Tsrc - 1) : t;
  const uint8_t* frame = p.frames + ((long long)b * p.Tsrc + ts) * p.H0 * row_bytes;
  int loaded = -1;   // resized row whose source rows are in shared memory
  for (int v = 0; v < p.V; ++v) {
    const int yr = p.y0[v] + y;
    float l0 = 1.f, l1 = 0.f;
    if (yr != loaded) {
      int s0 = yr, s1 = yr;
      if (RESIZE) {
        const int2 yi = __ldg(reinterpret_cast<const int2*>(p.y_idx) + yr);
        s0 = min(max(yi.x, 0), p.H0 - 1), s1 = min(max(yi.y, 0), p.H0 - 1);
      }
      __syncthreads();   // the previous view's reads of the rows are done
      r0 = load_row_bytes(rows_s, frame + (long long)s0 * row_bytes, row_bytes);
      if (RESIZE) r1 = load_row_bytes(rows_s + row_pitch, frame + (long long)s1 * row_bytes, row_bytes);
      __syncthreads();
      loaded = yr;
    }
    if (RESIZE) {
      const float2 yw = __ldg(reinterpret_cast<const float2*>(p.y_wt) + yr);
      l0 = yw.x, l1 = yw.y;
    }
    const long long orow = ((long long)(b * p.V + v) * p.T + t) * p.S + y;   // (clip row, t, y) of the output
    const int x0 = p.x0[v];
    if (PACKED) {
      uint16_t* dst = static_cast<uint16_t*>(out) + orow * pitch;
      const int SC = p.S * p.C;
      for (int ck = threadIdx.x; ck < pitch / 8; ck += blockDim.x) {
        const int j0 = ck * 8 - lpad;
        int x = j0 >= 0 ? j0 / p.C : -1 - ((-1 - j0) / p.C);   // floor division: lpad need not be a multiple of C
        int c = j0 - x * p.C;
        float f[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int j = j0 + e;
          f[e] = (j >= 0 && j < SC) ? crop_value<RESIZE>(p, r0, r1, lut_s, x0 + x, c, p.chan_src[c], l0, l1) : 0.f;
          if (++c == p.C) c = 0, ++x;
        }
        uint4 o;
        o.x = pack16x2(f[0], f[1], f16);
        o.y = pack16x2(f[2], f[3], f16);
        o.z = pack16x2(f[4], f[5], f16);
        o.w = pack16x2(f[6], f[7], f16);
        *reinterpret_cast<uint4*>(dst + ck * 8) = o;
      }
    } else {
      // out[(b*V + v), c, t, y, :]: one thread = 4 consecutive x of one channel (16-byte store when S % 4 == 0)
      const int S4 = (p.S + 3) / 4;
      const bool vec = (p.S & 3) == 0;
      for (int i = threadIdx.x; i < p.C * S4; i += blockDim.x) {
        const int c = i / S4, xs = (i - c * S4) * 4;
        float f[4];
#pragma unroll
        for (int e = 0; e < 4; ++e)
          f[e] = xs + e < p.S ? crop_value<RESIZE>(p, r0, r1, lut_s, x0 + xs + e, c, p.chan_src[c], l0, l1) : 0.f;
        float* dst = static_cast<float*>(out) + ((((long long)(b * p.V + v) * p.C + c) * p.T + t) * p.S + y) * p.S + xs;
        if (vec) {
          *reinterpret_cast<float4*>(dst) = make_float4(f[0], f[1], f[2], f[3]);
        } else {
#pragma unroll
          for (int e = 0; e < 4; ++e)
            if (xs + e < p.S) dst[e] = f[e];
        }
      }
    }
  }
}

static int crop_params(CropParams* p, const char* who, const uint8_t* frames, int32_t B, int32_t Tsrc, int32_t H0,
                       int32_t W0, int32_t C, const int32_t* t_index, int32_t T, const int32_t* chan_src,
                       const float* lut32, const int32_t* y_index, const float* y_weight, int32_t Hr,
                       const int32_t* x_index, const float* x_weight, int32_t Wr, const int32_t* crop_yx_host,
                       int32_t V, int32_t S) {
  ESF_CHECK_ARG(frames && lut32 && crop_yx_host && B > 0 && Tsrc > 0 && T > 0 && H0 > 0 && W0 > 0 && C >= 1 && C <= 4,
                "%s: null/bad argument", who);
  ESF_CHECK_ARG(t_index || T == Tsrc, "%s: T (%d) != Tsrc (%d) needs a frame index", who, T, Tsrc);
  ESF_CHECK_ARG(W0 * C <= kCropMaxRowBytes, "%s: source rows of %d bytes exceed %d", who, W0 * C, kCropMaxRowBytes);
  ESF_CHECK_ARG(V >= 1 && V <= kCropMaxViews && S > 0 && Hr > 0 && Wr > 0, "%s: bad views (%d) / crop size (%d)", who, V, S);
  const bool resize = Hr != H0 || Wr != W0;
  ESF_CHECK_ARG(!resize || (y_index && y_weight && x_index && x_weight), "%s: resize tables missing", who);
  ESF_CHECK_ARG((long long)B * T * S < (1LL << 31), "%s: grid too large", who);
  p->frames = frames, p->t_index = t_index, p->lut = lut32;
  p->B = B, p->Tsrc = Tsrc, p->T = T, p->H0 = H0, p->W0 = W0, p->C = C;
  for (int c = 0; c < 4; ++c) {
    p->chan_src[c] = (chan_src && c < C) ? chan_src[c] : c;
    ESF_CHECK_ARG(c >= C || (p->chan_src[c] >= 0 && p->chan_src[c] < C), "%s: chan_src[%d] out of range", who, c);
  }
  p->y_idx = y_index, p->y_wt = y_weight, p->x_idx = x_index, p->x_wt = x_weight;
  p->Hr = Hr, p->Wr = Wr, p->S = S, p->V = V;
  for (int v = 0; v < kCropMaxViews; ++v) {
    p->y0[v] = v < V ? crop_yx_host[2 * v] : 0;
    p->x0[v] = v < V ? crop_yx_host[2 * v + 1] : 0;
    ESF_CHECK_ARG(v >= V || (p->y0[v] >= 0 && p->y0[v] + S <= Hr && p->x0[v] >= 0 && p->x0[v] + S <= Wr),
                  "%s: crop %d at (%d, %d) of size %d leaves the %d x %d frame", who, v, p->y0[v], p->x0[v], S, Hr, Wr);
  }
  return ESF_OK;
}

template <bool PACKED>
static int crop_launch(const char* who, const CropParams& p, int pitch, int lpad, int f16, void* out, void* stream) {
  const bool resize = p.Hr != p.H0 || p.Wr != p.W0;
  const size_t smem = 2 * (size_t)(((p.W0 * p.C + 15) & ~15) + 16);
  const unsigned grid = (unsigned)((long long)p.B * p.T * p.S);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (resize)
    crop_frames_kernel<true, PACKED><<<grid, kCropThreads, smem, s>>>(p, pitch, lpad, f16, out);
  else
    crop_frames_kernel<false, PACKED><<<grid, kCropThreads, smem, s>>>(p, pitch, lpad, f16, out);
  return check_launch(who);
}

}  // namespace esf

using namespace esf;

extern "C" int esf_stem_pack_u8_crop(const uint8_t* frames, int32_t B, int32_t Tsrc, int32_t H0, int32_t W0, int32_t C,
                                     const int32_t* t_index, int32_t T, const int32_t* chan_src, const float* lut32,
                                     const int32_t* y_index, const float* y_weight, int32_t Hr, const int32_t* x_index,
                                     const float* x_weight, int32_t Wr, const int32_t* crop_yx_host, int32_t V, int32_t S,
                                     int32_t dtype, int32_t pitch, int32_t lpad, void* xp, void* stream) {
  CropParams p;
  const int rc = crop_params(&p, "esf_stem_pack_u8_crop", frames, B, Tsrc, H0, W0, C, t_index, T, chan_src, lut32,
                             y_index, y_weight, Hr, x_index, x_weight, Wr, crop_yx_host, V, S);
  if (rc != ESF_OK) return rc;
  ESF_CHECK_ARG(xp && is16(dtype), "esf_stem_pack_u8_crop: null output / bad dtype");
  ESF_CHECK_ARG(pitch % 8 == 0 && lpad >= 0 && pitch >= lpad + S * C && (reinterpret_cast<uintptr_t>(xp) & 15) == 0,
                "esf_stem_pack_u8_crop: bad pitch %d / lpad %d", pitch, lpad);
  return crop_launch<true>("crop_frames_kernel (packed)", p, pitch, lpad, dtype == ESF_F16, xp, stream);
}

extern "C" int esf_frames_to_clip_crop(const uint8_t* frames, int32_t B, int32_t Tsrc, int32_t H0, int32_t W0, int32_t C,
                                       const int32_t* t_index, int32_t T, const int32_t* chan_src, const float* lut32,
                                       const int32_t* y_index, const float* y_weight, int32_t Hr, const int32_t* x_index,
                                       const float* x_weight, int32_t Wr, const int32_t* crop_yx_host, int32_t V,
                                       int32_t S, float* clip, void* stream) {
  CropParams p;
  const int rc = crop_params(&p, "esf_frames_to_clip_crop", frames, B, Tsrc, H0, W0, C, t_index, T, chan_src, lut32,
                             y_index, y_weight, Hr, x_index, x_weight, Wr, crop_yx_host, V, S);
  if (rc != ESF_OK) return rc;
  ESF_CHECK_ARG(clip && ((S & 3) != 0 || (reinterpret_cast<uintptr_t>(clip) & 15) == 0),
                "esf_frames_to_clip_crop: null / misaligned clip");
  return crop_launch<false>("crop_frames_kernel (clip)", p, 0, 0, 0, clip, stream);
}
