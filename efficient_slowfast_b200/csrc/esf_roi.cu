// RoI head of the AVA detection models (ResNetRoIHead, SlowFast/slowfast/models/head_helper.py:12-130): the temporal
// AvgPool3d of every pathway (inside the CUDA graph) and RoIAlign + spatial MaxPool2d per box (launched per call, the
// box count changes from call to call).  Channels-last throughout: a bilinear tap is one coalesced read of C floats.
#include <math_constants.h>

#include <algorithm>
#include <cmath>

#include "esf_common.cuh"
#include "esf_host.h"

namespace esf {

// Upper bound of the adaptive sampling grid per bin and axis (sampling_ratio = 0: ceil(roi_extent / R)).  A bin only
// reaches it when the box spans more than 64 * R feature cells (> 7 000 pixels at R = 7 and stride 16), i.e. far more
// than any map this model produces; beyond it the bin is sampled on a 64 x 64 grid.  The bound keeps the work of a
// block finite whatever the box values are.
constexpr int kRoiMaxGrid = 64;
constexpr int kRoiThreads = 128;

struct TmeanParams {
  const __nv_bfloat16* x;
  int B, T, H, W, C;
  long long sB, sT, sH, sW;
  int f16;
  float* y;  // (B, H, W, C) dense
};

// y[b, h, w, c] = sum_t x[b, t, h, w, c] / T, one thread per (position, 8 channels) with 16-byte loads
__global__ void __launch_bounds__(256) temporal_mean_vec_kernel(const TmeanParams p) {
  const int cg = p.C >> 3;
  const long long total = (long long)p.B * p.H * p.W * cg;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int g = (int)(i % cg);
    long long r = i / cg;
    const int w = (int)(r % p.W);
    r /= p.W;
    const int h = (int)(r % p.H);
    const int b = (int)(r / p.H);
    const __nv_bfloat16* src = p.x + b * p.sB + h * p.sH + w * p.sW + g * 8;
    float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int t = 0; t < p.T; ++t) {
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(src + t * p.sT));
      const uint32_t wd[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 f = unpack16x2(wd[e], p.f16);
        s[2 * e] += f.x, s[2 * e + 1] += f.y;
      }
    }
    const float n = (float)p.T;
    float4* dst = reinterpret_cast<float4*>(p.y + ((((long long)b * p.H + h) * p.W + w) * p.C) + g * 8);
    dst[0] = make_float4(s[0] / n, s[1] / n, s[2] / n, s[3] / n);
    dst[1] = make_float4(s[4] / n, s[5] / n, s[6] / n, s[7] / n);
  }
}

__global__ void __launch_bounds__(256) temporal_mean_kernel(const TmeanParams p) {
  const long long total = (long long)p.B * p.H * p.W * p.C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % p.C);
    long long r = i / p.C;
    const int w = (int)(r % p.W);
    r /= p.W;
    const int h = (int)(r % p.H);
    const int b = (int)(r / p.H);
    const __nv_bfloat16* src = p.x + b * p.sB + h * p.sH + w * p.sW + c;
    float s = 0.f;
    for (int t = 0; t < p.T; ++t) s += h162f(src[t * p.sT], p.f16);
    p.y[i] = s / (float)p.T;
  }
}

struct RoiParams {
  const float* map;  // (B, H, W, C) dense FP32
  int B, H, W, C;
  const float* boxes;  // (K, 5): batch index, x1, y1, x2, y2 in input pixels
  float scale;
  int R, aligned;
  float* feat;
  int feat_stride, c_off;
};

// torchvision's roi_align bilinear tap (ops/csrc/ops/cuda/roi_align_kernel.cu, bilinear_interpolate): zero outside
// [-1, H] x [-1, W], coordinates clamped to the map otherwise.  Only the channel index differs between the threads of a
// block, so the four reads of a tap are coalesced rows.
__device__ __forceinline__ float roi_tap(const float* __restrict__ m, int H, int W, int C, float y, float x) {
  if (y < -1.f || y > (float)H || x < -1.f || x > (float)W) return 0.f;
  if (y <= 0.f) y = 0.f;
  if (x <= 0.f) x = 0.f;
  int y0 = (int)y, x0 = (int)x, y1, x1;
  if (y0 >= H - 1) {
    y1 = y0 = H - 1;
    y = (float)y0;
  } else {
    y1 = y0 + 1;
  }
  if (x0 >= W - 1) {
    x1 = x0 = W - 1;
    x = (float)x0;
  } else {
    x1 = x0 + 1;
  }
  const float ly = y - y0, lx = x - x0, hy = 1.f - ly, hx = 1.f - lx;
  const float v1 = __ldg(m + ((long long)y0 * W + x0) * C), v2 = __ldg(m + ((long long)y0 * W + x1) * C);
  const float v3 = __ldg(m + ((long long)y1 * W + x0) * C), v4 = __ldg(m + ((long long)y1 * W + x1) * C);
  return hy * hx * v1 + hy * lx * v2 + ly * hx * v3 + ly * lx * v4;
}

// feat[k, c_off + c] = max over the R x R bins of the mean of the bin's grid_h x grid_w bilinear samples
// (ROIAlign(R, 1 / scale, sampling_ratio 0, aligned) followed by MaxPool2d(R, stride 1)).  Block = (box, 128
// channels); boxes run along grid.x, so any K fits.  No atomics: every output element has one writer.
__global__ void __launch_bounds__(kRoiThreads) roi_align_max_kernel(const RoiParams p) {
  const int k = blockIdx.x;
  const int c = blockIdx.y * kRoiThreads + threadIdx.x;
  if (c >= p.C) return;
  const float* bx = p.boxes + (long long)k * 5;
  const float off = p.aligned ? 0.5f : 0.f;
  const float sw = bx[1] * p.scale - off, sh = bx[2] * p.scale - off;
  const float ew = bx[3] * p.scale - off, eh = bx[4] * p.scale - off;
  float rw = ew - sw, rh = eh - sh;
  if (!p.aligned) {
    rw = fmaxf(rw, 1.f);
    rh = fmaxf(rh, 1.f);
  }
  const float bin_h = rh / (float)p.R, bin_w = rw / (float)p.R;
  float* dst = p.feat + (long long)k * p.feat_stride + p.c_off + c;
  // non-finite geometry (NaN / inf coordinates or overflow of the scaled box): the row is NaN, nothing is sampled.  The
  // end corner is tested before the legacy 1-cell clamp can hide it (fmaxf(NaN, 1) = 1).
  if (!(isfinite(bx[0]) && isfinite(sw) && isfinite(sh) && isfinite(ew) && isfinite(eh) && isfinite(bin_h) &&
        isfinite(bin_w))) {
    *dst = CUDART_NAN_F;
    return;
  }
  const int b = (int)fminf(fmaxf(bx[0], 0.f), (float)(p.B - 1));
  // grid sizes are clamped as floats before the conversion: huge boxes cannot overflow the int or the loop bound
  const int gh = (int)fminf(fmaxf(ceilf(rh / (float)p.R), 0.f), (float)kRoiMaxGrid);
  const int gw = (int)fminf(fmaxf(ceilf(rw / (float)p.R), 0.f), (float)kRoiMaxGrid);
  const float count = (float)max(gh * gw, 1);
  const float* m = p.map + (long long)b * p.H * p.W * p.C + c;
  float best = -CUDART_INF_F;
  for (int ph = 0; ph < p.R; ++ph)
    for (int pw = 0; pw < p.R; ++pw) {
      float acc = 0.f;
      for (int iy = 0; iy < gh; ++iy) {
        const float y = sh + ph * bin_h + (iy + .5f) * bin_h / (float)gh;
        for (int ix = 0; ix < gw; ++ix) {
          const float x = sw + pw * bin_w + (ix + .5f) * bin_w / (float)gw;
          acc += roi_tap(m, p.H, p.W, p.C, y, x);
        }
      }
      best = fmaxf(best, acc / count);
    }
  *dst = best;
}

}  // namespace esf

using namespace esf;

extern "C" int esf_temporal_mean(const esf_view* x, float* y, void* stream) {
  ESF_CHECK_ARG(view_ok(x) && y && is16(x->dtype), "esf_temporal_mean: null/bad argument");
  TmeanParams p;
  p.x = static_cast<const __nv_bfloat16*>(x->ptr);
  p.B = x->B, p.T = x->T, p.H = x->H, p.W = x->W, p.C = x->C;
  p.sB = x->sB, p.sT = x->sT, p.sH = x->sH, p.sW = x->sW;
  p.f16 = x->dtype == ESF_F16;
  p.y = y;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const bool vec = x->C % 8 == 0 && (reinterpret_cast<uintptr_t>(x->ptr) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0 &&
                   x->sB % 8 == 0 && x->sT % 8 == 0 && x->sH % 8 == 0 && x->sW % 8 == 0;
  const long long items = (long long)x->B * x->H * x->W * (vec ? x->C / 8 : x->C);
  const int grid = (int)std::min<long long>((items + 255) / 256, 148LL * 16);
  if (vec) {
    temporal_mean_vec_kernel<<<grid, 256, 0, s>>>(p);
    return check_launch("temporal_mean_vec_kernel");
  }
  temporal_mean_kernel<<<grid, 256, 0, s>>>(p);
  return check_launch("temporal_mean_kernel");
}

extern "C" int esf_roi_align_max(const float* map, int32_t B, int32_t H, int32_t W, int32_t C, const float* boxes,
                                 int32_t K, float spatial_scale, int32_t resolution, int32_t aligned, float* feat,
                                 int32_t feat_stride, int32_t c_off, void* stream) {
  ESF_CHECK_ARG(map && boxes && feat && B > 0 && H > 0 && W > 0 && C > 0 && K > 0 && resolution > 0 && c_off >= 0 &&
                    feat_stride >= c_off + C && C <= 65535 * kRoiThreads && std::isfinite(spatial_scale) && spatial_scale > 0.f,
                "esf_roi_align_max: null/bad argument");
  RoiParams p;
  p.map = map, p.B = B, p.H = H, p.W = W, p.C = C;
  p.boxes = boxes, p.scale = spatial_scale, p.R = resolution, p.aligned = aligned != 0;
  p.feat = feat, p.feat_stride = feat_stride, p.c_off = c_off;
  roi_align_max_kernel<<<dim3(K, cdiv(C, kRoiThreads)), kRoiThreads, 0, static_cast<cudaStream_t>(stream)>>>(p);
  return check_launch("roi_align_max_kernel");
}
