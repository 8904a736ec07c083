// FP32-accurate path (cfg.ESF.PRECISION = "fp32"): the glue kernels around the tcgen05 implicit GEMM.
//
// The reference computes everything in FP32 (resnet_helper.py:182-240, wdf_attention_helper.py:42-53).  The tensor cores
// take 16-bit operands, so in this mode every operand is carried as a PAIR of FP16 numbers x = hi + lo (hi = fp16(x),
// lo = fp16(x - hi): 22 mantissa bits) and a product is evaluated as three FP16 MMAs with FP32 accumulation,
//     x . w  ~=  x_hi . w_hi + x_lo . w_hi + x_hi . w_lo          (the dropped lo . lo term is 2^-24 relative).
// No new GEMM kernel is needed for that: an activation is stored channels-last as THREE planes [hi | lo | hi] and the
// folded weight as [w_hi | w_hi | w_lo] along its input-channel axis, which makes the split product an ordinary
// convolution with 3x the input channels on the existing igemm kernel (FP32 output).  What remains -- and lives in
// this file -- is FP32 element-wise work: the GEMM's post-pass (per-channel scale + bias, residual, activation, split
// into planes), max/avg pooling, the ECA fuse, the head's global average, all on FP32 channels-last views.
// Weight rows are pre-scaled by a power of two (so that w_lo stays a normal FP16 number) and `scale` undoes it.
//
// These are HBM-bound helper kernels of an accuracy mode, written for clarity: one thread per 8 (or 1) channels,
// coalesced over the channel axis.
#include <math_constants.h>

#include <algorithm>

#include "esf_common.cuh"
#include "esf_host.h"

namespace esf {

struct V32 {
  char* ptr;
  int B, T, H, W, C;
  long long sB, sT, sH, sW;
};
static V32 to_v32(const esf_view* v) {
  V32 r;
  r.ptr = static_cast<char*>(v->ptr);
  r.B = v->B, r.T = v->T, r.H = v->H, r.W = v->W, r.C = v->C;
  r.sB = v->sB, r.sT = v->sT, r.sH = v->sH, r.sW = v->sW;
  return r;
}
static V32 null_v32() {
  V32 r;
  memset(&r, 0, sizeof(r));
  return r;
}
__device__ __forceinline__ long long off32(const V32& v, int b, int t, int h, int w) {
  return b * v.sB + t * v.sT + h * v.sH + w * v.sW;
}
__device__ __forceinline__ void split_hi_lo(float x, __half& hi, __half& lo) {
  hi = __float2half_rn(fminf(fmaxf(x, -65504.f), 65504.f));
  lo = __float2half_rn(x - __half2float(hi));
}

static int p32_grid(long long total, int threads) {
  long long g = (total + threads - 1) / threads;
  return (int)std::max(1LL, std::min(g, 148LL * 32));
}

// ------------------------------------------------------------------------------------------- GEMM post-pass / split
// v = act(acc * scale[c] + bias[c] + res);  y32 = v;  y3 planes = [hi(v) | lo(v) | hi(v)]
struct PostParams {
  V32 acc, acc2, acc3;     // acc2 / acc3 (optional): further partial accumulators added BEFORE the scale (split stem)
  V32 res, y32, y3;   // y3: FP16 view of the hi plane's slice; the other planes follow at +plane, +2*plane elements
  const float* scale;
  const float* bias;
  int act, plane;
  int worder;   // 0: activation planes [hi | lo | hi];  1: weight-operand planes [hi | hi | lo] (per-clip "weights")
};

// IDX: unsigned when the element count fits 32 bits (every shape of the zoo), long long otherwise -- the four 64-bit
// divisions of the index decomposition were ~500 instructions per 8 elements and bound the pass, not HBM (the same
// finding as for the 16-bit helper kernels, DESIGN.md 3.4)
template <int VEC, typename IDX>
__global__ void __launch_bounds__(256) p32_post_kernel(const PostParams p) {
  const IDX groups = (IDX)((p.acc.C + VEC - 1) / VEC);
  const IDX total = (IDX)p.acc.B * (IDX)p.acc.T * (IDX)p.acc.H * (IDX)p.acc.W * groups;
  const IDX W_ = (IDX)p.acc.W, H_ = (IDX)p.acc.H, T_ = (IDX)p.acc.T;
  for (IDX idx = (IDX)blockIdx.x * (IDX)blockDim.x + threadIdx.x; idx < total; idx += (IDX)gridDim.x * (IDX)blockDim.x) {
    const int g = (int)(idx % groups);
    IDX pos = idx / groups;
    const int w = (int)(pos % W_);
    pos /= W_;
    const int h = (int)(pos % H_);
    pos /= H_;
    const int t = (int)(pos % T_);
    const int b = (int)(pos / T_);
    const int c0 = g * VEC;
    float v[VEC];
    const float* a = reinterpret_cast<const float*>(p.acc.ptr) + off32(p.acc, b, t, h, w) + c0;
    if constexpr (VEC == 8) {
      const float4 a0 = *reinterpret_cast<const float4*>(a), a1 = *reinterpret_cast<const float4*>(a + 4);
      v[0] = a0.x, v[1] = a0.y, v[2] = a0.z, v[3] = a0.w, v[4] = a1.x, v[5] = a1.y, v[6] = a1.z, v[7] = a1.w;
    } else {
      v[0] = a[0];
    }
    for (int extra = 0; extra < 2; ++extra) {
      const V32& e = extra ? p.acc3 : p.acc2;
      if (!e.ptr) continue;
      const float* a2 = reinterpret_cast<const float*>(e.ptr) + off32(e, b, t, h, w) + c0;
      if constexpr (VEC == 8) {
        const float4 r0 = *reinterpret_cast<const float4*>(a2), r1 = *reinterpret_cast<const float4*>(a2 + 4);
        v[0] += r0.x, v[1] += r0.y, v[2] += r0.z, v[3] += r0.w, v[4] += r1.x, v[5] += r1.y, v[6] += r1.z, v[7] += r1.w;
      } else {
        v[0] += a2[0];
      }
    }
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      if (p.scale) v[j] *= __ldg(p.scale + c0 + j);
      if (p.bias) v[j] += __ldg(p.bias + c0 + j);
    }
    if (p.res.ptr) {
      const float* r = reinterpret_cast<const float*>(p.res.ptr) + off32(p.res, b, t, h, w) + c0;
      if constexpr (VEC == 8) {
        const float4 r0 = *reinterpret_cast<const float4*>(r), r1 = *reinterpret_cast<const float4*>(r + 4);
        v[0] += r0.x, v[1] += r0.y, v[2] += r0.z, v[3] += r0.w, v[4] += r1.x, v[5] += r1.y, v[6] += r1.z, v[7] += r1.w;
      } else {
        v[0] += r[0];
      }
    }
#pragma unroll
    for (int j = 0; j < VEC; ++j) v[j] = apply_act(v[j], p.act);
    if (p.y32.ptr) {
      float* y = reinterpret_cast<float*>(p.y32.ptr) + off32(p.y32, b, t, h, w) + c0;
      if constexpr (VEC == 8) {
        *reinterpret_cast<float4*>(y) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4*>(y + 4) = make_float4(v[4], v[5], v[6], v[7]);
      } else {
        y[0] = v[0];
      }
    }
    if (p.y3.ptr) {
      __half* y = reinterpret_cast<__half*>(p.y3.ptr) + off32(p.y3, b, t, h, w) + c0;
      __half hi[VEC], lo[VEC];
#pragma unroll
      for (int j = 0; j < VEC; ++j) split_hi_lo(v[j], hi[j], lo[j]);
      if constexpr (VEC == 8) {
        const uint4 H = *reinterpret_cast<const uint4*>(hi), L = *reinterpret_cast<const uint4*>(lo);
        *reinterpret_cast<uint4*>(y) = H;
        *reinterpret_cast<uint4*>(y + p.plane) = p.worder ? H : L;
        *reinterpret_cast<uint4*>(y + 2 * p.plane) = p.worder ? L : H;
      } else {
        y[0] = hi[0];
        y[p.plane] = p.worder ? hi[0] : lo[0];
        y[2 * p.plane] = p.worder ? lo[0] : hi[0];
      }
    }
  }
}

// ------------------------------------------------------------------------------------------- pooling (FP32)
struct Pool32Params {
  V32 x, y;
  int kT, kH, kW, sT, sH, sW, pT, pH, pW, is_avg;
};
// VEC = 4: one thread = four consecutive channels of one output position (16-byte loads and stores)
template <typename IDX, int VEC>
__global__ void __launch_bounds__(256) p32_pool_kernel(const Pool32Params p) {
  const IDX C_ = (IDX)(p.y.C / VEC), W_ = (IDX)p.y.W, H_ = (IDX)p.y.H, T_ = (IDX)p.y.T;
  const IDX total = (IDX)p.y.B * T_ * H_ * W_ * C_;
  for (IDX idx = (IDX)blockIdx.x * (IDX)blockDim.x + threadIdx.x; idx < total; idx += (IDX)gridDim.x * (IDX)blockDim.x) {
    const int c = (int)(idx % C_) * VEC;
    IDX pos = idx / C_;
    const int w = (int)(pos % W_);
    pos /= W_;
    const int h = (int)(pos % H_);
    pos /= H_;
    const int t = (int)(pos % T_);
    const int b = (int)(pos / T_);
    float m[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) m[j] = p.is_avg ? 0.f : -CUDART_INF_F;
    for (int kt = 0; kt < p.kT; ++kt) {
      const int ti = t * p.sT + kt - p.pT;
      if (ti < 0 || ti >= p.x.T) continue;
      for (int kh = 0; kh < p.kH; ++kh) {
        const int hi = h * p.sH + kh - p.pH;
        if (hi < 0 || hi >= p.x.H) continue;
        for (int kw = 0; kw < p.kW; ++kw) {
          const int wi = w * p.sW + kw - p.pW;
          if (wi < 0 || wi >= p.x.W) continue;
          const float* xp = reinterpret_cast<const float*>(p.x.ptr) + off32(p.x, b, ti, hi, wi) + c;
          float v[VEC];
          if constexpr (VEC == 4) {
            const float4 q = *reinterpret_cast<const float4*>(xp);
            v[0] = q.x, v[1] = q.y, v[2] = q.z, v[3] = q.w;
          } else {
            v[0] = xp[0];
          }
#pragma unroll
          for (int j = 0; j < VEC; ++j) m[j] = p.is_avg ? m[j] + v[j] : fmaxf(m[j], v[j]);
        }
      }
    }
    if (p.is_avg) {
#pragma unroll
      for (int j = 0; j < VEC; ++j) m[j] /= (float)(p.kT * p.kH * p.kW);   // count_include_pad = True, as nn.AvgPool3d
    }
    float* yp = reinterpret_cast<float*>(p.y.ptr) + off32(p.y, b, t, h, w) + c;
    if constexpr (VEC == 4) *reinterpret_cast<float4*>(yp) = make_float4(m[0], m[1], m[2], m[3]);
    else yp[0] = m[0];
  }
}

// ------------------------------------------------------------------------------------------- ECA fuse (FP32)
// pass 1: partial[b][chunk][c] = sum over the chunk's (t', h, w) of max_r x[b, alpha t' + r, h, w, c]   (deterministic)
// pass 2: y = relu(bn(maxpool_t(x) * sigmoid(conv1d_k(mean)[c])))
constexpr int kEcaChunks = 64;
struct Eca32Params {
  V32 x, y;
  int alpha, k;
  const float* w;
  const float* bn_scale;
  const float* bn_shift;
  float* partial;   // [B][kEcaChunks][C]
};
__global__ void __launch_bounds__(256) p32_eca_partial_kernel(const Eca32Params p) {
  __shared__ float red[256];
  const int C = p.x.C, b = blockIdx.y, chunk = blockIdx.x;
  const int To = p.x.T / p.alpha, W = p.x.W, H = p.x.H;
  const int npos = To * H * W;               // positions of one clip: 32-bit (checked on the host)
  const int per = (npos + kEcaChunks - 1) / kEcaChunks;
  const int p0 = chunk * per, p1 = min(npos, p0 + per);
  const int lanes = 256 / C;                 // C divides 256 (checked on the host)
  const int c = threadIdx.x % C, pl = threadIdx.x / C;
  const float* xb = reinterpret_cast<const float*>(p.x.ptr) + b * p.x.sB + c;
  float s = 0.f;
  for (int q = p0 + pl; q < p1; q += lanes) {
    const int w = q % W, r = q / W;
    const int h = r % H, t = r / H;
    const float* xp = xb + (long long)t * p.alpha * p.x.sT + h * p.x.sH + w * p.x.sW;
    float m = -CUDART_INF_F;
    for (int a = 0; a < p.alpha; ++a) m = fmaxf(m, xp[a * p.x.sT]);
    s += m;
  }
  red[threadIdx.x] = s;
  __syncthreads();
  if (pl == 0) {
    float tot = 0.f;
    for (int l = 0; l < lanes; ++l) tot += red[l * C + c];   // fixed order
    p.partial[((long long)b * kEcaChunks + chunk) * C + c] = tot;
  }
}
// grid (chunks, B): the channel gate of the block's clip is computed once per block (first version: per element, 64 x k
// loads of the partial sums each), then the block walks its share of the clip's positions with 32-bit indices
__global__ void __launch_bounds__(256) p32_eca_apply_kernel(const Eca32Params p) {
  __shared__ float mean_sh[256], gate_sh[256];
  const int C = p.x.C, b = blockIdx.y;
  const int To = p.x.T / p.alpha, W = p.x.W, H = p.x.H;
  const float inv = 1.f / ((float)To * p.x.H * p.x.W);
  if (threadIdx.x < C) {
    float mean = 0.f;
    for (int ch = 0; ch < kEcaChunks; ++ch) mean += p.partial[((long long)b * kEcaChunks + ch) * C + threadIdx.x];
    mean_sh[threadIdx.x] = mean;
  }
  __syncthreads();
  if (threadIdx.x < C) {
    const int c = threadIdx.x;
    float z = 0.f;
    for (int j = 0; j < p.k; ++j) {
      const int cc = c + j - (p.k - 1) / 2;
      if (cc < 0 || cc >= C) continue;
      z = fmaf(__ldg(p.w + j), mean_sh[cc] * inv, z);
    }
    gate_sh[c] = 1.f / (1.f + expf(-z));
  }
  __syncthreads();
  const int npos = To * H * W;
  const int per = (npos + gridDim.x - 1) / gridDim.x;
  const int p0 = blockIdx.x * per, p1 = min(npos, p0 + per);
  const int lanes = 256 / C;
  const int c = threadIdx.x % C, pl = threadIdx.x / C;
  const float gate = gate_sh[c], sc = __ldg(p.bn_scale + c), sh = __ldg(p.bn_shift + c);
  const float* xb = reinterpret_cast<const float*>(p.x.ptr) + b * p.x.sB + c;
  float* yb = reinterpret_cast<float*>(p.y.ptr) + b * p.y.sB + c;
  for (int q = p0 + pl; q < p1; q += lanes) {
    const int w = q % W, r = q / W;
    const int h = r % H, t = r / H;
    const float* xp = xb + (long long)t * p.alpha * p.x.sT + h * p.x.sH + w * p.x.sW;
    float m = -CUDART_INF_F;
    for (int a = 0; a < p.alpha; ++a) m = fmaxf(m, xp[a * p.x.sT]);
    yb[t * p.y.sT + h * p.y.sH + w * p.y.sW] = fmaxf(fmaf(m * gate, sc, sh), 0.f);
  }
}

// ------------------------------------------------------------------------------------------- head pool (FP32)
// feat[b][off + c] = mean over (t, h, w) of x[b, t, h, w, c]; one block per (clip, 256-channel group), fixed order
// block = 32 channels x 8 position lanes (first version: one thread per channel walking every position of the clip --
// 16 .. 128 blocks in all); the eight partial sums of a channel are added in a fixed order
__global__ void __launch_bounds__(256) p32_head_pool_kernel(const V32 x, float* __restrict__ feat, int feat_stride, int off) {
  __shared__ float red[256];
  const int b = blockIdx.y, cl = threadIdx.x & 31, lane = threadIdx.x >> 5, c = blockIdx.x * 32 + cl;
  const int HW = x.H * x.W, npos = x.T * HW;
  float s = 0.f;
  if (c < x.C) {
    const float* xb = reinterpret_cast<const float*>(x.ptr) + b * x.sB + c;
    for (int q = lane; q < npos; q += 8) {
      const int t = q / HW, r = q - t * HW, h = r / x.W, w = r - h * x.W;
      s += xb[t * x.sT + h * x.sH + w * x.sW];
    }
  }
  red[threadIdx.x] = s;
  __syncthreads();
  if (lane == 0 && c < x.C) {
    float tot = 0.f;
    for (int l = 0; l < 8; ++l) tot += red[l * 32 + cl];
    feat[(long long)b * feat_stride + off + c] = tot / ((float)x.T * x.H * x.W);
  }
}

// ------------------------------------------------------------------------------------------- position attention (FP32)
// out[i] = relu(bn(gamma * sum_j softmax_j(q_i . k_j) v_j + x_i)) in FP32 on the CUDA cores, flash style: the tcgen05
// kernel of the 16-bit plan rounds P and V to FP16 (2^-11), which is the whole error budget of this mode.  proj rows are
// [x_d | q | k | v] (D FP32 each).  A block owns 128 / G query rows, G = D / DT threads per row (DT = min(D, 32) channels
// of q and O per thread); key tiles of 32 rows of K and V go through shared memory, every thread computes the 32 logits
// of its row (partial dot over its channels, summed across the G lanes), one online-softmax update per tile, then
// O += P V on its channels.  The N x N matrix is never formed.  The head dim d may be below D (the smallest of 8, 16,
// 32, 64, 128 that holds it): channels [d, D) are zeros in registers and shared memory and are not stored.
template <int D>
__global__ void __launch_bounds__(128) p32_attn_kernel(const float* __restrict__ proj, int d, int N, int T, int H, int W,
                                                       float gamma, const float* __restrict__ bn_scale,
                                                       const float* __restrict__ bn_shift, int alpha,
                                                       float* __restrict__ y, long long ysB, long long ysT, long long ysH,
                                                       long long ysW) {
  constexpr int DT = D < 32 ? D : 32;
  constexpr int G = D / DT;
  constexpr int R = 128 / G;          // query rows per block
  constexpr int KT = 32;              // keys per tile
  constexpr int PITCH = D + 4 * G;    // sub-row g starts at g * (DT + 4): 16-byte aligned, G lanes hit different banks
  __shared__ __align__(16) float Ks[KT * PITCH];
  __shared__ __align__(16) float Vs[KT * PITCH];
  const int b = blockIdx.y;
  const int g = threadIdx.x % G;
  const int row = blockIdx.x * R + threadIdx.x / G;
  const bool valid = row < N;
  const float* base = proj + (long long)b * N * 4 * d;
  float q[DT], o[DT];
  {
    const float* qr = base + (long long)(valid ? row : 0) * 4 * d + d + g * DT;
#pragma unroll
    for (int c = 0; c < DT; ++c) q[c] = (valid && g * DT + c < d) ? qr[c] : 0.f, o[c] = 0.f;
  }
  float m = -CUDART_INF_F, l = 0.f;
  const float kLog2e = 1.4426950408889634f;
  for (int j0 = 0; j0 < N; j0 += KT) {
    __syncthreads();
    // cooperative tile load: KT rows x D floats of K and of V (float4 when d % 4 == 0, coalesced within a row)
    for (int i = threadIdx.x; i < KT * (D / 4); i += 128) {
      const int j = i / (D / 4), c4 = i % (D / 4);
      const int c = c4 * 4, sub = c / DT, cc = c % DT;
      float4 kv = make_float4(0.f, 0.f, 0.f, 0.f), vv = kv;
      if (j0 + j < N && c < d) {
        const float* r = base + (long long)(j0 + j) * 4 * d;
        if (d % 4 == 0) {
          kv = *reinterpret_cast<const float4*>(r + 2 * d + c);
          vv = *reinterpret_cast<const float4*>(r + 3 * d + c);
        } else {
          float kk[4], vk[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) kk[e] = c + e < d ? r[2 * d + c + e] : 0.f, vk[e] = c + e < d ? r[3 * d + c + e] : 0.f;
          kv = make_float4(kk[0], kk[1], kk[2], kk[3]);
          vv = make_float4(vk[0], vk[1], vk[2], vk[3]);
        }
      }
      *reinterpret_cast<float4*>(&Ks[j * PITCH + sub * (DT + 4) + cc]) = kv;
      *reinterpret_cast<float4*>(&Vs[j * PITCH + sub * (DT + 4) + cc]) = vv;
    }
    __syncthreads();
    float sc[KT];
#pragma unroll
    for (int j = 0; j < KT; ++j) {
      const float* kr = &Ks[j * PITCH + g * (DT + 4)];
      float a0 = 0.f, a1 = 0.f;
#pragma unroll
      for (int c = 0; c < DT; c += 4) {
        const float4 k4 = *reinterpret_cast<const float4*>(kr + c);
        a0 = fmaf(q[c], k4.x, a0);
        a1 = fmaf(q[c + 1], k4.y, a1);
        a0 = fmaf(q[c + 2], k4.z, a0);
        a1 = fmaf(q[c + 3], k4.w, a1);
      }
      float a = a0 + a1;
#pragma unroll
      for (int sh = 1; sh < G; sh <<= 1) a += __shfl_xor_sync(0xffffffffu, a, sh);   // the G lanes of a row are adjacent
      sc[j] = (j0 + j < N) ? a : -CUDART_INF_F;
    }
    float mx = sc[0];
#pragma unroll
    for (int j = 1; j < KT; ++j) mx = fmaxf(mx, sc[j]);
    const float m_new = fmaxf(m, mx);
    const float f = exp2f((m - m_new) * kLog2e);     // first tile: exp2(-inf) = 0
    m = m_new;
    l *= f;
#pragma unroll
    for (int c = 0; c < DT; ++c) o[c] *= f;
#pragma unroll
    for (int j = 0; j < KT; ++j) {
      const float pj = exp2f((sc[j] - m) * kLog2e);
      l += pj;
      const float* vr = &Vs[j * PITCH + g * (DT + 4)];
#pragma unroll
      for (int c = 0; c < DT; c += 4) {
        const float4 v4 = *reinterpret_cast<const float4*>(vr + c);
        o[c] = fmaf(pj, v4.x, o[c]);
        o[c + 1] = fmaf(pj, v4.y, o[c + 1]);
        o[c + 2] = fmaf(pj, v4.z, o[c + 2]);
        o[c + 3] = fmaf(pj, v4.w, o[c + 3]);
      }
    }
  }
  if (!valid) return;
  const float inv = 1.f / l;
  const int HW = H * W;
  const int t = row / HW, hw = row % HW, hh = hw / W, ww = hw % W;
  const float* xr = base + (long long)row * 4 * d + g * DT;
  float* yb = y + b * ysB + hh * ysH + ww * ysW + g * DT;
#pragma unroll
  for (int c = 0; c < DT; ++c) {
    const int ch = g * DT + c;
    if (ch < d) {
      const float a = fmaf(gamma, o[c] * inv, xr[c]);
      o[c] = fmaxf(fmaf(a, __ldg(bn_scale + ch), __ldg(bn_shift + ch)), 0.f);
    }
  }
  for (int r = 0; r < alpha; ++r) {
    float* yp = yb + (long long)(t * alpha + r) * ysT;
#pragma unroll
    for (int c = 0; c < DT; ++c)
      if (g * DT + c < d) yp[c] = o[c];
  }
}

// ------------------------------------------------------------------------------------------- Non-local row softmax (FP32)
// P[r][:] = softmax(scale * S[r][:]) (mode 0) or scale * S[r][:] (mode 1), written as the three planes [hi | lo | hi]
// (plane pitch `plane` elements, row pitch p_pitch) that the second product reads as its A operand.  One warp per row.
__global__ void __launch_bounds__(256) p32_row_softmax_kernel(const float* __restrict__ S, long long rows, int n,
                                                              long long s_pitch, float scale, int mode,
                                                              __half* __restrict__ P, long long p_pitch, int plane) {
  const int lane = threadIdx.x & 31;
  const long long r = blockIdx.x * 8LL + (threadIdx.x >> 5);
  if (r >= rows) return;
  const float* s = S + r * s_pitch;
  float m = -CUDART_INF_F, l = 1.f;
  if (mode == 0) {
    for (int j = lane; j < n; j += 32) m = fmaxf(m, s[j] * scale);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    l = 0.f;
    for (int j = lane; j < n; j += 32) l += expf(s[j] * scale - m);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
  }
  const float inv = 1.f / l;
  __half* p = P + r * p_pitch;
  for (int j = lane; j < n; j += 32) {
    const float v = mode == 0 ? expf(s[j] * scale - m) * inv : s[j] * scale;
    __half hi, lo;
    split_hi_lo(v, hi, lo);
    p[j] = hi, p[plane + j] = lo, p[2 * plane + j] = hi;
  }
}

static bool f32_view_ok(const esf_view* v) { return view_ok(v) && v->dtype == ESF_F32; }
static bool same_pos(const esf_view* a, const esf_view* b) {
  return a->B == b->B && a->T == b->T && a->H == b->H && a->W == b->W;
}
static bool vec8_ok(const esf_view* v, int elem) {
  const int q = 16 / elem;
  return v->C % 8 == 0 && reinterpret_cast<uintptr_t>(v->ptr) % 16 == 0 && v->sW % q == 0 && v->sH % q == 0 &&
         v->sT % q == 0 && v->sB % q == 0;
}

}  // namespace esf

using namespace esf;

extern "C" int esf_p32_post(const esf_view* acc, const float* scale, const float* bias, const esf_view* res, int32_t act,
                            const esf_view* y32, const esf_view* y3, int32_t plane, int32_t weight_order, void* stream) {
  ESF_CHECK_ARG(f32_view_ok(acc), "esf_p32_post: acc must be an FP32 view");
  ESF_CHECK_ARG(!res || !res->ptr || (f32_view_ok(res) && same_pos(res, acc) && res->C == acc->C),
                "esf_p32_post: residual must be an FP32 view of the accumulator's shape");
  ESF_CHECK_ARG(!y32 || !y32->ptr || (f32_view_ok(y32) && same_pos(y32, acc) && y32->C == acc->C),
                "esf_p32_post: y32 must be an FP32 view of the accumulator's shape");
  ESF_CHECK_ARG(!y3 || !y3->ptr || (view_ok(y3) && y3->dtype == ESF_F16 && same_pos(y3, acc) && y3->C == acc->C &&
                                    plane >= acc->C && y3->sW >= 3LL * plane),
                "esf_p32_post: y3 must be the FP16 hi-plane slice of a [hi|lo|hi] buffer (plane %d)", plane);
  PostParams p;
  p.acc = to_v32(acc);
  p.acc2 = p.acc3 = null_v32();
  p.res = (res && res->ptr) ? to_v32(res) : null_v32();
  p.y32 = (y32 && y32->ptr) ? to_v32(y32) : null_v32();
  p.y3 = (y3 && y3->ptr) ? to_v32(y3) : null_v32();
  p.scale = scale, p.bias = bias, p.act = act, p.plane = plane, p.worder = weight_order != 0;
  const long long pos = (long long)acc->B * acc->T * acc->H * acc->W;
  const bool v8 = vec8_ok(acc, 4) && (!p.res.ptr || vec8_ok(res, 4)) && (!p.y32.ptr || vec8_ok(y32, 4)) &&
                  (!p.y3.ptr || (vec8_ok(y3, 2) && plane % 8 == 0));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const bool small = pos * acc->C < 0x7fffffffLL - 148LL * 32 * 256;     // the grid-stride index stays below 2^31
  if (v8 && small) p32_post_kernel<8, unsigned><<<p32_grid(pos * (acc->C / 8), 256), 256, 0, s>>>(p);
  else if (v8) p32_post_kernel<8, long long><<<p32_grid(pos * (acc->C / 8), 256), 256, 0, s>>>(p);
  else if (small) p32_post_kernel<1, unsigned><<<p32_grid(pos * acc->C, 256), 256, 0, s>>>(p);
  else p32_post_kernel<1, long long><<<p32_grid(pos * acc->C, 256), 256, 0, s>>>(p);
  return check_launch("p32_post_kernel");
}

// esf_p32_post with three partial accumulators: v = act((acc + acc2 + acc3) * scale + bias) -- the banded stem GEMM cannot
// chain its three split products along K (5 x 7 x 3 taps exceed its tap table), so they are three launches
extern "C" int esf_p32_post3(const esf_view* acc, const esf_view* acc2, const esf_view* acc3, const float* scale,
                             const float* bias, int32_t act, const esf_view* y32, const esf_view* y3, int32_t plane,
                             void* stream) {
  ESF_CHECK_ARG(f32_view_ok(acc) && f32_view_ok(acc2) && f32_view_ok(acc3) && same_pos(acc, acc2) && same_pos(acc, acc3) &&
                    acc2->C == acc->C && acc3->C == acc->C,
                "esf_p32_post3: three FP32 accumulators of one shape expected");
  ESF_CHECK_ARG(!y32 || !y32->ptr || (f32_view_ok(y32) && same_pos(y32, acc) && y32->C == acc->C), "esf_p32_post3: bad y32");
  ESF_CHECK_ARG(!y3 || !y3->ptr || (view_ok(y3) && y3->dtype == ESF_F16 && same_pos(y3, acc) && y3->C == acc->C &&
                                    plane >= acc->C && y3->sW >= 3LL * plane),
                "esf_p32_post3: bad y3");
  PostParams p;
  p.acc = to_v32(acc), p.acc2 = to_v32(acc2), p.acc3 = to_v32(acc3);
  p.res = null_v32();
  p.y32 = (y32 && y32->ptr) ? to_v32(y32) : null_v32();
  p.y3 = (y3 && y3->ptr) ? to_v32(y3) : null_v32();
  p.scale = scale, p.bias = bias, p.act = act, p.plane = plane, p.worder = 0;
  const long long pos = (long long)acc->B * acc->T * acc->H * acc->W;
  const bool v8 = vec8_ok(acc, 4) && vec8_ok(acc2, 4) && vec8_ok(acc3, 4) && (!p.y32.ptr || vec8_ok(y32, 4)) &&
                  (!p.y3.ptr || (vec8_ok(y3, 2) && plane % 8 == 0));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const bool small = pos * acc->C < 0x7fffffffLL - 148LL * 32 * 256;     // the grid-stride index stays below 2^31
  if (v8 && small) p32_post_kernel<8, unsigned><<<p32_grid(pos * (acc->C / 8), 256), 256, 0, s>>>(p);
  else if (v8) p32_post_kernel<8, long long><<<p32_grid(pos * (acc->C / 8), 256), 256, 0, s>>>(p);
  else if (small) p32_post_kernel<1, unsigned><<<p32_grid(pos * acc->C, 256), 256, 0, s>>>(p);
  else p32_post_kernel<1, long long><<<p32_grid(pos * acc->C, 256), 256, 0, s>>>(p);
  return check_launch("p32_post_kernel");
}

extern "C" int esf_p32_pool3d(const esf_view* x, const esf_view* y, int32_t kT, int32_t kH, int32_t kW, int32_t sT,
                              int32_t sH, int32_t sW, int32_t pT, int32_t pH, int32_t pW, int32_t is_avg, void* stream) {
  ESF_CHECK_ARG(f32_view_ok(x) && f32_view_ok(y) && x->C == y->C && x->B == y->B, "esf_p32_pool3d: FP32 views expected");
  ESF_CHECK_ARG(y->T == (x->T + 2 * pT - kT) / sT + 1 && y->H == (x->H + 2 * pH - kH) / sH + 1 &&
                    y->W == (x->W + 2 * pW - kW) / sW + 1,
                "esf_p32_pool3d: output shape does not match the window");
  Pool32Params p;
  p.x = to_v32(x), p.y = to_v32(y);
  p.kT = kT, p.kH = kH, p.kW = kW, p.sT = sT, p.sH = sH, p.sW = sW, p.pT = pT, p.pH = pH, p.pW = pW, p.is_avg = is_avg;
  const long long total = (long long)y->B * y->T * y->H * y->W * y->C;
  auto al16 = [](const esf_view* v) {
    return (reinterpret_cast<uintptr_t>(v->ptr) & 15) == 0 && v->C % 4 == 0 && v->sW % 4 == 0 && v->sH % 4 == 0 &&
           v->sT % 4 == 0 && v->sB % 4 == 0;
  };
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool small = total < 0x7fffffffLL - 148LL * 32 * 256;
  if (al16(x) && al16(y)) {
    if (small) p32_pool_kernel<unsigned, 4><<<p32_grid(total / 4, 256), 256, 0, st>>>(p);
    else p32_pool_kernel<long long, 4><<<p32_grid(total / 4, 256), 256, 0, st>>>(p);
  } else {
    if (small) p32_pool_kernel<unsigned, 1><<<p32_grid(total, 256), 256, 0, st>>>(p);
    else p32_pool_kernel<long long, 1><<<p32_grid(total, 256), 256, 0, st>>>(p);
  }
  return check_launch("p32_pool_kernel");
}

extern "C" int64_t esf_p32_eca_scratch_floats(int32_t B, int32_t C) { return (int64_t)B * kEcaChunks * C; }

extern "C" int esf_p32_eca_fuse(const esf_view* x_fast, int32_t alpha, const float* eca_w, int32_t eca_k,
                                const float* bn_scale, const float* bn_shift, float* partial, const esf_view* y,
                                void* stream) {
  ESF_CHECK_ARG(f32_view_ok(x_fast) && f32_view_ok(y) && eca_w && bn_scale && bn_shift && partial,
                "esf_p32_eca_fuse: null / non-FP32 argument");
  ESF_CHECK_ARG(alpha >= 1 && x_fast->T % alpha == 0 && y->T == x_fast->T / alpha && y->H == x_fast->H &&
                    y->W == x_fast->W && y->C == x_fast->C && y->B == x_fast->B,
                "esf_p32_eca_fuse: shapes do not match");
  ESF_CHECK_ARG(x_fast->C <= 256 && 256 % x_fast->C == 0, "esf_p32_eca_fuse: C = %d must divide 256", x_fast->C);
  ESF_CHECK_ARG((long long)x_fast->T * x_fast->H * x_fast->W < 0x7fffffffLL, "esf_p32_eca_fuse: clip too large");
  Eca32Params p;
  p.x = to_v32(x_fast), p.y = to_v32(y);
  p.alpha = alpha, p.k = eca_k, p.w = eca_w, p.bn_scale = bn_scale, p.bn_shift = bn_shift, p.partial = partial;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  p32_eca_partial_kernel<<<dim3(kEcaChunks, x_fast->B), 256, 0, s>>>(p);
  int rc = check_launch("p32_eca_partial_kernel");
  if (rc) return rc;
  const long long npos = (long long)y->T * y->H * y->W;
  const int chunks = (int)std::max(1LL, std::min(npos * y->C / 4096, 592LL / std::max(1, y->B) + 1));   // ~4 blocks per SM in all
  p32_eca_apply_kernel<<<dim3(chunks, y->B), 256, 0, s>>>(p);
  return check_launch("p32_eca_apply_kernel");
}

extern "C" int esf_p32_head_pool(const esf_view* x, float* feat, int32_t feat_stride, int32_t feat_off, void* stream) {
  ESF_CHECK_ARG(f32_view_ok(x) && feat && feat_stride >= feat_off + x->C, "esf_p32_head_pool: bad argument");
  p32_head_pool_kernel<<<dim3((x->C + 31) / 32, x->B), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      to_v32(x), feat, feat_stride, feat_off);
  return check_launch("p32_head_pool_kernel");
}

extern "C" int esf_p32_attention(const float* proj, int32_t B, int32_t T, int32_t H, int32_t W, int32_t d, float gamma,
                                 const float* bn_scale, const float* bn_shift, int32_t alpha, const esf_view* y,
                                 void* stream) {
  ESF_CHECK_ARG(proj && bn_scale && bn_shift && f32_view_ok(y), "esf_p32_attention: null / non-FP32 argument");
  ESF_CHECK_ARG(y->B == B && y->T == T * alpha && y->H == H && y->W == W && y->C == d,
                "esf_p32_attention: output slice shape mismatch");
  ESF_CHECK_ARG(reinterpret_cast<uintptr_t>(proj) % 16 == 0, "esf_p32_attention: proj must be 16-byte aligned");
  const int N = T * H * W;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  float* yp = static_cast<float*>(y->ptr);
#define ESF_P32_ATTN(DD)                                                                                              \
  p32_attn_kernel<DD><<<dim3(cdiv(N, 128 / (DD / (DD < 32 ? DD : 32))), B), 128, 0, s>>>(                             \
      proj, d, N, T, H, W, gamma, bn_scale, bn_shift, alpha, yp, y->sB, y->sT, y->sH, y->sW)
  if (d <= 0 || d > 128) return set_error(ESF_ERR_UNSUPPORTED, "esf_p32_attention: head dim %d (1 ... 128)", d);
  if (d <= 8) ESF_P32_ATTN(8);
  else if (d <= 16) ESF_P32_ATTN(16);
  else if (d <= 32) ESF_P32_ATTN(32);
  else if (d <= 64) ESF_P32_ATTN(64);
  else ESF_P32_ATTN(128);
#undef ESF_P32_ATTN
  return check_launch("p32_attn_kernel");
}

extern "C" int esf_p32_row_softmax(const float* S, int64_t rows, int32_t n, int64_t s_pitch, float scale, int32_t mode,
                                   void* P3, int64_t p_pitch, int32_t plane, void* stream) {
  ESF_CHECK_ARG(S && P3 && rows > 0 && n > 0 && s_pitch >= n && plane >= n && p_pitch >= 3LL * plane,
                "esf_p32_row_softmax: bad argument");
  ESF_CHECK_ARG(rows <= 8LL * 0x7fffffff, "esf_p32_row_softmax: too many rows");
  p32_row_softmax_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      S, rows, n, s_pitch, scale, mode, static_cast<__half*>(P3), p_pitch, plane);
  return check_launch("p32_row_softmax_kernel");
}
