// Memory-bound CUDA-core kernels of the clip forward path: stem convolution on the raw FP32 clip, thin
// (grouped / depthwise / tiny-channel) convolutions, pooling, the ECA channel-attention fuse, and the head.
// All activations are channels-last BF16 views (include/esf.h); accumulation is FP32.
#include <math_constants.h>

#include <algorithm>
#include <cstdlib>

#include "esf_common.cuh"
#include "esf_host.h"

namespace esf {

struct View {
  char* ptr;
  int B, T, H, W, C;
  long long sB, sT, sH, sW;
  int f16;  // 16-bit storage is IEEE half (else BF16)
};
static View to_view(const esf_view* v) {
  View r;
  r.ptr = static_cast<char*>(v->ptr);
  r.B = v->B, r.T = v->T, r.H = v->H, r.W = v->W, r.C = v->C;
  r.sB = v->sB, r.sT = v->sT, r.sH = v->sH, r.sW = v->sW;
  r.f16 = v->dtype == ESF_F16;
  return r;
}
__device__ __forceinline__ long long voff(const View& v, int b, int t, int h, int w) {
  return b * v.sB + t * v.sT + h * v.sH + w * v.sW;
}
__device__ __forceinline__ float ldbf(const View& v, long long idx) {
  return h162f(reinterpret_cast<const __nv_bfloat16*>(v.ptr)[idx], v.f16);
}
__device__ __forceinline__ void sth(const View& v, long long idx, float x) {
  reinterpret_cast<__nv_bfloat16*>(v.ptr)[idx] = f2h16(x, v.f16);
}

// ------------------------------------------------------------------------------------------- stem conv
// One thread = one output position x CO_T consecutive output channels; the clip is FP32 NCDHW.
struct StemParams {
  const float* x;
  int B, Cin, T, H, W;
  const float* w;  // [kT][kH][kW][Cin][Cout]
  const float* bias;
  int Cout, kT, kH, kW, sT, sH, sW, pT, pH, pW, act;
  int To, Ho, Wo;
  View y;
  int y_f32;   // FP32 destination (the FP32-accurate path, esf_precise.cu) instead of the 16-bit storage format
};

template <int CO_T>
__global__ void __launch_bounds__(256) stem_conv_kernel(const StemParams p) {
  const int cgroups = p.Cout / CO_T;
  const long long total = (long long)p.B * p.To * p.Ho * p.Wo * cgroups;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int cg = idx % cgroups;
    long long pos = idx / cgroups;
    const int wo = pos % p.Wo;
    pos /= p.Wo;
    const int ho = pos % p.Ho;
    pos /= p.Ho;
    const int to = pos % p.To;
    const int b = pos / p.To;
    float acc[CO_T];
#pragma unroll
    for (int j = 0; j < CO_T; ++j) acc[j] = __ldg(p.bias + cg * CO_T + j);
    for (int kt = 0; kt < p.kT; ++kt) {
      const int ti = to * p.sT + kt - p.pT;
      if (ti < 0 || ti >= p.T) continue;
      for (int kh = 0; kh < p.kH; ++kh) {
        const int hi = ho * p.sH + kh - p.pH;
        if (hi < 0 || hi >= p.H) continue;
        for (int kw = 0; kw < p.kW; ++kw) {
          const int wi = wo * p.sW + kw - p.pW;
          if (wi < 0 || wi >= p.W) continue;
          for (int ci = 0; ci < p.Cin; ++ci) {
            const float xv = __ldg(p.x + ((((long long)b * p.Cin + ci) * p.T + ti) * p.H + hi) * p.W + wi);
            const float* wp = p.w + ((((long long)kt * p.kH + kh) * p.kW + kw) * p.Cin + ci) * p.Cout + cg * CO_T;
#pragma unroll
            for (int j = 0; j < CO_T; ++j) acc[j] = fmaf(xv, __ldg(wp + j), acc[j]);
          }
        }
      }
    }
    if (p.y_f32) {
      float* yf = reinterpret_cast<float*>(p.y.ptr) + voff(p.y, b, to, ho, wo) + cg * CO_T;
#pragma unroll
      for (int j = 0; j < CO_T; ++j) yf[j] = apply_act(acc[j], p.act);
      continue;
    }
    __nv_bfloat16* yp = reinterpret_cast<__nv_bfloat16*>(p.y.ptr) + voff(p.y, b, to, ho, wo) + cg * CO_T;
    if constexpr (CO_T == 8) {
      uint4 o;
      o.x = pack16x2(apply_act(acc[0], p.act), apply_act(acc[1], p.act), p.y.f16);
      o.y = pack16x2(apply_act(acc[2], p.act), apply_act(acc[3], p.act), p.y.f16);
      o.z = pack16x2(apply_act(acc[4], p.act), apply_act(acc[5], p.act), p.y.f16);
      o.w = pack16x2(apply_act(acc[6], p.act), apply_act(acc[7], p.act), p.y.f16);
      *reinterpret_cast<uint4*>(yp) = o;
    } else {
#pragma unroll
      for (int j = 0; j < CO_T; ++j) yp[j] = f2h16(apply_act(acc[j], p.act), p.y.f16);
    }
  }
}

// ------------------------------------------------------------------------------------------- stem pack
// FP32 (B,Cin,T,H,W) clip -> BF16 channels-last rows [B][T][H][pitch] with xp[.., lpad + w*Cin + c] = x[b,c,t,h,w] and
// zeros in the left/right padding (the zero padding of the stem conv along W, made explicit so that every banded
// GEMM block starts 16-byte aligned).  One thread per 8 consecutive output elements (one 16 B store).
template <int CIN>   // channel count at compile time (0: run-time Cin_rt) -- the per-element division is the hot loop
__global__ void __launch_bounds__(256) stem_pack_kernel(const float* __restrict__ x, int B, int Cin_rt, int T, int H, int W,
                                                        int pitch, int lpad, int f16, __nv_bfloat16* __restrict__ xp,
                                                        int Tsrc, const int32_t* __restrict__ t_index, int lo_part) {
  // block = 128 chunk lanes x 2 rows; one (b, t, h) row per threadIdx.y, decomposed once with 32-bit arithmetic
  const int Cin = CIN ? CIN : Cin_rt;
  const int chunks = pitch / 8;
  const long long nrows = (long long)B * T * H;
  // frame gather (esf_stem_pack_gather): output frame t reads source frame t_index[t] of a clip with Tsrc frames
  const long long plane = (long long)Tsrc * H * W;
  for (long long row = blockIdx.x * 2LL + threadIdx.y; row < nrows; row += 2LL * gridDim.x) {
    const int h = (int)(row % H);
    const int bt = (int)(row / H);
    const int t = bt % T, b = bt / T;
    const int ts = t_index ? __ldg(t_index + t) : t;
    const float* xrow = x + (long long)b * Cin * plane + ((long long)ts * H + h) * W;   // channel 0 of this row
    __nv_bfloat16* orow = xp + row * pitch;
    for (int ck = threadIdx.x; ck < chunks; ck += blockDim.x) {
      float v[8];
      const int j0 = ck * 8 - lpad;
      int w = j0 >= 0 ? j0 / Cin : -1 - ((-1 - j0) / Cin);   // floor division
      int c = j0 - w * Cin;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        v[e] = (w >= 0 && w < W) ? __ldg(xrow + c * plane + w) : 0.f;
        if (lo_part) v[e] -= h162f(f2h16(v[e], f16), f16);   // the low half of the (hi, lo) pair (FP32-accurate plan)
        if (++c == Cin) c = 0, ++w;
      }
      uint4 o;
      o.x = pack16x2(v[0], v[1], f16);
      o.y = pack16x2(v[2], v[3], f16);
      o.z = pack16x2(v[4], v[5], f16);
      o.w = pack16x2(v[6], v[7], f16);
      *reinterpret_cast<uint4*>(orow + ck * 8) = o;
    }
  }
}

// The same packing with the clip rows staged in shared memory: the kernel above issues eight scalar loads per 16-byte
// store (ncu, round 2, profiles/r2_ncu_small_kernels.md: 28 sectors per load request instead of 4, 76 % of the issue
// slots busy, 2.7 TB/s = 0.41 of the HBM peak).
// Here a block of 256 threads owns kPackRows rows: phase 1 copies their Cin x W floats with coalesced 16-byte loads,
// phase 2 builds the interleaved (w, c) 16-byte chunks out of shared memory.
constexpr int kPackRows = 4;
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
// ncu of the first two versions of this kernel (profiles/r2_ncu_small_kernels.md): 76 % of the issue slots busy and
// ~590 thread instructions per 16-byte chunk -- not the conversions but the INDEX ARITHMETIC: 64-bit row % H, row / H and
// run-time i % n, i / n per element.  Here the (b, t, h) decomposition happens once per row in shared memory
// (32-bit), loops run row-outer / lane-inner without divisions, the rows of the next group are in flight (cp.async)
// while this group is packed, and Cin = 3 uses a static pattern: element 6 u of a row is channel 0 of pixel
// 2 u - lpad / 3, so a thread turns two whole pixels into three packed words written to a staging row (stride 3 words:
// conflict-free) that leaves with coalesced 16-byte stores.
template <int CIN>
__global__ void __launch_bounds__(256) stem_pack_smem_kernel(const float* __restrict__ x, int B, int Cin_rt, int T, int H,
                                                             int W, int pitch, int lpad, int f16,
                                                             __nv_bfloat16* __restrict__ xp, int Tsrc,
                                                             const int32_t* __restrict__ t_index, int lo_part) {
  extern __shared__ __align__(16) float tile_all[];   // 2 x [kPackRows][Cin][W] FP32, then [kPackRows][pitch] 16-bit
  __shared__ long long src_off[2][kPackRows];          // element offset of channel 0 of every row of a group
  const int Cin = CIN ? CIN : Cin_rt;
  const int chunks = pitch / 8;
  const int w4 = W / 4;
  const int tile_floats = kPackRows * Cin * W;
  const int nrows = B * T * H;                          // < 2^31 (checked on the host)
  const long long plane = (long long)Tsrc * H * W;
  const int stride = gridDim.x * kPackRows;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  auto issue = [&](int buf, int row0) {
    const int nr = min(kPackRows, nrows - row0);
    if (threadIdx.x < nr) {
      const int row = row0 + threadIdx.x;
      const int h = row % H, bt = row / H, t = bt % T, b = bt / T;
      const int ts = t_index ? __ldg(t_index + t) : t;
      src_off[buf][threadIdx.x] = (long long)b * Cin * plane + ((long long)ts * H + h) * W;
    }
    __syncthreads();
    float* tile = tile_all + buf * tile_floats;
    for (int rc = warp; rc < nr * Cin; rc += 8) {        // one (row, channel) line per warp, 16 bytes per lane
      const int r = CIN ? rc / CIN : rc / Cin, c = rc - r * Cin;
      const float* src = x + src_off[buf][r] + c * plane;
      float* dst = tile + rc * W;
      for (int q = lane; q < w4; q += 32) cp_async16(dst + q * 4, src + q * 4);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  int buf = 0;
  int row0 = blockIdx.x * kPackRows;
  if (row0 < nrows) issue(0, row0);
  for (; row0 < nrows; row0 += stride, buf ^= 1) {
    const int nr = min(kPackRows, nrows - row0);
    const float* tile = tile_all + buf * tile_floats;
    if (row0 + stride < nrows) {
      issue(buf ^ 1, row0 + stride);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
    if (CIN == 3 && lpad % 3 == 0) {
      uint32_t* outw = reinterpret_cast<uint32_t*>(tile_all + 2 * tile_floats);   // [kPackRows][pitch / 2] words
      const int words = pitch / 2, U = (words + 2) / 3;
      const int w_first = -(lpad / 3);
      for (int r = 0; r < nr; ++r) {
        const float* trow = tile + r * 3 * W;
        uint32_t* orow = outw + r * words;
        for (int u = threadIdx.x; u < U; u += 256) {
          const int wa = 2 * u + w_first, wb = wa + 1;
          const bool ia = wa >= 0 && wa < W, ib = wb >= 0 && wb < W;
          float a0 = ia ? trow[wa] : 0.f, a1 = ia ? trow[W + wa] : 0.f, a2 = ia ? trow[2 * W + wa] : 0.f;
          float b0 = ib ? trow[wb] : 0.f, b1 = ib ? trow[W + wb] : 0.f, b2 = ib ? trow[2 * W + wb] : 0.f;
          if (lo_part) {
            a0 -= h162f(f2h16(a0, f16), f16), a1 -= h162f(f2h16(a1, f16), f16), a2 -= h162f(f2h16(a2, f16), f16);
            b0 -= h162f(f2h16(b0, f16), f16), b1 -= h162f(f2h16(b1, f16), f16), b2 -= h162f(f2h16(b2, f16), f16);
          }
          orow[3 * u] = pack16x2(a0, a1, f16);
          if (3 * u + 1 < words) orow[3 * u + 1] = pack16x2(a2, b0, f16);
          if (3 * u + 2 < words) orow[3 * u + 2] = pack16x2(b1, b2, f16);
        }
      }
      __syncthreads();
      for (int r = 0; r < nr; ++r) {
        const uint4* srow = reinterpret_cast<const uint4*>(outw + r * words);
        uint4* drow = reinterpret_cast<uint4*>(xp + (long long)(row0 + r) * pitch);
        for (int ck = threadIdx.x; ck < chunks; ck += 256) drow[ck] = srow[ck];
      }
    } else {
      for (int r = 0; r < nr; ++r) {
        const float* trow = tile + r * Cin * W;
        for (int ck = threadIdx.x; ck < chunks; ck += 256) {
          float v[8];
          const int j0 = ck * 8 - lpad;
          int w = j0 >= 0 ? j0 / Cin : -1 - ((-1 - j0) / Cin);   // floor division
          int c = j0 - w * Cin;
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            v[e] = (w >= 0 && w < W) ? trow[c * W + w] : 0.f;
            if (lo_part) v[e] -= h162f(f2h16(v[e], f16), f16);
            if (++c == Cin) c = 0, ++w;
          }
          uint4 o;
          o.x = pack16x2(v[0], v[1], f16);
          o.y = pack16x2(v[2], v[3], f16);
          o.z = pack16x2(v[4], v[5], f16);
          o.w = pack16x2(v[6], v[7], f16);
          *reinterpret_cast<uint4*>(xp + (long long)(row0 + r) * pitch + ck * 8) = o;
        }
      }
    }
    // the barrier at the top of the next iteration (inside issue) orders this group's reads before the refill
  }
}

// ------------------------------------------------------------------------------------------- uint8 frames
// The decoder's frames arrive as uint8 (B, Tsrc, H, W, C) -- already channels-last.  The reference normalises them on
// the host (tensor_normalize: x/255 - mean, /std, datasets/utils.py:298-315), permutes to C,T,H,W and gathers the slow
// pathway's frames by index (pack_pathway_output, datasets/utils.py:73-112), then ships FP32.  Here the byte frames
// are shipped and these kernels do all of it: lut[c][u] holds the normalised value of byte u in (output) channel c,
// built on the host with the reference's own FP32 operations, so the values are bit-identical; chan_src maps an output
// channel to its source channel (DATA.REVERSE_INPUT_CHANNEL); t_index (device, T entries, or null) is the frame gather.
struct FramesParams {
  const uint8_t* frames;
  const int32_t* t_index;
  int B, Tsrc, T, H, W, C;
  int chan_src[4];
};

// Frame addressing policies: the frame (index into `frames`, H * W * C bytes each) that output row b reads for pathway
// frame t.  ClipFrames: B clips of Tsrc frames, t_index (or the identity) picks the frame of each clip.  RingFrames: a
// bank of rings of Tsrc = L frames per camera; rows[b] = (camera, oldest slot) and t_index holds the window positions
// (oldest frame = 0), so the frame is ring slot (pos[t] + oldest) % L of that camera.  The host checks camera < N and
// pos, oldest in [0, L), hence one conditional subtraction is the modulo.
struct ClipFrames {
  __device__ __forceinline__ long long operator()(const FramesParams& p, int b, int t) const {
    const int ts = p.t_index ? __ldg(p.t_index + t) : t;
    return (long long)b * p.Tsrc + ts;
  }
};

struct RingFrames {
  const int32_t* rows;
  __device__ __forceinline__ long long operator()(const FramesParams& p, int b, int t) const {
    const int camera = __ldg(rows + 2 * b), oldest = __ldg(rows + 2 * b + 1);
    int slot = __ldg(p.t_index + t) + oldest;
    if (slot >= p.Tsrc) slot -= p.Tsrc;
    return (long long)camera * p.Tsrc + slot;
  }
};

// -> packed 16-bit stem rows [B][T][H][pitch] (see stem_pack_kernel): one thread = 8 consecutive row elements
template <class Frames>
__global__ void __launch_bounds__(256) stem_pack_u8_kernel(const FramesParams p, const uint16_t* __restrict__ lut, int pitch,
                                                           int lpad, uint16_t* __restrict__ xp, const Frames frame_of) {
  __shared__ uint16_t lut_s[4 * 256];
  for (int i = threadIdx.x; i < p.C * 256; i += blockDim.x) lut_s[i] = lut[i];
  __syncthreads();
  const int chunks = pitch / 8;
  const int WC = p.W * p.C;
  const bool direct = p.chan_src[0] == 0 && p.chan_src[1] == 1 && p.chan_src[2] == 2 && p.chan_src[3] == 3;
  const long long total = (long long)p.B * p.T * p.H * chunks;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int ck = idx % chunks;
    long long r = idx / chunks;
    const int h = r % p.H;
    r /= p.H;
    const int t = r % p.T;
    const int b = r / p.T;
    const uint8_t* row = p.frames + (frame_of(p, b, t) * p.H + h) * WC;
    const int j0 = ck * 8 - lpad;
    int c = ((j0 % p.C) + p.C) % p.C;
    uint16_t v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int j = j0 + e;
      uint16_t o = 0;
      if (j >= 0 && j < WC) {
        const int js = direct ? j : j - c + p.chan_src[c];
        o = lut_s[c * 256 + __ldg(row + js)];
      }
      v[e] = o;
      c = (c + 1 == p.C) ? 0 : c + 1;
    }
    uint4 o4;
    o4.x = v[0] | (uint32_t)v[1] << 16;
    o4.y = v[2] | (uint32_t)v[3] << 16;
    o4.z = v[4] | (uint32_t)v[5] << 16;
    o4.w = v[6] | (uint32_t)v[7] << 16;
    *reinterpret_cast<uint4*>(xp + (((long long)b * p.T + t) * p.H + h) * pitch + ck * 8) = o4;
  }
}

// -> FP32 NCDHW clip (B, C, T, H, W): the generic route for stems that do not take packed rows.  One thread = 4
// consecutive w of one (b, c, t, h) row (16-byte store).
template <class Frames>
__global__ void __launch_bounds__(256) frames_to_clip_kernel(const FramesParams p, const float* __restrict__ lut,
                                                             float* __restrict__ clip, const Frames frame_of) {
  __shared__ float lut_s[4 * 256];
  for (int i = threadIdx.x; i < p.C * 256; i += blockDim.x) lut_s[i] = lut[i];
  __syncthreads();
  const int W4 = (p.W + 3) / 4;
  const bool vec = (p.W % 4 == 0) && ((reinterpret_cast<uintptr_t>(clip) & 15) == 0);
  const long long total = (long long)p.B * p.C * p.T * p.H * W4;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int w0 = (idx % W4) * 4;
    long long r = idx / W4;
    const int h = r % p.H;
    r /= p.H;
    const int t = r % p.T;
    r /= p.T;
    const int c = r % p.C;
    const int b = r / p.C;
    const uint8_t* src = p.frames + ((frame_of(p, b, t) * p.H + h) * p.W + w0) * p.C + p.chan_src[c];
    float v[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) v[e] = (w0 + e < p.W) ? lut_s[c * 256 + __ldg(src + e * p.C)] : 0.f;
    float* dst = clip + ((((long long)b * p.C + c) * p.T + t) * p.H + h) * p.W + w0;
    if (vec) {
      *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if (w0 + e < p.W) dst[e] = v[e];
    }
  }
}

// ------------------------------------------------------------------------------------------- Nonlocal helpers
// Non-local block (SlowFast/slowfast/models/nonlocal_helper.py:105-148).  The two matrix products of a clip run as
// implicit GEMMs whose "weights" are the clip's own phi rows / transposed g rows (engine.Plan.nonlocal_block); these
// two kernels are the glue: the row normalisation of the affinity matrix and the g transpose.
// mode 0: P = softmax_j(scale * S)  (instantiation "softmax", scale = dim_inner^-0.5, nonlocal_helper.py:127-130)
// mode 1: P = scale * S             (instantiation "dot_product", scale = 1 / N_keys, nonlocal_helper.py:131-133)
// One warp per row: the row (n <= a few thousand FP32) is read three times, the second and third from L1.
__global__ void __launch_bounds__(256) row_softmax_kernel(const float* __restrict__ S, long long rows, int n, long long s_pitch,
                                                          float scale, int mode, int f16, __nv_bfloat16* __restrict__ P,
                                                          long long p_pitch) {
  const int lane = threadIdx.x & 31;
  const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long r = blockIdx.x * (long long)(blockDim.x >> 5) + (threadIdx.x >> 5); r < rows; r += warps) {
    const float* s = S + r * s_pitch;
    __nv_bfloat16* p = P + r * p_pitch;
    float m = 0.f, inv = 1.f;
    if (mode == 0) {
      m = -CUDART_INF_F;
      for (int j = lane; j < n; j += 32) m = fmaxf(m, s[j]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
      float l = 0.f;
      for (int j = lane; j < n; j += 32) l += expf((s[j] - m) * scale);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
      inv = 1.f / l;
    }
    for (int j = lane; j < n; j += 32) {
      const float v = mode == 0 ? expf((s[j] - m) * scale) * inv : s[j] * scale;
      p[j] = f2h16(v, f16);
    }
  }
}

// out[b][c][r] = in[b][r][c] for 16-bit elements; 32 x 32 tiles through shared memory
__global__ void __launch_bounds__(256) transpose16_kernel(const uint16_t* __restrict__ in, int rows, int cols,
                                                          long long in_bstride, long long in_pitch,
                                                          uint16_t* __restrict__ out, long long out_bstride,
                                                          long long out_pitch) {
  __shared__ uint16_t tile[32][33];
  const int b = blockIdx.z;
  const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
  for (int i = ty; i < 32; i += 8) {
    const int r = r0 + i, c = c0 + tx;
    tile[i][tx] = (r < rows && c < cols) ? in[b * in_bstride + r * in_pitch + c] : 0;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int c = c0 + i, r = r0 + tx;
    if (c < cols && r < rows) out[b * out_bstride + c * out_pitch + r] = tile[tx][i];
  }
}

// out[b][k] = mean_p in[b][p][k]: the `x.mean([1, 2, 3])` of fully-convolutional inference (head_helper.py:218-220)
__global__ void __launch_bounds__(256) group_mean_kernel(const float* __restrict__ in, int B, int P, int K,
                                                         float* __restrict__ out) {
  const int total = B * K;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int b = i / K, k = i - b * K;
    float acc = 0.f;
    for (int q = 0; q < P; ++q) acc += in[((long long)b * P + q) * K + k];
    out[i] = acc / (float)P;
  }
}

// ------------------------------------------------------------------------------------------- direct conv
struct DirectParams {
  View x, y, res;
  const float* w;  // [Cout][kT][kH][kW][Cin/groups]
  const float* bias;
  int kT, kH, kW, sT, sH, sW, pT, pH, pW, dT, dH, dW, groups, act, has_res, out_f32;
  int c_real;   // depthwise over padded rows (esf_dwconv_padded): channels >= c_real have zero weights / bias
  int y_pad;    // pointwise over padded output rows (esf_pointwise_padded): channels [C, y_pad) of y may be written (zeros)
};

__global__ void __launch_bounds__(256) conv_direct_kernel(const DirectParams p) {
  const int Cout = p.y.C;
  const int cin_g = p.x.C / p.groups;
  const int cout_g = Cout / p.groups;
  const long long total = (long long)p.y.B * p.y.T * p.y.H * p.y.W * Cout;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int co = idx % Cout;
    long long pos = idx / Cout;
    const int wo = pos % p.y.W;
    pos /= p.y.W;
    const int ho = pos % p.y.H;
    pos /= p.y.H;
    const int to = pos % p.y.T;
    const int b = pos / p.y.T;
    const int g = co / cout_g;
    float acc = __ldg(p.bias + co);
    const float* wbase = p.w + (long long)co * p.kT * p.kH * p.kW * cin_g;
    for (int kt = 0; kt < p.kT; ++kt) {
      const int ti = to * p.sT + kt * p.dT - p.pT;
      if (ti < 0 || ti >= p.x.T) continue;
      for (int kh = 0; kh < p.kH; ++kh) {
        const int hi = ho * p.sH + kh * p.dH - p.pH;
        if (hi < 0 || hi >= p.x.H) continue;
        for (int kw = 0; kw < p.kW; ++kw) {
          const int wi = wo * p.sW + kw * p.dW - p.pW;
          if (wi < 0 || wi >= p.x.W) continue;
          const long long xo = voff(p.x, b, ti, hi, wi) + g * cin_g;
          const float* wp = wbase + ((kt * p.kH + kh) * p.kW + kw) * cin_g;
          for (int ci = 0; ci < cin_g; ++ci) acc = fmaf(ldbf(p.x, xo + ci), __ldg(wp + ci), acc);
        }
      }
    }
    const long long yo = voff(p.y, b, to, ho, wo) + co;
    if (p.has_res) acc += ldbf(p.res, voff(p.res, b, to, ho, wo) + co);
    acc = apply_act(acc, p.act);
    if (p.out_f32) reinterpret_cast<float*>(p.y.ptr)[yo] = acc;
    else sth(p.y, yo, acc);
  }
}

// Depthwise k x k x 3 convolution (groups == C), the HBM-bound half of the efficient backbones.  One thread = VEC
// channels x OW consecutive output columns of one (b, t, h) row: every input column it loads is reused by up to three
// kw taps and OW outputs, loads are VEC * 2 bytes wide (16 B when C % 8 == 0), and consecutive threads walk the channel
// groups, i.e. contiguous memory.  A block owns a fixed range of <= 32 channel groups whose weights and bias are staged
// in shared memory transposed to [tap][channel].
template <int VEC>
__device__ __forceinline__ void load_vec(const __nv_bfloat16* ptr, int f16, float* v) {
  if constexpr (VEC == 8) {
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(ptr));
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = unpack16x2(w[e], f16);
      v[2 * e] = f.x, v[2 * e + 1] = f.y;
    }
  } else if constexpr (VEC == 4) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(ptr));
    const float2 a = unpack16x2(u.x, f16), b = unpack16x2(u.y, f16);
    v[0] = a.x, v[1] = a.y, v[2] = b.x, v[3] = b.y;
  } else if constexpr (VEC == 2) {
    const float2 a = unpack16x2(__ldg(reinterpret_cast<const uint32_t*>(ptr)), f16);
    v[0] = a.x, v[1] = a.y;
  } else {
    v[0] = h162f(*ptr, f16);
  }
}
template <int VEC>
__device__ __forceinline__ void store_vec(__nv_bfloat16* ptr, int f16, const float* v) {
  if constexpr (VEC == 8) {
    uint4 o;
    o.x = pack16x2(v[0], v[1], f16), o.y = pack16x2(v[2], v[3], f16);
    o.z = pack16x2(v[4], v[5], f16), o.w = pack16x2(v[6], v[7], f16);
    *reinterpret_cast<uint4*>(ptr) = o;
  } else if constexpr (VEC == 4) {
    *reinterpret_cast<uint2*>(ptr) = make_uint2(pack16x2(v[0], v[1], f16), pack16x2(v[2], v[3], f16));
  } else if constexpr (VEC == 2) {
    *reinterpret_cast<uint32_t*>(ptr) = pack16x2(v[0], v[1], f16);
  } else {
    *ptr = f2h16(v[0], f16);
  }
}

// Pointwise (1x1x1, stride 1, dense) convolution with a tiny channel count on one side (C_in < 8 or C_out < 8: the
// first fast-pathway layers of the efficient backbones, which the tensor-core GEMM cannot address).  One thread = one
// position x one group of up to 8 output channels; the weights sit in shared memory as [c_in][c_out]; inputs are read
// with the widest aligned vector, outputs written as one 16-byte store when the group is full and aligned.
// FLAT: x, y and res are dense over their positions (offset = position * sW), so an item needs no (b, t, h, w)
// decomposition at all; I: 32-bit item index when the item count allows.  With run-time 64-bit divisions the index
// arithmetic of an item (four div/mod pairs) outweighed its cin x 8 FMAs several times over.
template <int VIN, bool FLAT, typename I>
__global__ void __launch_bounds__(256) pw_small_kernel(const DirectParams p, int vec_out) {
  extern __shared__ float pw_sm[];  // w[cin][coutp], bias[coutp]
  const int cin = p.x.C, cout = p.y.C, cogs = (cout + 7) / 8, coutp = cogs * 8;
  for (int i = threadIdx.x; i < cin * coutp; i += blockDim.x) {
    const int ci = i / coutp, co = i - ci * coutp;
    pw_sm[i] = co < cout ? __ldg(p.w + (long long)co * cin + ci) : 0.f;
  }
  float* bias_s = pw_sm + cin * coutp;
  for (int i = threadIdx.x; i < coutp; i += blockDim.x) bias_s[i] = i < cout ? __ldg(p.bias + i) : 0.f;
  __syncthreads();
  // thread = one position, looping over its groups of 8 output channels (the first version gave every (position, group)
  // its own thread: a run-time division per thread -- as many instructions as the cin x 8 FMAs of a 2 -> 12 layer)
  const I total = (I)p.y.B * p.y.T * p.y.H * p.y.W;
  for (I idx = blockIdx.x * (I)blockDim.x + threadIdx.x; idx < total; idx += (I)gridDim.x * blockDim.x) {
    I pos = idx;
    long long xo, yo0, ro0 = 0;
    if constexpr (FLAT) {
      xo = (long long)pos * p.x.sW, yo0 = (long long)pos * p.y.sW;
      if (p.has_res) ro0 = (long long)pos * p.res.sW;
    } else {
      const int w = (int)(pos % p.y.W);
      pos /= p.y.W;
      const int h = (int)(pos % p.y.H);
      pos /= p.y.H;
      const int t = (int)(pos % p.y.T);
      const int b = (int)(pos / p.y.T);
      xo = voff(p.x, b, t, h, w), yo0 = voff(p.y, b, t, h, w);
      if (p.has_res) ro0 = voff(p.res, b, t, h, w);
    }
    const __nv_bfloat16* xr = reinterpret_cast<const __nv_bfloat16*>(p.x.ptr) + xo;
    for (int cog = 0; cog < cogs; ++cog) {
      float acc[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = bias_s[cog * 8 + j];
      for (int c0 = 0; c0 < cin; c0 += VIN) {
        float xv[VIN];
        load_vec<VIN>(xr + c0, p.x.f16, xv);
#pragma unroll
        for (int e = 0; e < VIN; ++e) {
          const float* wr = pw_sm + (c0 + e) * coutp + cog * 8;
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[j] = fmaf(xv[e], wr[j], acc[j]);
        }
      }
      const long long yo = yo0 + cog * 8;
      // y_pad: the row padding may be written too (zero weights + bias there => zeros), which turns the 24-byte row of a
      // 12-channel output into one full 32-byte sector instead of a partial-sector write (read-modify-write in L2)
      const int valid = min(8, (p.y_pad ? p.y_pad : cout) - cog * 8);
      if (p.has_res) {
        const long long ro = ro0 + cog * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (cog * 8 + j < cout) acc[j] += ldbf(p.res, ro + j);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = apply_act(acc[j], p.act);
      __nv_bfloat16* yp = reinterpret_cast<__nv_bfloat16*>(p.y.ptr) + yo;
      if (valid == 8 && vec_out) {
        store_vec<8>(yp, p.y.f16, acc);
      } else if (vec_out) {
        // ragged last group (12 = 8 + 4, 18 = 16 + 2 output channels): the widest aligned pieces, not a scalar loop
        if (valid >= 4) {
          store_vec<4>(yp, p.y.f16, acc);
          if (valid >= 6) {
            store_vec<2>(yp + 4, p.y.f16, acc + 4);
            if (valid == 7) sth(p.y, yo + 6, acc[6]);
          } else if (valid == 5) {
            sth(p.y, yo + 4, acc[4]);
          }
        } else if (valid >= 2) {
          store_vec<2>(yp, p.y.f16, acc);
          if (valid == 3) sth(p.y, yo + 2, acc[2]);
        } else {
          sth(p.y, yo, acc[0]);
        }
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (j < valid) sth(p.y, yo + j, acc[j]);
      }
    }
  }
}

// acc += x * w on 16-bit operands with FP32 accumulation in ONE instruction (sm_100 mixed-precision FMA, SASS FHFMA with
// .H0/.H1 operand selectors): the depthwise inner loop needs no 16->32 bit unpacking at all.
template <bool F16>
__device__ __forceinline__ void mac2(float& a0, float& a1, uint32_t x, uint32_t w) {
  const unsigned short x0 = x & 0xffffu, x1 = x >> 16, w0 = w & 0xffffu, w1 = w >> 16;
  if constexpr (F16) {
    asm("fma.rn.f32.f16 %0, %1, %2, %0;" : "+f"(a0) : "h"(x0), "h"(w0));
    asm("fma.rn.f32.f16 %0, %1, %2, %0;" : "+f"(a1) : "h"(x1), "h"(w1));
  } else {
    asm("fma.rn.f32.bf16 %0, %1, %2, %0;" : "+f"(a0) : "h"(x0), "h"(w0));
    asm("fma.rn.f32.bf16 %0, %1, %2, %0;" : "+f"(a1) : "h"(x1), "h"(w1));
  }
}
template <bool F16>
__device__ __forceinline__ void mac1(float& a0, uint32_t x, uint32_t w) {
  const unsigned short x0 = x & 0xffffu, w0 = w & 0xffffu;
  if constexpr (F16) asm("fma.rn.f32.f16 %0, %1, %2, %0;" : "+f"(a0) : "h"(x0), "h"(w0));
  else asm("fma.rn.f32.bf16 %0, %1, %2, %0;" : "+f"(a0) : "h"(x0), "h"(w0));
}
// VEC 16-bit elements as (VEC + 1) / 2 raw 32-bit words
template <int VEC>
__device__ __forceinline__ void load_raw(const __nv_bfloat16* ptr, uint32_t* v) {
  if constexpr (VEC == 8) {
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(ptr));
    v[0] = u.x, v[1] = u.y, v[2] = u.z, v[3] = u.w;
  } else if constexpr (VEC == 4) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(ptr));
    v[0] = u.x, v[1] = u.y;
  } else if constexpr (VEC == 2) {
    v[0] = __ldg(reinterpret_cast<const uint32_t*>(ptr));
  } else {
    v[0] = __ldg(reinterpret_cast<const unsigned short*>(ptr));
  }
}

// A block owns <= 8 channel groups and walks a (4 x 8 rows x 4 column-blocks) output tile: its input footprint
// (6 x 10 x 18 positions x 64 channels = 138 KB) fits the SM's L1, so the 9 (kt, kh) re-reads of every input row are L1
// hits, and the footprint of all resident blocks fits the L2, so halo re-reads between neighbouring tiles never reach
// DRAM (the first version walked whole rows over 256 channels: 3.1x the algorithmic DRAM reads, ncu).
constexpr int kDwCgPerBlock = 8;
constexpr int kDwTileT = 4, kDwTileH = 8, kDwTileWB = 4;
template <int VEC, int OW, int SW, int KW, bool F16>
__global__ void __launch_bounds__(256, 3) dwconv_kernel(const DirectParams p, int res_vec) {
  extern __shared__ float dw_sm[];  // bias[cb * VEC] (FP32), then w[taps][cb * VEC] in the activations' 16-bit format
  constexpr int NW = (VEC + 1) / 2;
  const int C = p.x.C, cgs = C / VEC;
  const int cg0 = blockIdx.y * kDwCgPerBlock;
  const int cb = min(cgs - cg0, kDwCgPerBlock);  // channel groups of this block
  const int chb = cb * VEC;
  const int taps = p.kT * p.kH * KW;
  float* bias_s = dw_sm;
  __nv_bfloat16* w_s = reinterpret_cast<__nv_bfloat16*>(dw_sm + kDwCgPerBlock * VEC);
  const int c_real = p.c_real ? p.c_real : C;
  for (int i = threadIdx.x; i < taps * chb; i += blockDim.x) {
    const int tap = i / chb, c = i - tap * chb;
    w_s[i] = f2h16(cg0 * VEC + c < c_real ? __ldg(p.w + (long long)(cg0 * VEC + c) * taps + tap) : 0.f, F16);
  }
  for (int i = threadIdx.x; i < chb; i += blockDim.x) bias_s[i] = cg0 * VEC + i < c_real ? __ldg(p.bias + cg0 * VEC + i) : 0.f;
  __syncthreads();
  const int lanes = blockDim.x / cb;
  const int cgl = threadIdx.x % cb, lane = threadIdx.x / cb;
  if (lane >= lanes) return;
  const int wblocks = (p.y.W + OW - 1) / OW;
  const int nth = (p.y.H + kDwTileH - 1) / kDwTileH, ntt = (p.y.T + kDwTileT - 1) / kDwTileT;
  const int nws = (wblocks + kDwTileWB - 1) / kDwTileWB;
  const long long tiles = (long long)p.y.B * ntt * nth * nws;
  constexpr int NCOL = (OW - 1) * SW + KW;
  const __nv_bfloat16* xb = reinterpret_cast<const __nv_bfloat16*>(p.x.ptr) + (cg0 + cgl) * VEC;
  __nv_bfloat16* yb = reinterpret_cast<__nv_bfloat16*>(p.y.ptr) + (cg0 + cgl) * VEC;
  const __nv_bfloat16* rb = reinterpret_cast<const __nv_bfloat16*>(p.res.ptr) + (cg0 + cgl) * VEC;
  const __nv_bfloat16* ws = w_s + cgl * VEC;
  constexpr int per_tile = kDwTileT * kDwTileH * kDwTileWB;
  for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int wsi = tile % nws;
    long long r = tile / nws;
    const int th = r % nth;
    r /= nth;
    const int tt = r % ntt;
    const int b = r / ntt;
    for (int item = lane; item < per_tile; item += lanes) {
      const int wb = wsi * kDwTileWB + item % kDwTileWB, row = item / kDwTileWB;
      const int to = tt * kDwTileT + row / kDwTileH, ho = th * kDwTileH + row % kDwTileH;
      if (to >= p.y.T || ho >= p.y.H || wb >= wblocks) continue;
      const int wi0 = wb * OW * SW - p.pW;
      float acc[OW][2 * NW];
#pragma unroll
      for (int o = 0; o < OW; ++o)
#pragma unroll
        for (int e = 0; e < 2 * NW; ++e) acc[o][e] = e < VEC ? bias_s[cgl * VEC + e] : 0.f;
      for (int kt = 0; kt < p.kT; ++kt) {
        const int ti = to * p.sT + kt - p.pT;
        if (ti < 0 || ti >= p.x.T) continue;
        for (int kh = 0; kh < p.kH; ++kh) {
          const int hi = ho * p.sH + kh - p.pH;
          if (hi < 0 || hi >= p.x.H) continue;
          const __nv_bfloat16* wt = ws + ((kt * p.kH + kh) * KW) * chb;
          uint32_t wv[KW][NW];
#pragma unroll
          for (int kw = 0; kw < KW; ++kw) {
            if constexpr (VEC == 8) {
              const uint4 u = *reinterpret_cast<const uint4*>(wt + kw * chb);
              wv[kw][0] = u.x, wv[kw][1] = u.y, wv[kw][2] = u.z, wv[kw][3] = u.w;
            } else if constexpr (VEC == 4) {
              const uint2 u = *reinterpret_cast<const uint2*>(wt + kw * chb);
              wv[kw][0] = u.x, wv[kw][1] = u.y;
            } else if constexpr (VEC == 2) {
              wv[kw][0] = *reinterpret_cast<const uint32_t*>(wt + kw * chb);
            } else {
              wv[kw][0] = *reinterpret_cast<const unsigned short*>(wt + kw * chb);
            }
          }
          const long long rowoff = voff(p.x, b, ti, hi, 0);
          uint32_t xv[NCOL][NW];   // all columns of the row first: NCOL independent loads in flight
#pragma unroll
          for (int col = 0; col < NCOL; ++col) {
            const int wi = wi0 + col;
            if (wi >= 0 && wi < p.x.W) load_raw<VEC>(xb + rowoff + wi * p.x.sW, xv[col]);
            else {
#pragma unroll
              for (int q = 0; q < NW; ++q) xv[col][q] = 0u;
            }
          }
#pragma unroll
          for (int col = 0; col < NCOL; ++col) {
#pragma unroll
            for (int kw = 0; kw < KW; ++kw) {
              if ((col - kw) % SW == 0 && col - kw >= 0 && (col - kw) / SW < OW) {
                const int o = (col - kw) / SW;
#pragma unroll
                for (int q = 0; q < NW; ++q) {
                  if constexpr (VEC == 1) mac1<F16>(acc[o][0], xv[col][0], wv[kw][0]);
                  else mac2<F16>(acc[o][2 * q], acc[o][2 * q + 1], xv[col][q], wv[kw][q]);
                }
              }
            }
          }
        }
      }
#pragma unroll
      for (int o = 0; o < OW; ++o) {
        const int wo = wb * OW + o;
        if (wo >= p.y.W) break;
        if (p.has_res) {
          const long long ro = voff(p.res, b, to, ho, wo);
          float rv[VEC];
          if (res_vec) load_vec<VEC>(rb + ro, F16, rv);
          else {
#pragma unroll
            for (int e = 0; e < VEC; ++e) rv[e] = h162f(rb[ro + e], F16);
          }
#pragma unroll
          for (int e = 0; e < VEC; ++e) acc[o][e] += rv[e];
        }
#pragma unroll
        for (int e = 0; e < VEC; ++e) acc[o][e] = apply_act(acc[o][e], p.act);
        store_vec<VEC>(yb + voff(p.y, b, to, ho, wo), F16, acc[o]);
      }
    }
  }
}

// Depthwise kT x 3 x 3 (pad 1 in H and W, stride 1 or 2) as a MARCH down the rows: one thread = VEC channels x OW output
// columns of one (b, t_out) and walks `hs` consecutive output rows.  Every input row is loaded ONCE per kt (NCOL 16-byte
// loads) and feeds all three kh taps out of registers -- the rolling accumulators of the 3 (stride 1) / 2 (stride 2)
// output rows that are in flight live in registers with compile-time slot numbers (the row loop is unrolled by the
// rotation period).  The tile kernel above re-read every input row for each (kt, kh) from L1: per output element it
// moved 27 B through the L1 next to 27 FMAs, i.e. the 128 B/clk L1 port and the FMA pipe saturated together (ncu: FMA
// 37 %, issue 69 %).  Here the L1 traffic is 3x lower and the FMAs are what is left.  Consecutive threads are
// consecutive channel groups, then `wbg` column blocks, then t_out -- a block covers a few output planes of the same
// columns, so the kt re-reads of a row by the neighbouring planes hit L1.  All weights of the layer sit in shared memory
// in the activations' 16-bit format ([tap][C]); blocks are persistent (grid-stride), so they are staged once.
template <int VEC, int OW, int SW, bool F16>
struct DwMarch {
  static constexpr int NW = (VEC + 1) / 2;
  static constexpr int NCOL = (OW - 1) * SW + 3;
  static constexpr int NS = SW == 1 ? 3 : 2;
  float acc[NS][OW][2 * NW];
  const DirectParams& p;
  const __nv_bfloat16* xb;   // x + b * sB + channel offset
  const __nv_bfloat16* ws;   // smem weights + channel offset, [tap][C]
  const float* bias_s;       // smem bias + channel offset
  int C, to, wi0, colmask;
  __device__ __forceinline__ DwMarch(const DirectParams& p_) : p(p_) {}

  template <int S>
  __device__ __forceinline__ void reset() {
#pragma unroll
    for (int o = 0; o < OW; ++o)
#pragma unroll
      for (int e = 0; e < 2 * NW; ++e) acc[S][o][e] = e < VEC ? bias_s[e] : 0.f;
  }
  template <int S>
  __device__ __forceinline__ void fma_kh(const uint32_t (&xv)[NCOL][NW], const __nv_bfloat16* wt) {
    if constexpr (S >= 0) {
      uint32_t wv[3][NW];
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        if constexpr (VEC == 8) {
          const uint4 u = *reinterpret_cast<const uint4*>(wt + kw * C);
          wv[kw][0] = u.x, wv[kw][1] = u.y, wv[kw][2] = u.z, wv[kw][3] = u.w;
        } else if constexpr (VEC == 4) {
          const uint2 u = *reinterpret_cast<const uint2*>(wt + kw * C);
          wv[kw][0] = u.x, wv[kw][1] = u.y;
        } else if constexpr (VEC == 2) {
          wv[kw][0] = *reinterpret_cast<const uint32_t*>(wt + kw * C);
        } else {
          wv[kw][0] = *reinterpret_cast<const unsigned short*>(wt + kw * C);
        }
      }
#pragma unroll
      for (int col = 0; col < NCOL; ++col) {
#pragma unroll
        for (int kw = 0; kw < 3; ++kw) {
          if ((col - kw) % SW == 0 && col - kw >= 0 && (col - kw) / SW < OW) {
            const int o = (col - kw) / SW;
#pragma unroll
            for (int q = 0; q < NW; ++q) {
              if constexpr (VEC == 1) mac1<F16>(acc[S][o][0], xv[col][0], wv[kw][0]);
              else mac2<F16>(acc[S][o][2 * q], acc[S][o][2 * q + 1], xv[col][q], wv[kw][q]);
            }
          }
        }
      }
    }
  }
  // input row hi: tap kh accumulates into slot S<kh> when m<kh> (the output row of that tap is one of ours)
  template <int S0, int S1, int S2>
  __device__ __forceinline__ void step(int hi, bool m0, bool m1, bool m2) {
    if (hi < 0 || hi >= p.x.H) return;
    const __nv_bfloat16* xrow = xb + (long long)hi * p.x.sH;
    for (int kt = 0; kt < p.kT; ++kt) {
      const int ti = to * p.sT + kt - p.pT;
      if (ti < 0 || ti >= p.x.T) continue;
      const __nv_bfloat16* rp = xrow + (long long)ti * p.x.sT;
      uint32_t xv[NCOL][NW];
#pragma unroll
      for (int col = 0; col < NCOL; ++col) {
        if ((colmask >> col) & 1) load_raw<VEC>(rp + (long long)(wi0 + col) * p.x.sW, xv[col]);
        else {
#pragma unroll
          for (int q = 0; q < NW; ++q) xv[col][q] = 0u;
        }
      }
      const __nv_bfloat16* wt = ws + kt * 9 * C;
      if (S0 >= 0 && m0) fma_kh<S0>(xv, wt);
      if (S1 >= 0 && m1) fma_kh<S1>(xv, wt + 3 * C);
      if (S2 >= 0 && m2) fma_kh<S2>(xv, wt + 6 * C);
    }
  }
  template <int S>
  __device__ __forceinline__ void store(long long yrow, int wb, int res_vec, const __nv_bfloat16* rb,
                                        __nv_bfloat16* yb) {
#pragma unroll
    for (int o = 0; o < OW; ++o) {
      const int wo = wb * OW + o;
      if (wo < p.y.W) {
        if (p.has_res) {
          // res has the geometry of y but its own strides
          float rv[VEC];
          const long long ro = yrow_res + wo * p.res.sW;
          if (res_vec) load_vec<VEC>(rb + ro, F16, rv);
          else {
#pragma unroll
            for (int e = 0; e < VEC; ++e) rv[e] = h162f(rb[ro + e], F16);
          }
#pragma unroll
          for (int e = 0; e < VEC; ++e) acc[S][o][e] += rv[e];
        }
#pragma unroll
        for (int e = 0; e < VEC; ++e) acc[S][o][e] = apply_act(acc[S][o][e], p.act);
        store_vec<VEC>(yb + yrow + wo * p.y.sW, F16, acc[S][o]);
      }
    }
    reset<S>();
  }
  long long yrow_res;
};

template <int VEC, int OW, int SW, bool F16>
__global__ void __launch_bounds__(128) dwconv_march_kernel(const DirectParams p, int res_vec, int hs, int wbg) {
  extern __shared__ float dwm_sm[];  // bias[C] (FP32), then w[kT * 9][C] in the activations' 16-bit format
  using M = DwMarch<VEC, OW, SW, F16>;
  const int C = p.x.C, cgs = C / VEC;
  const int taps = p.kT * 9;
  float* bias_all = dwm_sm;
  __nv_bfloat16* w_all = reinterpret_cast<__nv_bfloat16*>(dwm_sm + C);
  const int c_real = p.c_real ? p.c_real : C;
  for (int i = threadIdx.x; i < taps * C; i += blockDim.x) {
    const int tap = i / C, c = i - tap * C;
    w_all[i] = f2h16(c < c_real ? __ldg(p.w + (long long)c * taps + tap) : 0.f, F16);
  }
  for (int i = threadIdx.x; i < C; i += blockDim.x) bias_all[i] = i < c_real ? __ldg(p.bias + i) : 0.f;
  __syncthreads();
  const int wblocks = (p.y.W + OW - 1) / OW, nwg = (wblocks + wbg - 1) / wbg, nseg = (p.y.H + hs - 1) / hs;
  const long long items = (long long)p.y.B * nseg * nwg * p.y.T * wbg * cgs;
  M m(p);
  m.C = C;
  for (long long item = blockIdx.x * (long long)blockDim.x + threadIdx.x; item < items;
       item += (long long)gridDim.x * blockDim.x) {
    const int cg = (int)(item % cgs);
    long long r = item / cgs;
    const int wl = (int)(r % wbg);
    r /= wbg;
    const int to = (int)(r % p.y.T);
    r /= p.y.T;
    const int wg = (int)(r % nwg);
    r /= nwg;
    const int seg = (int)(r % nseg);
    const int b = (int)(r / nseg);
    const int wb = wg * wbg + wl;
    if (wb >= wblocks) continue;
    const int ho0 = seg * hs, ho1 = min(ho0 + hs, p.y.H);
    m.to = to;
    m.wi0 = wb * OW * SW - 1;
    int mask = 0;
#pragma unroll
    for (int col = 0; col < M::NCOL; ++col) mask |= (m.wi0 + col >= 0 && m.wi0 + col < p.x.W) ? (1 << col) : 0;
    m.colmask = mask;
    m.xb = reinterpret_cast<const __nv_bfloat16*>(p.x.ptr) + b * p.x.sB + cg * VEC;
    m.ws = w_all + cg * VEC;
    m.bias_s = bias_all + cg * VEC;
    __nv_bfloat16* yb = reinterpret_cast<__nv_bfloat16*>(p.y.ptr) + b * p.y.sB + to * p.y.sT + cg * VEC;
    const __nv_bfloat16* rb = reinterpret_cast<const __nv_bfloat16*>(p.res.ptr) + b * p.res.sB + to * p.res.sT + cg * VEC;
    m.template reset<0>();
    m.template reset<1>();
    if constexpr (SW == 1) m.template reset<2>();
#define DW_STORE(S, ho)                                                     \
  do {                                                                      \
    m.yrow_res = (long long)(ho) * p.res.sH;                                \
    m.template store<S>((long long)(ho) * p.y.sH, wb, res_vec, rb, yb);     \
  } while (0)
    if constexpr (SW == 1) {
      // stride 1: input row hi feeds output rows hi+1 (kh 0), hi (kh 1), hi-1 (kh 2); row hi-1 is complete after it
      int hi = ho0 - 1;
      while (true) {
        m.template step<2, 1, 0>(hi, hi + 1 < ho1, hi >= ho0 && hi < ho1, hi - 1 >= ho0);
        if (hi - 1 >= ho0) DW_STORE(0, hi - 1);
        if (hi >= ho1) break;
        ++hi;
        m.template step<0, 2, 1>(hi, hi + 1 < ho1, hi >= ho0 && hi < ho1, hi - 1 >= ho0);
        if (hi - 1 >= ho0) DW_STORE(1, hi - 1);
        if (hi >= ho1) break;
        ++hi;
        m.template step<1, 0, 2>(hi, hi + 1 < ho1, hi >= ho0 && hi < ho1, hi - 1 >= ho0);
        if (hi - 1 >= ho0) DW_STORE(2, hi - 1);
        if (hi >= ho1) break;
        ++hi;
      }
    } else {
      // stride 2: output row ho reads input rows 2ho-1 (kh 0), 2ho (kh 1), 2ho+1 (kh 2); row 2ho+1 is also kh 0 of ho+1
      m.template step<0, -1, -1>(2 * ho0 - 1, true, false, false);
      int ho = ho0;
      while (true) {
        m.template step<-1, 0, -1>(2 * ho, false, true, false);
        m.template step<1, -1, 0>(2 * ho + 1, ho + 1 < ho1, false, true);
        DW_STORE(0, ho);
        if (++ho >= ho1) break;
        m.template step<-1, 1, -1>(2 * ho, false, true, false);
        m.template step<0, -1, 1>(2 * ho + 1, ho + 1 < ho1, false, true);
        DW_STORE(1, ho);
        if (++ho >= ho1) break;
      }
    }
#undef DW_STORE
  }
}

// Depthwise kT x 3 x 3 with SHARED-MEMORY HALO STAGING: the march above, fed by TMA instead of per-thread global loads.
// A block of 128 threads owns a tile of cb channel groups (cb x 8 channels = one <= 128-byte row) x wbt column blocks of
// 4 outputs x tt output planes and marches down `hs` output rows.  Per input row ONE 5-D TMA box
// {cb*8 channels, ncols, 1 row, planes, 1 clip} lands in a ring of `stages` buffers (mbarrier complete_tx); the filter
// halo in W and T is part of the box, zero padding is TMA out-of-bounds fill, so the compute loop has no bounds tests
// and no global-load latency at all: 6 (stride 1) / 9 (stride 2) LDS.128 of activations and 9 LDS.128 of weights per
// 288 / 144 FMAs, the three kh taps of a row served from registers.  Measured against the tile kernel and the
// global-load march: DESIGN.md 3.5.
struct DwTmaParams {
  DirectParams p;
  int cb, wbt, tt, hs, stages, ncols, planes, nct, nwt, ntt, nseg, cgs, wblocks;
  uint32_t stage_bytes, stage_stride;   // TMA box bytes; ring pitch (128-byte aligned destinations)
  long long tiles;
};
constexpr int kDwTmaMaxStages = 4;
constexpr int kDwTmaHeader = 128;    // mbarriers

template <int SW, int KT, bool F16>
struct DwTma {
  // thread = 2 channels (one 32-bit word per position) x OW output columns: the KT x 9 filter taps of its channel pair
  // stay in registers for the whole kernel, a warp reads 32 consecutive words of a staged row per LDS (one wavefront)
  static constexpr int OW = 8, NCOL = (OW - 1) * SW + 3, NS = SW == 1 ? 3 : 2;
  float acc[NS][OW][2];
  uint32_t w[KT * 9];
  float bias[2];
  const DirectParams& p;
  uint32_t xoff, pitch, plane_bytes;
  __device__ __forceinline__ DwTma(const DirectParams& p_) : p(p_) {}
  template <int S>
  __device__ __forceinline__ void reset() {
#pragma unroll
    for (int o = 0; o < OW; ++o) acc[S][o][0] = bias[0], acc[S][o][1] = bias[1];
  }
  template <int S, int KT_, int KH>
  __device__ __forceinline__ void fma_kh(const uint32_t (&xv)[NCOL]) {
    if constexpr (S >= 0) {
#pragma unroll
      for (int col = 0; col < NCOL; ++col) {
#pragma unroll
        for (int kw = 0; kw < 3; ++kw) {
          if ((col - kw) % SW == 0 && col - kw >= 0 && (col - kw) / SW < OW) {
            const int o = (col - kw) / SW;
            mac2<F16>(acc[S][o][0], acc[S][o][1], xv[col], w[(KT_ * 3 + KH) * 3 + kw]);
          }
        }
      }
    }
  }
  template <int S0, int S1, int S2, int KT_>
  __device__ __forceinline__ void plane(const char* xp, bool m0, bool m1, bool m2) {
    uint32_t xv[NCOL];
#pragma unroll
    for (int col = 0; col < NCOL; ++col) xv[col] = *reinterpret_cast<const uint32_t*>(xp + col * pitch);
    if (S0 >= 0 && m0) fma_kh<S0, KT_, 0>(xv);
    if (S1 >= 0 && m1) fma_kh<S1, KT_, 1>(xv);
    if (S2 >= 0 && m2) fma_kh<S2, KT_, 2>(xv);
  }
  template <int S0, int S1, int S2>
  __device__ __forceinline__ void compute(const char* stage, bool m0, bool m1, bool m2) {
    const char* xp = stage + xoff;
    plane<S0, S1, S2, 0>(xp, m0, m1, m2);
    if constexpr (KT == 3) {
      plane<S0, S1, S2, 1>(xp + plane_bytes, m0, m1, m2);
      plane<S0, S1, S2, 2>(xp + 2 * plane_bytes, m0, m1, m2);
    }
  }
  // Row store.  ncu on the first version: the per-column 64-bit address arithmetic, bounds test, residual / activation
  // branches of this path cost ~90 instructions per output column -- with 2 channels per thread as many issue slots as
  // the 432 FMAs of the row.  Now: 32-bit column offsets from a per-row pointer, activation as a clamp, the residual
  // decided once per row.
  float act_lo, act_hi;
  int y_sw, r_sw;
  template <int S, bool RES>
  __device__ __forceinline__ void store_row(__nv_bfloat16* yrow, const __nv_bfloat16* rrow, int nvalid) {
#pragma unroll
    for (int o = 0; o < OW; ++o) {
      if (o < nvalid) {
        float v0 = acc[S][o][0], v1 = acc[S][o][1];
        if constexpr (RES) {
          const float2 rv = unpack16x2(__ldg(reinterpret_cast<const uint32_t*>(rrow + o * r_sw)), F16);
          v0 += rv.x, v1 += rv.y;
        }
        v0 = fmaxf(v0, act_lo), v1 = fmaxf(v1, act_lo);
        if (p.act == 2) v0 = fminf(v0, act_hi), v1 = fminf(v1, act_hi);
        *reinterpret_cast<uint32_t*>(yrow + o * y_sw) = pack16x2(v0, v1, F16);
      }
    }
    reset<S>();
  }
  template <int S>
  __device__ __forceinline__ void store(__nv_bfloat16* yrow, const __nv_bfloat16* rrow, int nvalid) {
    if (p.has_res) store_row<S, true>(yrow, rrow, nvalid);
    else store_row<S, false>(yrow, rrow, nvalid);
  }
};

template <int SW, int KT, bool F16>
__global__ void __launch_bounds__(256, 2) dwconv_tma_kernel(const __grid_constant__ CUtensorMap xmap,
                                                            const __grid_constant__ DwTmaParams q) {
  extern __shared__ __align__(128) char dwt_sm[];
  using M = DwTma<SW, KT, F16>;
  const DirectParams& p = q.p;
  uint64_t* full = reinterpret_cast<uint64_t*>(dwt_sm);
  char* stages = dwt_sm + kDwTmaHeader;
  const int tid = threadIdx.x;
  const int cb = q.cb, chb = cb * 2;   // channel pairs / channels of a block tile
  constexpr int taps = KT * 9;
  const int c_real = p.c_real ? p.c_real : p.x.C;
  if (tid == 0) {
    for (int i = 0; i < q.stages; ++i) mbar_init(&full[i], 1);
    fence_barrier_init();
    prefetch_tmap(&xmap);
  }
  __syncthreads();
  const int cg = tid % cb, lane = tid / cb;
  const int wb = lane % q.wbt, tl = lane / q.wbt;
  // ---- producer cursor (thread 0): one TMA box per valid input row of every tile of this block, q.stages ahead
  // (the cursor lives in shared memory: only thread 0 touches it, and the compute threads need every register)
  struct Cursor {
    long long tile;
    int hi, hi_end, c0, w0, t0, b;
  };
  Cursor& pc = *reinterpret_cast<Cursor*>(dwt_sm + 64);
#define p_tile pc.tile
#define p_hi pc.hi
#define p_hi_end pc.hi_end
#define p_c0 pc.c0
#define p_w0 pc.w0
#define p_t0 pc.t0
#define p_b pc.b
  auto decode = [&](long long tile, int& wt, int& tt, int& seg, int& b, int& ct) {
    // channel tile fastest: the tiles of one spatial region run at the same time, so the 256-byte L2 promotion of a
    // < 128-byte tile row is shared (ncu with the channel tile slowest: 2.5x the algorithmic DRAM reads at C = 144)
    ct = (int)(tile % q.nct);
    long long r = tile / q.nct;
    wt = (int)(r % q.nwt);
    r /= q.nwt;
    tt = (int)(r % q.ntt);
    r /= q.ntt;
    seg = (int)(r % q.nseg);
    b = (int)(r / q.nseg);
  };
  auto open_tile = [&]() {
    if (p_tile >= q.tiles) return;
    int wt, tt, seg, b, ct;
    decode(p_tile, wt, tt, seg, b, ct);
    const int ho0 = seg * q.hs, ho1 = min(ho0 + q.hs, p.y.H);   // input rows the segment consumes, clipped
    p_hi = max(ho0 * SW - 1, 0);
    p_hi_end = min((ho1 - 1) * SW + 1, p.x.H - 1);
    p_c0 = ct * chb, p_w0 = wt * q.wbt * M::OW * SW - 1, p_t0 = tt * q.tt * p.sT - p.pT, p_b = b;
  };
  auto issue_next = [&](uint32_t s) {   // s: the ring slot to fill (the one the block has just finished reading)
    if (p_tile >= q.tiles) return;
    mbar_arrive_expect_tx(&full[s], q.stage_bytes);
    tma_load_5d(stages + (size_t)s * q.stage_stride, &xmap, &full[s], p_c0, p_w0, p_hi, p_t0, p_b);
    if (++p_hi > p_hi_end) {
      p_tile += gridDim.x;
      open_tile();
    }
  };
  if (tid == 0) {
    p_tile = blockIdx.x;
    open_tile();
    for (int i = 0; i < q.stages; ++i) issue_next(i);
  }
#undef p_tile
#undef p_hi
#undef p_hi_end
#undef p_c0
#undef p_w0
#undef p_t0
#undef p_b
  M m(p);
  m.pitch = chb * 2;
  m.plane_bytes = q.ncols * m.pitch;
  m.xoff = (uint32_t)((tl * p.sT * q.ncols + wb * M::OW * SW) * (int)m.pitch + cg * 4);
  m.act_lo = p.act == 0 ? -CUDART_INF_F : 0.f;
  m.act_hi = p.act == 2 ? 6.f : CUDART_INF_F;
  m.y_sw = (int)p.y.sW, m.r_sw = (int)p.res.sW;
  uint32_t rs = 0, rph = 0;   // ring slot and phase parity of the next row to consume
  int cur_ct = -1;
  for (long long tile = blockIdx.x; tile < q.tiles; tile += gridDim.x) {
    int wt, tt, seg, b, ct;
    decode(tile, wt, tt, seg, b, ct);
    const int ch = ct * chb + cg * 2;
    if (ct != cur_ct) {   // filter taps + bias of this thread's channel pair
#pragma unroll
      for (int tap = 0; tap < taps; ++tap) {
        const float w0 = ch < c_real ? __ldg(p.w + (long long)ch * taps + tap) : 0.f;
        const float w1 = ch + 1 < c_real ? __ldg(p.w + (long long)(ch + 1) * taps + tap) : 0.f;
        m.w[tap] = pack16x2(w0, w1, F16);
      }
      m.bias[0] = ch < c_real ? __ldg(p.bias + ch) : 0.f;
      m.bias[1] = ch + 1 < c_real ? __ldg(p.bias + ch + 1) : 0.f;
      cur_ct = ct;
    }
    const int ho0 = seg * q.hs, ho1 = min(ho0 + q.hs, p.y.H);
    const int to = tt * q.tt + tl, wbg = wt * q.wbt + wb;
    const bool active = tl < q.tt && to < p.y.T && wbg < q.wblocks && ch < p.x.C;
    const int nvalid = p.y.W - wbg * M::OW;   // output columns of this thread inside the tensor (>= OW: all)
    __nv_bfloat16* yb = reinterpret_cast<__nv_bfloat16*>(p.y.ptr) + b * p.y.sB + to * p.y.sT +
                        (long long)wbg * M::OW * p.y.sW + ch;
    const __nv_bfloat16* rb = reinterpret_cast<const __nv_bfloat16*>(p.res.ptr) + b * p.res.sB + to * p.res.sT +
                              (long long)wbg * M::OW * p.res.sW + ch;
    m.template reset<0>();
    m.template reset<1>();
    if constexpr (SW == 1) m.template reset<2>();
#define DW_ROW(S0, S1, S2, hi, m0, m1, m2)                                                        \
  do {                                                                                            \
    if ((hi) >= 0 && (hi) < p.x.H) {                                                              \
      mbar_wait(&full[rs], rph, 7);                                                               \
      if (active) m.template compute<S0, S1, S2>(stages + rs * q.stage_stride, m0, m1, m2);       \
      __syncthreads();                                                                            \
      if (tid == 0) issue_next(rs);                                                               \
      if (++rs == (uint32_t)q.stages) rs = 0, rph ^= 1;                                           \
    }                                                                                             \
  } while (0)
#define DW_STORE(S, ho)                                                                                 \
  do {                                                                                                  \
    if (active) m.template store<S>(yb + (long long)(ho) * p.y.sH, rb + (long long)(ho) * p.res.sH, nvalid); \
  } while (0)
    if constexpr (SW == 1) {
      // stride 1: input row hi feeds output rows hi+1 (kh 0), hi (kh 1), hi-1 (kh 2); row hi-1 is complete after it
      int hi = ho0 - 1;
      while (true) {
        DW_ROW(2, 1, 0, hi, hi + 1 < ho1, hi >= ho0 && hi < ho1, hi - 1 >= ho0);
        if (hi - 1 >= ho0) DW_STORE(0, hi - 1);
        if (hi >= ho1) break;
        ++hi;
        DW_ROW(0, 2, 1, hi, hi + 1 < ho1, hi >= ho0 && hi < ho1, hi - 1 >= ho0);
        if (hi - 1 >= ho0) DW_STORE(1, hi - 1);
        if (hi >= ho1) break;
        ++hi;
        DW_ROW(1, 0, 2, hi, hi + 1 < ho1, hi >= ho0 && hi < ho1, hi - 1 >= ho0);
        if (hi - 1 >= ho0) DW_STORE(2, hi - 1);
        if (hi >= ho1) break;
        ++hi;
      }
    } else {
      // stride 2: output row ho reads input rows 2ho-1 (kh 0), 2ho (kh 1), 2ho+1 (kh 2); row 2ho+1 is also kh 0 of ho+1
      DW_ROW(0, -1, -1, 2 * ho0 - 1, true, false, false);
      int ho = ho0;
      while (true) {
        DW_ROW(-1, 0, -1, 2 * ho, false, true, false);
        DW_ROW(1, -1, 0, 2 * ho + 1, ho + 1 < ho1, false, true);
        DW_STORE(0, ho);
        if (++ho >= ho1) break;
        DW_ROW(-1, 1, -1, 2 * ho, false, true, false);
        DW_ROW(0, -1, 1, 2 * ho + 1, ho + 1 < ho1, false, true);
        DW_STORE(1, ho);
        if (++ho >= ho1) break;
      }
    }
#undef DW_ROW
#undef DW_STORE
  }
}

static bool vec_ok(const View& v, int vec);
// false = geometry not covered (caller falls back to the global-load kernels)
static bool launch_dwconv_tma(const DirectParams& p, cudaStream_t s) {
  if (!vec_ok(p.x, 8) || !vec_ok(p.y, 2) || p.x.C % 8 != 0 || (p.kT != 1 && p.kT != 3)) return false;
  if (p.has_res && !vec_ok(p.res, 2)) return false;
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return false;
  constexpr int OW = 8, kThreads = 256;
  DwTmaParams q;
  q.p = p;
  const int SW = p.sW;
  // Tile search: channels per block (a multiple of 8 = 16-byte TMA rows; 2 per thread), column blocks and output
  // planes per block, maximising the fraction of the 256 threads that own real outputs (C = 144: 48 channels x 1 x 8
  // planes or 72 x 7 x 1 instead of 64-channel tiles with a quarter of the lanes idle -- ncu: barrier stalls 2.2 per
  // issue), then the smallest halo; the stage has to leave room for >= 3 stages x 2 blocks per SM.
  const int c8 = p.x.C / 8;
  q.cgs = p.x.C / 2;
  q.wblocks = cdiv(p.y.W, OW);
  int cb = 0, wbt = 1, tt = 1;
  double best = -1;
  for (int ch8 = std::min(c8, 16); ch8 >= 1; --ch8) {
    const int cbc = ch8 * 4;
    if (cbc > kThreads) continue;
    if (ch8 == 1 && c8 > 1) continue;   // 16-byte rows: too many TMA rows / DRAM sectors per byte
    const int lanes = kThreads / cbc, nct = cdiv(c8, ch8);
    for (int w = 1; w <= std::min(lanes, q.wblocks); ++w) {
      int t = std::min(p.y.T, lanes / w);
      t = cdiv(p.y.T, cdiv(p.y.T, t));
      const int ncols = (w * OW - 1) * SW + 3, planes = (t - 1) * p.sT + p.kT;
      const size_t bytes = (size_t)cbc * 4 * ncols * planes;
      if (bytes > 24 * 1024 || ncols > 256 || planes > 256) continue;
      const double eff = (double)(p.x.C / 2) * q.wblocks * p.y.T /
                         ((double)nct * cdiv(q.wblocks, w) * cdiv(p.y.T, t) * kThreads);
      const double halo = ((double)ncols / (w * OW * SW)) * ((double)planes / (t * p.sT));
      // full-warp channel rows read conflict-free; rows under 64 bytes cost TMA rows and partial DRAM bursts
      const double score = eff - 0.02 * halo - (cbc % 32 ? 0.01 : 0.0) - (ch8 < 4 ? 0.03 * (4 - ch8) : 0.0);
      if (score > best) best = score, cb = cbc, wbt = w, tt = t;
    }
  }
  if (cb == 0) return false;
  q.cb = cb;
  q.nct = cdiv(q.cgs, cb);
  q.wbt = wbt, q.tt = tt;
  q.ncols = (wbt * OW - 1) * SW + 3;
  q.planes = (tt - 1) * p.sT + p.kT;
  q.stage_bytes = (uint32_t)(cb * 4 * q.ncols * q.planes);
  q.stage_stride = (q.stage_bytes + 127u) & ~127u;
  if (q.ncols > 256 || q.planes > 256 || q.stage_bytes > 32 * 1024) return false;
  q.stages = std::max(2, std::min(kDwTmaMaxStages, (int)((100 * 1024 - kDwTmaHeader) / q.stage_stride)));
  q.nwt = cdiv(q.wblocks, wbt), q.ntt = cdiv(p.y.T, tt);
  // rows per segment: long segments amortise the two halo rows (16 rows: 18 row steps, 32 rows: 34), short ones fill
  // the last wave of the persistent grid; pick by (useful rows / row steps) x (tiles / tiles rounded up to whole waves)
  const long long per_seg = (long long)q.nct * p.y.B * q.ntt * q.nwt;
  const long long wave = (long long)std::max(num_sms(), 1) * 2;
  double best_hs = -1;
  for (int target : {16, 32, 56}) {
    const int nseg = cdiv(p.y.H, target), hs = cdiv(p.y.H, nseg);
    const long long tiles = per_seg * cdiv(p.y.H, hs);
    const double rows = (double)hs * SW / (hs * SW + (SW == 1 ? 2 : 1));
    const double waves = (double)tiles / (double)(cdiv((int)std::min<long long>(tiles, 1 << 30), (int)wave) * wave);
    if (rows * waves > best_hs) best_hs = rows * waves, q.hs = hs;
  }
  q.nseg = cdiv(p.y.H, q.hs);
  q.tiles = per_seg * q.nseg;
  CUtensorMap xmap;
  {
    const int c_map = p.c_real ? p.c_real : p.x.C;   // padding channels of the rows read as zeros
    cuuint64_t dims[5] = {(cuuint64_t)c_map, (cuuint64_t)p.x.W, (cuuint64_t)p.x.H, (cuuint64_t)p.x.T, (cuuint64_t)p.x.B};
    cuuint64_t strides[4] = {(cuuint64_t)p.x.sW * 2, (cuuint64_t)p.x.sH * 2, (cuuint64_t)p.x.sT * 2, (cuuint64_t)p.x.sB * 2};
    cuuint32_t box[5] = {(cuuint32_t)(cb * 2), (cuuint32_t)q.ncols, 1, (cuuint32_t)q.planes, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    if (enc(&xmap, p.x.f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, p.x.ptr, dims, strides,
            box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return false;
  }
  const size_t smem = kDwTmaHeader + (size_t)q.stages * q.stage_stride;
  const unsigned grid = (unsigned)std::min<long long>(q.tiles, (long long)std::max(num_sms(), 1) * 2);
  auto launch = [&](auto kern) {
    if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 104 * 1024);
    kern<<<grid, kThreads, smem, s>>>(xmap, q);
  };
  const int key = (p.x.f16 ? 4 : 0) | (SW == 2 ? 2 : 0) | (p.kT == 3 ? 1 : 0);
  switch (key) {
    case 0: launch(dwconv_tma_kernel<1, 1, false>); break;
    case 1: launch(dwconv_tma_kernel<1, 3, false>); break;
    case 2: launch(dwconv_tma_kernel<2, 1, false>); break;
    case 3: launch(dwconv_tma_kernel<2, 3, false>); break;
    case 4: launch(dwconv_tma_kernel<1, 1, true>); break;
    case 5: launch(dwconv_tma_kernel<1, 3, true>); break;
    case 6: launch(dwconv_tma_kernel<2, 1, true>); break;
    default: launch(dwconv_tma_kernel<2, 3, true>); break;
  }
  return true;
}

template <int VEC>
static bool launch_dwconv_march(const DirectParams& p, cudaStream_t s) {
  const int C = p.x.C, cgs = C / VEC;
  const int taps = p.kT * 9;
  const size_t smem = (size_t)C * (sizeof(float) + taps * 2);
  if (smem > 96 * 1024) return false;
  constexpr int OW = 4;
  const int res_vec = p.has_res && vec_ok(p.res, VEC);
  const int nseg = cdiv(p.y.H, 16);
  const int hs = cdiv(p.y.H, nseg);
  const int wblocks = cdiv(p.y.W, OW);
  const int wbg = std::max(1, std::min(wblocks, 32 / std::max(cgs, 1)));
  const long long items = (long long)p.y.B * cdiv(p.y.H, hs) * cdiv(wblocks, wbg) * p.y.T * wbg * cgs;
  const unsigned grid = (unsigned)std::min<long long>((items + 127) / 128, 148 * 16);
  auto launch = [&](auto kern) {
    if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
    kern<<<grid, 128, smem, s>>>(p, res_vec, hs, wbg);
  };
  if (p.x.f16) {
    if (p.sW == 1) launch(dwconv_march_kernel<VEC, OW, 1, true>);
    else launch(dwconv_march_kernel<VEC, OW, 2, true>);
  } else {
    if (p.sW == 1) launch(dwconv_march_kernel<VEC, OW, 1, false>);
    else launch(dwconv_march_kernel<VEC, OW, 2, false>);
  }
  return true;
}

template <int VEC, int KW>
static bool launch_dwconv(const DirectParams& p, cudaStream_t s) {
  if constexpr (KW == 3) {
    if (p.kH == 3 && p.pH == 1 && p.pW == 1 && p.sH == p.sW) {
      // the TMA-staged march; rows that TMA cannot address (C < 8: 4- or 8-byte pitch) take the global-load march
      // (C = 4 @112^2: 0.286 -> 0.198 ms).  Either may decline a geometry: then the tile kernel below runs.
      if constexpr (VEC == 8) {
        if (launch_dwconv_tma(p, s)) return true;
      } else {
        if (launch_dwconv_march<VEC>(p, s)) return true;
      }
    }
  }
  const int cgs = p.x.C / VEC;
  const int taps = p.kT * p.kH * KW;
  const size_t smem = (size_t)kDwCgPerBlock * VEC * (sizeof(float) + taps * 2);
  if (smem > 48 * 1024) return false;
  const int res_vec = p.has_res && vec_ok(p.res, VEC);
  const int ow = p.sW == 1 ? 4 : 2;
  const long long tiles = (long long)p.y.B * cdiv(p.y.T, kDwTileT) * cdiv(p.y.H, kDwTileH) *
                          cdiv(cdiv(p.y.W, ow), kDwTileWB);
  dim3 grid((unsigned)std::min<long long>(tiles, 148 * 96), cdiv(cgs, kDwCgPerBlock));
  if (p.x.f16) {
    if (p.sW == 1) dwconv_kernel<VEC, 4, 1, KW, true><<<grid, 256, smem, s>>>(p, res_vec);
    else dwconv_kernel<VEC, 2, 2, KW, true><<<grid, 256, smem, s>>>(p, res_vec);
  } else {
    if (p.sW == 1) dwconv_kernel<VEC, 4, 1, KW, false><<<grid, 256, smem, s>>>(p, res_vec);
    else dwconv_kernel<VEC, 2, 2, KW, false><<<grid, 256, smem, s>>>(p, res_vec);
  }
  return true;
}
template <int KW>
static bool dispatch_dwconv(const DirectParams& p, cudaStream_t s) {
  const int C = p.x.C;
  if (C % 8 == 0 && vec_ok(p.x, 8) && vec_ok(p.y, 8)) return launch_dwconv<8, KW>(p, s);
  if (C % 4 == 0 && vec_ok(p.x, 4) && vec_ok(p.y, 4)) return launch_dwconv<4, KW>(p, s);
  if (C % 2 == 0 && vec_ok(p.x, 2) && vec_ok(p.y, 2)) return launch_dwconv<2, KW>(p, s);
  return launch_dwconv<1, KW>(p, s);
}

static bool vec_ok(const View& v, int vec) {
  return reinterpret_cast<uintptr_t>(v.ptr) % (2 * vec) == 0 && v.sB % vec == 0 && v.sT % vec == 0 && v.sH % vec == 0 &&
         v.sW % vec == 0;
}

// ------------------------------------------------------------------------------------------- pooling
struct PoolParams {
  View x, y;
  int kT, kH, kW, sT, sH, sW, pT, pH, pW, is_avg, act;
};
// One thread = one group of up to 8 channels of one output position.  XV / YV: widest access the rows of x / y allow --
// 8 (16-byte aligned rows: a full group is one 16-byte access), 2 (4-byte aligned rows: channel pairs), 1 (scalar).
// A ragged last group (C % 8 != 0) is handled pair- / element-wise by the same thread.  The first version had only
// "C % 8 == 0, everything 16-byte aligned" and otherwise one THREAD PER ELEMENT with four divisions each: the C = 6
// stem pool and the C = 30 / 60 shortcut pools of SlowFastShuffleNet (odd channel offsets inside the concat buffer)
// ran at 0.64 / 0.38 / 0.20 ms against 0.03 / 0.04 / 0.02 ms of HBM time.
// I: index type -- unsigned 32-bit whenever the element count allows (64-bit divisions cost ~5x more instructions).
// RAGGED = false (C % 8 == 0): every group is full, the tail logic compiles away.
// elementwise maximum of two packed 16-bit pairs (FP16 or BF16 bit patterns)
__device__ __forceinline__ uint32_t hmax2_bits(uint32_t a, uint32_t b, int f16) {
  if (f16) {
    const __half2 r = __hmax2(*reinterpret_cast<const __half2*>(&a), *reinterpret_cast<const __half2*>(&b));
    return *reinterpret_cast<const uint32_t*>(&r);
  }
  const __nv_bfloat162 r = __hmax2(*reinterpret_cast<const __nv_bfloat162*>(&a), *reinterpret_cast<const __nv_bfloat162*>(&b));
  return *reinterpret_cast<const uint32_t*>(&r);
}

// Max-pool of full 16-byte channel groups, one block per OUTPUT ROW (b, to, ho): the row is decomposed once per block,
// the threads walk (wo, channel group) without divisions (cv_shift: C / 8 is a power of two), and the maximum stays in
// the 16-bit format (packed HMNMX2, exact).  The general kernel below spends ~300 instructions per 16-byte output on
// seven 32-bit divisions and nine 64-bit address computations (ncu, round 2: 64 - 74 % of the issue slots at half the HBM
// peak); this is the path of the two R50 stem pools.
__global__ void __launch_bounds__(256) pool3d_rows_kernel(const PoolParams p, int cv_shift) {
  const int row = blockIdx.x;
  const int ho = row % p.y.H, bt = row / p.y.H, to = bt % p.y.T, b = bt / p.y.T;
  const int f16 = p.x.f16;
  const int cv = 1 << cv_shift, items = p.y.W << cv_shift;
  const __nv_bfloat16* xb = reinterpret_cast<const __nv_bfloat16*>(p.x.ptr) + (long long)b * p.x.sB;
  __nv_bfloat16* yrow = reinterpret_cast<__nv_bfloat16*>(p.y.ptr) + voff(p.y, b, to, ho, 0);
  const uint32_t ninf = f16 ? 0xFC00FC00u : 0xFF80FF80u;
  for (int i = threadIdx.x; i < items; i += blockDim.x) {
    const int cg = i & (cv - 1), wo = i >> cv_shift;
    uint4 m = make_uint4(ninf, ninf, ninf, ninf);
    for (int kt = 0; kt < p.kT; ++kt) {
      const int ti = to * p.sT + kt - p.pT;
      if (ti < 0 || ti >= p.x.T) continue;
      for (int kh = 0; kh < p.kH; ++kh) {
        const int hi = ho * p.sH + kh - p.pH;
        if (hi < 0 || hi >= p.x.H) continue;
        const __nv_bfloat16* xr = xb + ti * p.x.sT + hi * p.x.sH + cg * 8;
        for (int kw = 0; kw < p.kW; ++kw) {
          const int wi = wo * p.sW + kw - p.pW;
          if (wi < 0 || wi >= p.x.W) continue;
          const uint4 u = __ldg(reinterpret_cast<const uint4*>(xr + wi * p.x.sW));
          m.x = hmax2_bits(m.x, u.x, f16), m.y = hmax2_bits(m.y, u.y, f16);
          m.z = hmax2_bits(m.z, u.z, f16), m.w = hmax2_bits(m.w, u.w, f16);
        }
      }
    }
    *reinterpret_cast<uint4*>(yrow + wo * p.y.sW + cg * 8) = m;
  }
}

template <int XV, int YV, typename I, bool RAGGED>
__global__ void __launch_bounds__(256) pool3d_kernel(const PoolParams p) {
  const int C = p.y.C, cv = (C + 7) / 8;
  const I total = (I)p.y.B * p.y.T * p.y.H * p.y.W * cv;
  const float inv = 1.f / (p.kT * p.kH * p.kW);  // AvgPool3d default count_include_pad=True
  const int f16 = p.x.f16;
  for (I idx = blockIdx.x * (I)blockDim.x + threadIdx.x; idx < total; idx += (I)gridDim.x * blockDim.x) {
    const int c = (int)(idx % cv) * 8;
    I pos = idx / cv;
    const int wo = pos % p.y.W;
    pos /= p.y.W;
    const int ho = pos % p.y.H;
    pos /= p.y.H;
    const int to = pos % p.y.T;
    const int b = pos / p.y.T;
    const int nv = RAGGED ? min(8, C - c) : 8;   // channels of this group
    if (XV == 8 && YV == 8 && !RAGGED && !p.is_avg && p.act == 0) {
      // max-pool of full 16-byte groups without leaving the 16-bit format: the maximum of FP16 / BF16 numbers is exact in
      // that format, so four packed HMNMX2 per tap replace eight conversions and eight FP32 maxima (ncu, round 2: the
      // kernel was issue-bound, 64 - 74 % of the issue slots at 0.46 - 0.52 of the HBM peak)
      uint4 m = f16 ? make_uint4(0xFC00FC00u, 0xFC00FC00u, 0xFC00FC00u, 0xFC00FC00u)
                    : make_uint4(0xFF80FF80u, 0xFF80FF80u, 0xFF80FF80u, 0xFF80FF80u);   // -inf pairs
      for (int kt = 0; kt < p.kT; ++kt) {
        const int ti = to * p.sT + kt - p.pT;
        if (ti < 0 || ti >= p.x.T) continue;
        for (int kh = 0; kh < p.kH; ++kh) {
          const int hi = ho * p.sH + kh - p.pH;
          if (hi < 0 || hi >= p.x.H) continue;
          for (int kw = 0; kw < p.kW; ++kw) {
            const int wi = wo * p.sW + kw - p.pW;
            if (wi < 0 || wi >= p.x.W) continue;
            const uint4 u = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.x.ptr) +
                                                                 voff(p.x, b, ti, hi, wi) + c));
            m.x = hmax2_bits(m.x, u.x, f16), m.y = hmax2_bits(m.y, u.y, f16);
            m.z = hmax2_bits(m.z, u.z, f16), m.w = hmax2_bits(m.w, u.w, f16);
          }
        }
      }
      *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.y.ptr) + voff(p.y, b, to, ho, wo) + c) = m;
      continue;
    }
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = p.is_avg ? 0.f : -CUDART_INF_F;
    for (int kt = 0; kt < p.kT; ++kt) {
      const int ti = to * p.sT + kt - p.pT;
      if (ti < 0 || ti >= p.x.T) continue;
      for (int kh = 0; kh < p.kH; ++kh) {
        const int hi = ho * p.sH + kh - p.pH;
        if (hi < 0 || hi >= p.x.H) continue;
        for (int kw = 0; kw < p.kW; ++kw) {
          const int wi = wo * p.sW + kw - p.pW;
          if (wi < 0 || wi >= p.x.W) continue;
          const __nv_bfloat16* xp = reinterpret_cast<const __nv_bfloat16*>(p.x.ptr) + voff(p.x, b, ti, hi, wi) + c;
          float v[8];
          if (XV == 8 && nv == 8) {
            const uint4 u = *reinterpret_cast<const uint4*>(xp);
            const uint32_t uu[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 f = unpack16x2(uu[e], f16);
              v[2 * e] = f.x, v[2 * e + 1] = f.y;
            }
          } else if (XV >= 2) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              v[2 * e] = v[2 * e + 1] = 0.f;
              if (2 * e + 1 < nv) {
                const float2 f = unpack16x2(*reinterpret_cast<const uint32_t*>(xp + 2 * e), f16);
                v[2 * e] = f.x, v[2 * e + 1] = f.y;
              } else if (2 * e < nv) {
                v[2 * e] = h162f(xp[2 * e], f16);
              }
            }
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = j < nv ? h162f(xp[j], f16) : 0.f;
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[j] = p.is_avg ? acc[j] + v[j] : fmaxf(acc[j], v[j]);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = apply_act(p.is_avg ? acc[j] * inv : acc[j], p.act);
    __nv_bfloat16* yp = reinterpret_cast<__nv_bfloat16*>(p.y.ptr) + voff(p.y, b, to, ho, wo) + c;
    const int yf16 = p.y.f16;
    if (YV == 8 && nv == 8) {
      uint4 o;
      o.x = pack16x2(acc[0], acc[1], yf16), o.y = pack16x2(acc[2], acc[3], yf16);
      o.z = pack16x2(acc[4], acc[5], yf16), o.w = pack16x2(acc[6], acc[7], yf16);
      *reinterpret_cast<uint4*>(yp) = o;
    } else if (YV >= 2) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (2 * e + 1 < nv) *reinterpret_cast<uint32_t*>(yp + 2 * e) = pack16x2(acc[2 * e], acc[2 * e + 1], yf16);
        else if (2 * e < nv) yp[2 * e] = f2h16(acc[2 * e], yf16);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (j < nv) yp[j] = f2h16(acc[j], yf16);
    }
  }
}


// ------------------------------------------------------------------------------------------- ECA fuse
constexpr int kEcaBlocksPerClip = 64;
constexpr int kEcaThreads = 256;

struct EcaParams {
  View x;  // fast pathway (B, T, H, W, C)
  View y;  // slow concat slice (B, T/alpha, H, W, C)
  int alpha;
  const float* eca_w;
  int eca_k;
  const float* bn_scale;
  const float* bn_shift;
  float* partial;  // [B][kEcaBlocksPerClip][C]
  int dense;       // x and y are dense over their positions (sH = W sW, sT = H sH): division-free position walk
};

__device__ __forceinline__ float eca_tmax(const EcaParams& p, int b, long long pos, int c) {
  // pos indexes (t', h, w) of the temporally max-pooled tensor
  const int w = pos % p.x.W;
  const long long r = pos / p.x.W;
  const int h = r % p.x.H;
  const int tp = r / p.x.H;
  float m = -CUDART_INF_F;
  for (int a = 0; a < p.alpha; ++a) m = fmaxf(m, ldbf(p.x, voff(p.x, b, tp * p.alpha + a, h, w) + c));
  return m;
}

// pass 1: deterministic per-block partial sums of max_t(x) over a position chunk, per channel
__global__ void __launch_bounds__(kEcaThreads) eca_partial_kernel(const EcaParams p) {
  extern __shared__ float red[];  // [lanes][C]
  const int C = p.x.C;
  const int b = blockIdx.y;
  const long long npos = (long long)(p.x.T / p.alpha) * p.x.H * p.x.W;
  const long long chunk = (npos + gridDim.x - 1) / gridDim.x;
  const long long p0 = blockIdx.x * chunk, p1 = min(npos, p0 + chunk);
  for (int c0 = 0; c0 < C; c0 += kEcaThreads) {  // C <= 256 in every model: a single pass
    const int cw = min(C - c0, kEcaThreads);
    const int lanes = kEcaThreads / cw;
    const int c = c0 + threadIdx.x % cw;
    const int l = threadIdx.x / cw;
    float s = 0.f;
    if (l < lanes)
      for (long long pos = p0 + l; pos < p1; pos += lanes) s += eca_tmax(p, b, pos, c);
    if (l < lanes) red[l * cw + (c - c0)] = s;
    __syncthreads();
    if (threadIdx.x < cw) {
      float t = 0.f;
      for (int i = 0; i < lanes; ++i) t += red[i * cw + threadIdx.x];
      p.partial[((long long)b * gridDim.x + blockIdx.x) * C + c0 + threadIdx.x] = t;
    }
    __syncthreads();
  }
}

// pass 2: mean -> conv1d over the channel axis (zero padded) -> sigmoid -> x * s -> BN affine -> ReLU -> store
__global__ void __launch_bounds__(kEcaThreads) eca_apply_kernel(const EcaParams p, int nblk) {
  extern __shared__ float sm[];  // mean[C], mul[C]
  const int C = p.x.C;
  float* mean = sm;
  float* mul = sm + C;
  const int b = blockIdx.y;
  const long long npos = (long long)(p.x.T / p.alpha) * p.x.H * p.x.W;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float t = 0.f;
    for (int i = 0; i < nblk; ++i) t += p.partial[((long long)b * nblk + i) * C + c];
    mean[c] = t / (float)npos;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float a = 0.f;
    const int half = (p.eca_k - 1) / 2;
    for (int j = 0; j < p.eca_k; ++j) {
      const int cc = c + j - half;
      if (cc >= 0 && cc < C) a = fmaf(__ldg(p.eca_w + j), mean[cc], a);
    }
    const float sgm = 1.f / (1.f + __expf(-a));
    mul[c] = sgm * __ldg(p.bn_scale + c);
  }
  __syncthreads();
  const long long chunk = (npos + gridDim.x - 1) / gridDim.x;
  const long long p0 = blockIdx.x * chunk, p1 = min(npos, p0 + chunk);
  const long long items = (p1 - p0) * C;
  for (long long i = threadIdx.x; i < items; i += blockDim.x) {
    const int c = i % C;
    const long long pos = p0 + i / C;
    const float v = fmaxf(fmaf(eca_tmax(p, b, pos, c), mul[c], __ldg(p.bn_shift + c)), 0.f);
    const int w = pos % p.x.W;
    const long long r = pos / p.x.W;
    const int h = r % p.x.H;
    const int tp = r / p.x.H;
    sth(p.y, voff(p.y, b, tp, h, w) + c, v);
  }
}

// 16-byte variants (C % 8 == 0, C / 8 a power of two <= 256, 16-byte addressable views): one thread = 8 channels of one
// position; consecutive threads walk the channel groups of consecutive positions, i.e. contiguous memory.
__device__ __forceinline__ void unpack8(const uint4& u, int f16, float* v) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float2 f = unpack16x2(w[e], f16);
    v[2 * e] = f.x, v[2 * e + 1] = f.y;
  }
}
__device__ __forceinline__ void eca_tmax8(const EcaParams& p, int b, int pos, int cg, float* m) {
  const int w = pos % p.x.W;
  const int r = pos / p.x.W;
  const int h = r % p.x.H;
  const int tp = r / p.x.H;
  const __nv_bfloat16* base = reinterpret_cast<const __nv_bfloat16*>(p.x.ptr) + voff(p.x, b, tp * p.alpha, h, w) + cg * 8;
#pragma unroll
  for (int j = 0; j < 8; ++j) m[j] = -CUDART_INF_F;
  for (int a = 0; a < p.alpha; ++a) {
    float v[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(base + a * p.x.sT)), p.x.f16, v);
#pragma unroll
    for (int j = 0; j < 8; ++j) m[j] = fmaxf(m[j], v[j]);
  }
}

// eca_tmax8 for views that are dense over their positions (offset = b sB + t sT + hw sW): (tp, hw) are carried
// incrementally by the caller, no divisions in the position loop
__device__ __forceinline__ void eca_tmax8_dense(const EcaParams& p, const __nv_bfloat16* xb, int tp, int hw, int cg, float* m) {
  const __nv_bfloat16* base = xb + (long long)tp * p.alpha * p.x.sT + (long long)hw * p.x.sW + cg * 8;
#pragma unroll
  for (int j = 0; j < 8; ++j) m[j] = -CUDART_INF_F;
  for (int a = 0; a < p.alpha; ++a) {
    float v[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(base + a * p.x.sT)), p.x.f16, v);
#pragma unroll
    for (int j = 0; j < 8; ++j) m[j] = fmaxf(m[j], v[j]);
  }
}

__global__ void __launch_bounds__(kEcaThreads) eca_partial_vec_kernel(const EcaParams p) {
  __shared__ float red[kEcaThreads][9];
  const int C = p.x.C, cgs = (C + 7) >> 3;          // a ragged last group reads the row padding (never summed below)
  const int b = blockIdx.y;
  const int npos = (p.x.T / p.alpha) * p.x.H * p.x.W;
  const int chunk = (npos + gridDim.x - 1) / gridDim.x;
  const int p0 = blockIdx.x * chunk, p1 = min(npos, p0 + chunk);
  const int cg = threadIdx.x % cgs;                 // a thread keeps its channel group
  const int lanes = kEcaThreads / cgs;              // threads beyond lanes * cgs idle (cgs need not divide 256)
  float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (p.dense) {
    const int HW = p.x.H * p.x.W;
    const __nv_bfloat16* xb = reinterpret_cast<const __nv_bfloat16*>(p.x.ptr) + (long long)b * p.x.sB;
    int pos = threadIdx.x / cgs < lanes ? p0 + threadIdx.x / cgs : p1;
    int tp = pos / HW, hw = pos - tp * HW;
    for (; pos < p1; pos += lanes) {
      float m[8];
      eca_tmax8_dense(p, xb, tp, hw, cg, m);
#pragma unroll
      for (int j = 0; j < 8; ++j) s[j] += m[j];
      hw += lanes;
      while (hw >= HW) hw -= HW, ++tp;
    }
  } else {
    for (int pos = threadIdx.x / cgs < lanes ? p0 + threadIdx.x / cgs : p1; pos < p1; pos += lanes) {
      float m[8];
      eca_tmax8(p, b, pos, cg, m);
#pragma unroll
      for (int j = 0; j < 8; ++j) s[j] += m[j];
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) red[threadIdx.x][j] = s[j];
  __syncthreads();
  if (threadIdx.x < C) {
    const int g = threadIdx.x >> 3, j = threadIdx.x & 7;
    float t = 0.f;
    for (int i = 0; i < lanes; ++i) t += red[i * cgs + g][j];
    p.partial[((long long)b * gridDim.x + blockIdx.x) * C + threadIdx.x] = t;
  }
}

__global__ void __launch_bounds__(kEcaThreads) eca_apply_vec_kernel(const EcaParams p, int nblk) {
  extern __shared__ float sm[];  // mean[Cp], mul[Cp], shift[Cp], Cp = C rounded up to 8 (zeros behind C)
  const int C = p.x.C, cgs = (C + 7) >> 3, Cp = cgs * 8;
  float* mean = sm;
  float* mul = sm + Cp;
  float* shift = sm + 2 * Cp;
  const int b = blockIdx.y;
  const int npos = (p.x.T / p.alpha) * p.x.H * p.x.W;
  for (int c = threadIdx.x; c < Cp; c += blockDim.x) {
    float t = 0.f;
    if (c < C)
      for (int i = 0; i < nblk; ++i) t += p.partial[((long long)b * nblk + i) * C + c];
    mean[c] = t / (float)npos;
    shift[c] = c < C ? __ldg(p.bn_shift + c) : 0.f;
    mul[c] = 0.f;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float a = 0.f;
    const int half = (p.eca_k - 1) / 2;
    for (int j = 0; j < p.eca_k; ++j) {
      const int cc = c + j - half;
      if (cc >= 0 && cc < C) a = fmaf(__ldg(p.eca_w + j), mean[cc], a);
    }
    const float sgm = 1.f / (1.f + __expf(-a));
    mul[c] = sgm * __ldg(p.bn_scale + c);
  }
  __syncthreads();
  const int chunk = (npos + gridDim.x - 1) / gridDim.x;
  const int p0 = blockIdx.x * chunk, p1 = min(npos, p0 + chunk);
  const int cg = threadIdx.x % cgs;
  const int lanes = kEcaThreads / cgs;
  const int nv = min(8, C - cg * 8);   // channels of this thread's group (< 8: ragged last group)
  float ml[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) ml[j] = mul[cg * 8 + j], sh[j] = shift[cg * 8 + j];
  const int HW = p.x.H * p.x.W;
  const __nv_bfloat16* xb = reinterpret_cast<const __nv_bfloat16*>(p.x.ptr) + (long long)b * p.x.sB;
  int pos = threadIdx.x / cgs < lanes ? p0 + threadIdx.x / cgs : p1;
  int tpd = pos / HW, hwd = pos - tpd * HW;       // carried incrementally on the dense path
  for (; pos < p1; pos += lanes) {
    float m[8];
    __nv_bfloat16* yp;
    if (p.dense) {
      eca_tmax8_dense(p, xb, tpd, hwd, cg, m);
      yp = reinterpret_cast<__nv_bfloat16*>(p.y.ptr) + (long long)b * p.y.sB + (long long)tpd * p.y.sT +
           (long long)hwd * p.y.sW + cg * 8;
      hwd += lanes;
      while (hwd >= HW) hwd -= HW, ++tpd;
    } else {
      eca_tmax8(p, b, pos, cg, m);
      const int w = pos % p.x.W;
      const int r = pos / p.x.W;
      const int h = r % p.x.H;
      const int tp = r / p.x.H;
      yp = reinterpret_cast<__nv_bfloat16*>(p.y.ptr) + voff(p.y, b, tp, h, w) + cg * 8;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) m[j] = fmaxf(fmaf(m[j], ml[j], sh[j]), 0.f);
    if (nv == 8) {
      uint4 o;
      o.x = pack16x2(m[0], m[1], p.y.f16), o.y = pack16x2(m[2], m[3], p.y.f16);
      o.z = pack16x2(m[4], m[5], p.y.f16), o.w = pack16x2(m[6], m[7], p.y.f16);
      *reinterpret_cast<uint4*>(yp) = o;
    } else {   // the neighbours of the concat slice stay untouched
#pragma unroll
      for (int j = 0; j < 7; ++j)
        if (j < nv) yp[j] = f2h16(m[j], p.y.f16);
    }
  }
}

static bool dense_pos(const View& v) {
  return v.sH == (long long)v.W * v.sW && v.sT == (long long)v.H * v.sH && v.sB == (long long)v.T * v.sT;
}
static bool vec8_ok(const View& v) {
  return (reinterpret_cast<uintptr_t>(v.ptr) & 15) == 0 && v.sB % 8 == 0 && v.sT % 8 == 0 && v.sH % 8 == 0 && v.sW % 8 == 0;
}

// ------------------------------------------------------------------------------------------- global mean
// feat[b][c] = mean over (T, H, W) of x[b, :, :, :, c] for LARGE activations (the squeeze of SqueezeExcite,
// ghostnet_helper.py:46-52, runs on up to 32 x 56 x 56 positions; head_pool_kernel's one block per clip and 64
// channels ran at 47 GB/s there).  Two deterministic passes: kGmBlocks partial sums per clip, then their sum.
constexpr int kGmBlocks = 64;
template <int VEC>
__global__ void __launch_bounds__(256) global_sum_partial_kernel(const View x, int npos, float* __restrict__ partial) {
  __shared__ float red[256][VEC + 1];
  const int C = x.C, cgs = C / VEC;
  const int lanes = 256 / cgs;                 // host guarantees cgs <= 256
  const int b = blockIdx.y;
  const int chunk = (npos + gridDim.x - 1) / gridDim.x;
  const int p0 = blockIdx.x * chunk, p1 = min(npos, p0 + chunk);
  const int cg = threadIdx.x % cgs, lane = threadIdx.x / cgs;
  float s[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) s[j] = 0.f;
  if (lane < lanes) {
    const int HW = x.H * x.W;
    for (int pos = p0 + lane; pos < p1; pos += lanes) {
      const int t = pos / HW, r = pos - t * HW, h = r / x.W, w = r - h * x.W;
      const __nv_bfloat16* px = reinterpret_cast<const __nv_bfloat16*>(x.ptr) + voff(x, b, t, h, w) + cg * VEC;
      if constexpr (VEC == 8) {
        float v[8];
        unpack8(__ldg(reinterpret_cast<const uint4*>(px)), x.f16, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) s[j] += v[j];
      } else {
        s[0] += h162f(px[0], x.f16);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < VEC; ++j) red[threadIdx.x][j] = s[j];
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const int g = c / VEC, j = c - g * VEC;
    float t = 0.f;
    for (int i = 0; i < lanes; ++i) t += red[i * cgs + g][j];
    partial[((long long)b * gridDim.x + blockIdx.x) * C + c] = t;
  }
}

__global__ void __launch_bounds__(256) global_mean_finish_kernel(const float* __restrict__ partial, int nblk, int C, int npos,
                                                                 float* __restrict__ feat, int feat_stride, int feat_off) {
  const int b = blockIdx.y;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float t = 0.f;
  for (int i = 0; i < nblk; ++i) t += partial[((long long)b * nblk + i) * C + c];
  feat[(long long)b * feat_stride + feat_off + c] = t / (float)npos;
}

// ------------------------------------------------------------------------------------------- head
// 16-byte variant of head_pool_kernel: block = (clip, up to 256 channels), thread = 8 channels x a strided set of positions
// gpb: channel groups per block (a power of two <= 32) -- few-channel tensors get narrow blocks so that the grid fills
// the GPU (the fast pathway's 256 channels ran as 64 blocks: 12 % occupancy, 0.65 TB/s, 80 us)
__global__ void __launch_bounds__(256) head_pool_vec_kernel(const View x, float* feat, int feat_stride, int feat_off,
                                                            int gpb) {
  __shared__ float red[256][9];
  const int b = blockIdx.y;
  const int cgs_total = x.C >> 3;
  const int cgs = min(cgs_total - blockIdx.x * gpb, gpb);   // channel groups of this block (power of two by construction)
  const int cg = threadIdx.x % cgs, l = threadIdx.x / cgs, lanes = 256 / cgs;
  const int npos = x.T * x.H * x.W;
  float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int pos = l; pos < npos; pos += lanes) {
    const int w = pos % x.W;
    const int r = pos / x.W;
    const int h = r % x.H;
    const int t = r / x.H;
    float v[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(x.ptr) + voff(x, b, t, h, w) +
                                                 (blockIdx.x * gpb + cg) * 8)),
            x.f16, v);
#pragma unroll
    for (int j = 0; j < 8; ++j) s[j] += v[j];
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) red[threadIdx.x][j] = s[j];
  __syncthreads();
  if (threadIdx.x < cgs * 8) {
    const int g = threadIdx.x >> 3, j = threadIdx.x & 7;
    float t = 0.f;
    for (int i = 0; i < lanes; ++i) t += red[i * cgs + g][j];
    feat[(long long)b * feat_stride + feat_off + blockIdx.x * gpb * 8 + threadIdx.x] = t / (float)npos;
  }
}

// feat[b][c] = mean over (T,H,W) of x[b,:,:,:,c]; one block per (clip, 64-channel group)
__global__ void __launch_bounds__(256) head_pool_kernel(const View x, float* feat, int feat_stride, int feat_off) {
  __shared__ float red[4][64];
  const int b = blockIdx.y;
  const int c = blockIdx.x * 64 + (threadIdx.x & 63);
  const int l = threadIdx.x >> 6;
  const long long npos = (long long)x.T * x.H * x.W;
  float s = 0.f;
  if (c < x.C)
    for (long long pos = l; pos < npos; pos += 4) {
      const int w = pos % x.W;
      const long long r = pos / x.W;
      const int h = r % x.H;
      const int t = r / x.H;
      s += ldbf(x, voff(x, b, t, h, w) + c);
    }
  red[l][threadIdx.x & 63] = s;
  __syncthreads();
  if (threadIdx.x < 64 && c < x.C)
    feat[(long long)b * feat_stride + feat_off + c] =
        (red[0][threadIdx.x] + red[1][threadIdx.x] + red[2][threadIdx.x] + red[3][threadIdx.x]) / (float)npos;
}

// out[b][k] = act(sum_c feat[b][c] * w[k][c] + bias[k]); one block per clip, one warp per class (strided)
__global__ void __launch_bounds__(256) head_fc_kernel(const float* feat, int Cin, int feat_stride, const float* w,
                                                      const float* bias, int K, int act, float* out, int out_stride) {
  extern __shared__ float sm[];  // feat[Cin], logits[K]
  float* f = sm;
  float* logit = sm + Cin;
  __shared__ float red[32];
  const int b = blockIdx.x;
  for (int c = threadIdx.x; c < Cin; c += blockDim.x) f[c] = feat[(long long)b * feat_stride + c];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int k = warp; k < K; k += nw) {
    float s = 0.f;
    for (int c = lane; c < Cin; c += 32) s = fmaf(f[c], __ldg(w + (long long)k * Cin + c), s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) logit[k] = s + __ldg(bias + k);
  }
  __syncthreads();
  if (act == 1) {  // softmax over classes
    float m = -CUDART_INF_F;
    for (int k = threadIdx.x; k < K; k += blockDim.x) m = fmaxf(m, logit[k]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) red[warp] = m;
    __syncthreads();
    m = red[0];
    for (int i = 1; i < nw; ++i) m = fmaxf(m, red[i]);
    __syncthreads();
    float s = 0.f;
    for (int k = threadIdx.x; k < K; k += blockDim.x) {
      const float e = expf(logit[k] - m);
      logit[k] = e;
      s += e;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) red[warp] = s;
    __syncthreads();
    s = 0.f;
    for (int i = 0; i < nw; ++i) s += red[i];
    for (int k = threadIdx.x; k < K; k += blockDim.x) out[(long long)b * out_stride + k] = logit[k] / s;
  } else {
    for (int k = threadIdx.x; k < K; k += blockDim.x) {
      float v = logit[k];
      if (act == 2) v = fmaxf(v, 0.f);
      else if (act == 3) v = 1.f / (1.f + expf(-v));
      else if (act == 4) v = fminf(fmaxf(v + 3.f, 0.f), 6.f) * (1.f / 6.f);  // hard sigmoid: relu6(x + 3) / 6
      out[(long long)b * out_stride + k] = v;
    }
  }
}

// Tiled variant for batches: block = 8 classes (one per warp) x 8 clips; every weight element is loaded once per block
// and reused for the 8 clips.  Writes act(logit) for the pointwise activations, raw logits for softmax (act 1), which
// head_softmax_kernel then normalises in place.
__global__ void __launch_bounds__(256) head_fc_tiled_kernel(const float* __restrict__ feat, int B, int Cin, int feat_stride,
                                                            const float* __restrict__ w, const float* __restrict__ bias,
                                                            int K, int act, float* out, int out_stride) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int k = blockIdx.x * 8 + warp;
  const int b0 = blockIdx.y * 8;
  if (k >= K) return;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  const float* wr = w + (long long)k * Cin;
  for (int c = lane; c < Cin; c += 32) {
    const float wv = __ldg(wr + c);
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (b0 + i < B) acc[i] = fmaf(__ldg(feat + (long long)(b0 + i) * feat_stride + c), wv, acc[i]);
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], o);
  }
  if (lane == 0) {
    const float bk = __ldg(bias + k);
    for (int i = 0; i < 8 && b0 + i < B; ++i) {
      float v = acc[i] + bk;
      if (act == 2) v = fmaxf(v, 0.f);
      else if (act == 3) v = 1.f / (1.f + expf(-v));
      else if (act == 4) v = fminf(fmaxf(v + 3.f, 0.f), 6.f) * (1.f / 6.f);
      out[(long long)(b0 + i) * out_stride + k] = v;
    }
  }
}

__global__ void __launch_bounds__(256) head_softmax_kernel(float* out, int K, int out_stride) {
  __shared__ float red[8];
  float* row = out + (long long)blockIdx.x * out_stride;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float m = -CUDART_INF_F;
  for (int k = threadIdx.x; k < K; k += 256) m = fmaxf(m, row[k]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (lane == 0) red[warp] = m;
  __syncthreads();
  m = red[0];
  for (int i = 1; i < 8; ++i) m = fmaxf(m, red[i]);
  __syncthreads();
  float s = 0.f;
  for (int k = threadIdx.x; k < K; k += 256) {
    const float e = expf(row[k] - m);
    row[k] = e;
    s += e;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) red[warp] = s;
  __syncthreads();
  s = 0.f;
  for (int i = 0; i < 8; ++i) s += red[i];
  for (int k = threadIdx.x; k < K; k += 256) row[k] = row[k] / s;
}

// ------------------------------------------------------------------------------------------- channel plumbing
// dst = channel_shuffle(cat(a, b), groups): input channel c = i * (C / groups) + j lands at j * groups + i
// (shufflenetv2_helper.py:32-43 / shufflenet_helper.py:24-34); b may be empty (cb == 0).
__global__ void __launch_bounds__(256) shuffle_concat_kernel(const View a, const View b, int cb, int groups, const View y) {
  const int C = y.C;
  const int cpg = C / groups;
  const long long total = (long long)y.B * y.T * y.H * y.W * C;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int o = idx % C;
    long long pos = idx / C;
    const int w = pos % y.W;
    pos /= y.W;
    const int h = pos % y.H;
    pos /= y.H;
    const int t = pos % y.T;
    const int bb = pos / y.T;
    const int c = (o % groups) * cpg + o / groups;  // source channel in cat(a, b)
    const __nv_bfloat16 v = c < a.C ? reinterpret_cast<const __nv_bfloat16*>(a.ptr)[voff(a, bb, t, h, w) + c]
                                    : reinterpret_cast<const __nv_bfloat16*>(b.ptr)[voff(b, bb, t, h, w) + (c - a.C)];
    reinterpret_cast<__nv_bfloat16*>(y.ptr)[voff(y, bb, t, h, w) + o] = v;
  }
}
// Same permutation, one thread = VEC consecutive OUTPUT channels: VEC gathered 2-byte loads (the row is L1 resident,
// a warp covers it completely) and one VEC*2-byte store.
template <int VEC>
__global__ void __launch_bounds__(256) shuffle_concat_vec_kernel(const View a, const View b, int cb, int groups,
                                                                 const View y, int flat32) {
  const int C = y.C, cv = C / VEC;
  const int cpg = C / groups;
  const long long total = (long long)y.B * y.T * y.H * y.W * cv;
  const unsigned short* ap = reinterpret_cast<const unsigned short*>(a.ptr);
  const unsigned short* bp = reinterpret_cast<const unsigned short*>(b.ptr);
  // dense views (offset = position * sW) and a 32-bit item count: no (b, t, h, w) decomposition, no 64-bit divisions
  const bool flat = flat32;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    int o0;
    long long ao, bo = 0, yo;
    if (flat) {
      const unsigned i32 = (unsigned)idx, pos = i32 / (unsigned)cv;
      o0 = (int)(i32 - pos * cv) * VEC;
      ao = (long long)pos * a.sW, yo = (long long)pos * y.sW;
      if (cb) bo = (long long)pos * b.sW;
    } else {
      o0 = (idx % cv) * VEC;
      long long pos = idx / cv;
      const int w = pos % y.W;
      pos /= y.W;
      const int h = pos % y.H;
      pos /= y.H;
      const int t = pos % y.T;
      const int bb = pos / y.T;
      ao = voff(a, bb, t, h, w), yo = voff(y, bb, t, h, w);
      if (cb) bo = voff(b, bb, t, h, w);
    }
    unsigned short v[VEC];
    int q = o0 / groups, r = o0 - q * groups;     // o = q * groups + r  ->  source channel r * cpg + q of cat(a, b)
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
      const int c = r * cpg + q;
      v[e] = c < a.C ? __ldg(ap + ao + c) : __ldg(bp + bo + (c - a.C));
      if (++r == groups) r = 0, ++q;
    }
    unsigned short* yp = reinterpret_cast<unsigned short*>(y.ptr) + yo + o0;
    if constexpr (VEC == 8) {
      *reinterpret_cast<uint4*>(yp) = make_uint4(v[0] | ((uint32_t)v[1] << 16), v[2] | ((uint32_t)v[3] << 16),
                                                  v[4] | ((uint32_t)v[5] << 16), v[6] | ((uint32_t)v[7] << 16));
    } else if constexpr (VEC == 4) {
      *reinterpret_cast<uint2*>(yp) = make_uint2(v[0] | ((uint32_t)v[1] << 16), v[2] | ((uint32_t)v[3] << 16));
    } else {
      *reinterpret_cast<uint32_t*>(yp) = v[0] | ((uint32_t)v[1] << 16);
    }
  }
}
// y = act(a + b) elementwise
__global__ void __launch_bounds__(256) eltwise_add_kernel(const View a, const View b, const View y, int act) {
  const int C = y.C;
  const long long total = (long long)y.B * y.T * y.H * y.W * C;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int c = idx % C;
    long long pos = idx / C;
    const int w = pos % y.W;
    pos /= y.W;
    const int h = pos % y.H;
    pos /= y.H;
    const int t = pos % y.T;
    const int bb = pos / y.T;
    const float v = ldbf(a, voff(a, bb, t, h, w) + c) + ldbf(b, voff(b, bb, t, h, w) + c);
    sth(y, voff(y, bb, t, h, w) + c, apply_act(v, act));
  }
}
// y = x * scale[b][c]  (squeeze-excite gate, ghostnet_helper.py:46-52)
// Fast path of eltwise_add / channel_scale: 8 channels per thread (16-byte accesses), views dense over their positions
// (offset = position * sW), 32-bit index arithmetic.  OP 0: y = act(a + b); OP 1: y = a * scale[batch][c].  The scalar
// kernels around it did five 64-bit div/mod pairs per ELEMENT (~600 GB/s).
template <int OP>
__global__ void __launch_bounds__(256) eltwise_vec8_kernel(const View a, const View b, const float* __restrict__ scale,
                                                           const View y, int act, unsigned npos_clip) {
  const unsigned cv = y.C >> 3;
  const unsigned total = (unsigned)y.B * npos_clip * cv;
  for (unsigned idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const unsigned pos = idx / cv, c0 = (idx - pos * cv) << 3;
    float va[8], vb[8];
    load_vec<8>(reinterpret_cast<const __nv_bfloat16*>(a.ptr) + (long long)pos * a.sW + c0, a.f16, va);
    if constexpr (OP == 0) {
      load_vec<8>(reinterpret_cast<const __nv_bfloat16*>(b.ptr) + (long long)pos * b.sW + c0, b.f16, vb);
#pragma unroll
      for (int j = 0; j < 8; ++j) va[j] = apply_act(va[j] + vb[j], act);
    } else {
      const float* sc = scale + (long long)(pos / npos_clip) * y.C + c0;
      const float4 s0 = __ldg(reinterpret_cast<const float4*>(sc)), s1 = __ldg(reinterpret_cast<const float4*>(sc) + 1);
      va[0] *= s0.x, va[1] *= s0.y, va[2] *= s0.z, va[3] *= s0.w;
      va[4] *= s1.x, va[5] *= s1.y, va[6] *= s1.z, va[7] *= s1.w;
    }
    store_vec<8>(reinterpret_cast<__nv_bfloat16*>(y.ptr) + (long long)pos * y.sW + c0, y.f16, va);
  }
}

__global__ void __launch_bounds__(256) channel_scale_kernel(const View x, const float* __restrict__ scale, const View y) {
  const int C = y.C;
  const long long total = (long long)y.B * y.T * y.H * y.W * C;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int c = idx % C;
    long long pos = idx / C;
    const int w = pos % y.W;
    pos /= y.W;
    const int h = pos % y.H;
    pos /= y.H;
    const int t = pos % y.T;
    const int bb = pos / y.T;
    const float v = ldbf(x, voff(x, bb, t, h, w) + c) * __ldg(scale + (long long)bb * C + c);
    sth(y, voff(y, bb, t, h, w) + c, v);
  }
}

static int grid_for(long long total, int threads) {
  long long g = (total + threads - 1) / threads;
  const long long cap = 148LL * 32;
  return (int)std::max(1LL, std::min(g, cap));
}

}  // namespace esf

using namespace esf;

extern "C" int esf_stem_conv(const float* x, int32_t B, int32_t Cin, int32_t T, int32_t H, int32_t W, const float* w,
                             const float* bias, int32_t Cout, int32_t kT, int32_t kH, int32_t kW, int32_t sT,
                             int32_t sH, int32_t sW, int32_t pT, int32_t pH, int32_t pW, int32_t act,
                             const esf_view* y, void* stream) {
  ESF_CHECK_ARG(x && w && bias && view_ok(y), "esf_stem_conv: null/bad argument");
  StemParams p;
  p.x = x, p.B = B, p.Cin = Cin, p.T = T, p.H = H, p.W = W, p.w = w, p.bias = bias, p.Cout = Cout;
  p.kT = kT, p.kH = kH, p.kW = kW, p.sT = sT, p.sH = sH, p.sW = sW, p.pT = pT, p.pH = pH, p.pW = pW, p.act = act;
  p.To = (T + 2 * pT - kT) / sT + 1;
  p.Ho = (H + 2 * pH - kH) / sH + 1;
  p.Wo = (W + 2 * pW - kW) / sW + 1;
  p.y = to_view(y);
  p.y_f32 = y->dtype == ESF_F32;
  ESF_CHECK_ARG(y->B == B && y->T == p.To && y->H == p.Ho && y->W == p.Wo && y->C == Cout,
                "esf_stem_conv: output view (%d,%d,%d,%d,%d) != expected (%d,%d,%d,%d,%d)", y->B, y->T, y->H, y->W,
                y->C, B, p.To, p.Ho, p.Wo, Cout);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const long long pos = (long long)B * p.To * p.Ho * p.Wo;
  const bool vec8 = Cout % 8 == 0 && (reinterpret_cast<uintptr_t>(y->ptr) % 16 == 0) && y->sW % 8 == 0 &&
                    y->sH % 8 == 0 && y->sT % 8 == 0 && y->sB % 8 == 0;
  if (vec8) stem_conv_kernel<8><<<grid_for(pos * (Cout / 8), 256), 256, 0, s>>>(p);
  else stem_conv_kernel<1><<<grid_for(pos * Cout, 256), 256, 0, s>>>(p);
  return check_launch("stem_conv_kernel");
}

static int stem_pack_launch(const char* who, const float* x, int32_t B, int32_t Cin, int32_t Tsrc, int32_t H, int32_t W,
                            const int32_t* t_index, int32_t T, int32_t pitch, int32_t lpad, int32_t dtype, void* xp,
                            void* stream, int lo_part = 0) {
  ESF_CHECK_ARG(is16(dtype), "%s: dtype must be BF16 or F16", who);
  ESF_CHECK_ARG(x && xp && B > 0 && Cin > 0 && T > 0 && Tsrc > 0 && H > 0 && W > 0, "%s: null/bad argument", who);
  ESF_CHECK_ARG(pitch % 8 == 0 && pitch >= lpad + W * Cin, "%s: bad pitch %d", who, pitch);
  const long long nrows = (long long)B * T * H;
  // two buffers of clip rows [kPackRows][Cin][W] FP32 + (Cin = 3 static path) packed output rows [kPackRows][pitch] 16-bit
  const size_t tile_bytes = 2 * (size_t)kPackRows * Cin * W * sizeof(float) + (size_t)kPackRows * pitch * 2;
  if (W % 4 == 0 && reinterpret_cast<uintptr_t>(x) % 16 == 0 && tile_bytes <= 48 * 1024 &&
      nrows < (1LL << 31) - 148LL * 16 * kPackRows) {
    const unsigned g2 = (unsigned)std::max(1LL, std::min((nrows + kPackRows - 1) / kPackRows, 148LL * 16));
    if (Cin == 3)
      stem_pack_smem_kernel<3><<<g2, 256, tile_bytes, static_cast<cudaStream_t>(stream)>>>(
          x, B, Cin, T, H, W, pitch, lpad, dtype == ESF_F16, static_cast<__nv_bfloat16*>(xp), Tsrc, t_index, lo_part);
    else
      stem_pack_smem_kernel<0><<<g2, 256, tile_bytes, static_cast<cudaStream_t>(stream)>>>(
          x, B, Cin, T, H, W, pitch, lpad, dtype == ESF_F16, static_cast<__nv_bfloat16*>(xp), Tsrc, t_index, lo_part);
    return check_launch("stem_pack_smem_kernel");
  }
  const unsigned grid = (unsigned)std::max(1LL, std::min((nrows + 1) / 2, 148LL * 64));
  if (Cin == 3)
    stem_pack_kernel<3><<<grid, dim3(128, 2), 0, static_cast<cudaStream_t>(stream)>>>(
        x, B, Cin, T, H, W, pitch, lpad, dtype == ESF_F16, static_cast<__nv_bfloat16*>(xp), Tsrc, t_index, lo_part);
  else
    stem_pack_kernel<0><<<grid, dim3(128, 2), 0, static_cast<cudaStream_t>(stream)>>>(
        x, B, Cin, T, H, W, pitch, lpad, dtype == ESF_F16, static_cast<__nv_bfloat16*>(xp), Tsrc, t_index, lo_part);
  return check_launch("stem_pack_kernel");
}

extern "C" int esf_stem_pack(const float* x, int32_t B, int32_t Cin, int32_t T, int32_t H, int32_t W, int32_t pitch,
                             int32_t lpad, int32_t dtype, void* xp, void* stream) {
  return stem_pack_launch("esf_stem_pack", x, B, Cin, T, H, W, nullptr, T, pitch, lpad, dtype, xp, stream);
}

extern "C" int esf_stem_pack_lo(const float* x, int32_t B, int32_t Cin, int32_t T, int32_t H, int32_t W, int32_t pitch,
                                int32_t lpad, int32_t dtype, void* xp, void* stream) {
  return stem_pack_launch("esf_stem_pack_lo", x, B, Cin, T, H, W, nullptr, T, pitch, lpad, dtype, xp, stream, 1);
}

extern "C" int esf_stem_pack_gather(const float* x, int32_t B, int32_t Cin, int32_t Tsrc, int32_t H, int32_t W,
                                    const int32_t* t_index, int32_t T, int32_t pitch, int32_t lpad, int32_t dtype,
                                    void* xp, void* stream) {
  ESF_CHECK_ARG(t_index != nullptr, "esf_stem_pack_gather: t_index is null");
  return stem_pack_launch("esf_stem_pack_gather", x, B, Cin, Tsrc, H, W, t_index, T, pitch, lpad, dtype, xp, stream);
}

static int frames_params(FramesParams* p, const uint8_t* frames, int32_t B, int32_t Tsrc, int32_t H, int32_t W, int32_t C,
                         const int32_t* t_index, int32_t T, const int32_t* chan_src, const char* who) {
  ESF_CHECK_ARG(frames && B > 0 && Tsrc > 0 && T > 0 && H > 0 && W > 0 && C >= 1 && C <= 4, "%s: null/bad argument", who);
  ESF_CHECK_ARG(t_index || T == Tsrc, "%s: T (%d) != Tsrc (%d) needs a frame index", who, T, Tsrc);
  p->frames = frames, p->t_index = t_index;
  p->B = B, p->Tsrc = Tsrc, p->T = T, p->H = H, p->W = W, p->C = C;
  for (int c = 0; c < 4; ++c) {
    p->chan_src[c] = (chan_src && c < C) ? chan_src[c] : c;
    ESF_CHECK_ARG(c >= C || (p->chan_src[c] >= 0 && p->chan_src[c] < C), "%s: chan_src[%d] out of range", who, c);
  }
  return ESF_OK;
}

extern "C" int esf_stem_pack_u8(const uint8_t* frames, int32_t B, int32_t Tsrc, int32_t H, int32_t W, int32_t C,
                                const int32_t* t_index, int32_t T, const int32_t* chan_src, const void* lut16,
                                int32_t pitch, int32_t lpad, void* xp, void* stream) {
  FramesParams p;
  const int rc = frames_params(&p, frames, B, Tsrc, H, W, C, t_index, T, chan_src, "esf_stem_pack_u8");
  if (rc != ESF_OK) return rc;
  ESF_CHECK_ARG(lut16 && xp, "esf_stem_pack_u8: null argument");
  ESF_CHECK_ARG(pitch % 8 == 0 && lpad >= 0 && pitch >= lpad + W * C, "esf_stem_pack_u8: bad pitch %d", pitch);
  const long long total = (long long)B * T * H * (pitch / 8);
  stem_pack_u8_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      p, static_cast<const uint16_t*>(lut16), pitch, lpad, static_cast<uint16_t*>(xp), ClipFrames{});
  return check_launch("stem_pack_u8_kernel");
}

extern "C" int esf_frames_to_clip(const uint8_t* frames, int32_t B, int32_t Tsrc, int32_t H, int32_t W, int32_t C,
                                  const int32_t* t_index, int32_t T, const int32_t* chan_src, const float* lut32,
                                  float* clip, void* stream) {
  FramesParams p;
  const int rc = frames_params(&p, frames, B, Tsrc, H, W, C, t_index, T, chan_src, "esf_frames_to_clip");
  if (rc != ESF_OK) return rc;
  ESF_CHECK_ARG(lut32 && clip, "esf_frames_to_clip: null argument");
  const long long total = (long long)B * C * T * H * ((W + 3) / 4);
  frames_to_clip_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(p, lut32, clip,
                                                                                             ClipFrames{});
  return check_launch("frames_to_clip_kernel");
}

// Ring bank (N, L, H, W, C): frames_params with B = R output rows and Tsrc = L, then the range checks that make the
// device-side slot arithmetic of RingFrames safe, on the host copies of the tables the kernel reads.
static int rings_params(FramesParams* p, const char* who, const uint8_t* bank, int32_t N, int32_t L, int32_t H, int32_t W,
                        int32_t C, const int32_t* rows, const int32_t* rows_host, int32_t R, const int32_t* pos,
                        const int32_t* pos_host, int32_t T, const int32_t* chan_src) {
  ESF_CHECK_ARG(N >= 1 && R >= 1 && rows && rows_host && pos && pos_host, "%s: null/bad argument (N %d, R %d)", who, N, R);
  const int rc = frames_params(p, bank, R, L, H, W, C, pos, T, chan_src, who);
  if (rc != ESF_OK) return rc;
  for (int r = 0; r < R; ++r) {
    ESF_CHECK_ARG(rows_host[2 * r] >= 0 && rows_host[2 * r] < N, "%s: row %d: camera %d not in [0, %d)", who, r,
                  rows_host[2 * r], N);
    ESF_CHECK_ARG(rows_host[2 * r + 1] >= 0 && rows_host[2 * r + 1] < L, "%s: row %d: oldest slot %d not in [0, %d)", who,
                  r, rows_host[2 * r + 1], L);
  }
  for (int t = 0; t < T; ++t)
    ESF_CHECK_ARG(pos_host[t] >= 0 && pos_host[t] < L, "%s: pos[%d] = %d not in [0, %d)", who, t, pos_host[t], L);
  return ESF_OK;
}

extern "C" int esf_stem_pack_u8_rings(const uint8_t* bank, int32_t N, int32_t L, int32_t H, int32_t W, int32_t C,
                                      const int32_t* rows, const int32_t* rows_host, int32_t R, const int32_t* pos,
                                      const int32_t* pos_host, int32_t T, const int32_t* chan_src, const void* lut16,
                                      int32_t pitch, int32_t lpad, void* xp, void* stream) {
  FramesParams p;
  const int rc = rings_params(&p, "esf_stem_pack_u8_rings", bank, N, L, H, W, C, rows, rows_host, R, pos, pos_host, T,
                              chan_src);
  if (rc != ESF_OK) return rc;
  ESF_CHECK_ARG(pitch % 8 == 0 && lpad >= 0 && pitch >= lpad + W * C, "esf_stem_pack_u8_rings: bad pitch %d", pitch);
  ESF_CHECK_ARG(lut16 && xp, "esf_stem_pack_u8_rings: null argument");
  const long long total = (long long)R * T * H * (pitch / 8);
  stem_pack_u8_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      p, static_cast<const uint16_t*>(lut16), pitch, lpad, static_cast<uint16_t*>(xp), RingFrames{rows});
  return check_launch("stem_pack_u8_kernel (rings)");
}

extern "C" int esf_frames_to_clip_rings(const uint8_t* bank, int32_t N, int32_t L, int32_t H, int32_t W, int32_t C,
                                        const int32_t* rows, const int32_t* rows_host, int32_t R, const int32_t* pos,
                                        const int32_t* pos_host, int32_t T, const int32_t* chan_src, const float* lut32,
                                        float* clip, void* stream) {
  FramesParams p;
  const int rc = rings_params(&p, "esf_frames_to_clip_rings", bank, N, L, H, W, C, rows, rows_host, R, pos, pos_host, T,
                              chan_src);
  if (rc != ESF_OK) return rc;
  ESF_CHECK_ARG(lut32 && clip, "esf_frames_to_clip_rings: null argument");
  const long long total = (long long)R * C * T * H * ((W + 3) / 4);
  frames_to_clip_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(p, lut32, clip,
                                                                                             RingFrames{rows});
  return check_launch("frames_to_clip_kernel (rings)");
}

extern "C" int esf_row_softmax(const float* S, int64_t rows, int32_t n, int64_t s_pitch, float scale, int32_t mode,
                               int32_t dtype, void* P, int64_t p_pitch, void* stream) {
  ESF_CHECK_ARG(S && P && rows > 0 && n > 0 && s_pitch >= n && p_pitch >= n, "esf_row_softmax: null/bad argument");
  ESF_CHECK_ARG(is16(dtype) && (mode == 0 || mode == 1), "esf_row_softmax: bad dtype / mode");
  const long long blocks = (rows + 7) / 8;
  row_softmax_kernel<<<(unsigned)std::min(blocks, 148LL * 64), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      S, rows, n, s_pitch, scale, mode, dtype == ESF_F16, static_cast<__nv_bfloat16*>(P), p_pitch);
  return check_launch("row_softmax_kernel");
}

extern "C" int esf_transpose16(const void* in, int32_t B, int32_t rows, int32_t cols, int64_t in_bstride, int64_t in_pitch,
                               void* out, int64_t out_bstride, int64_t out_pitch, void* stream) {
  ESF_CHECK_ARG(in && out && B > 0 && rows > 0 && cols > 0 && in_pitch >= cols && out_pitch >= rows && B <= 65535,
                "esf_transpose16: null/bad argument");
  dim3 grid((cols + 31) / 32, (rows + 31) / 32, B);
  ESF_CHECK_ARG(grid.y <= 65535, "esf_transpose16: too many rows");
  transpose16_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint16_t*>(in), rows, cols, in_bstride, in_pitch, static_cast<uint16_t*>(out), out_bstride,
      out_pitch);
  return check_launch("transpose16_kernel");
}

extern "C" int esf_group_mean(const float* in, int32_t B, int32_t P, int32_t K, float* out, void* stream) {
  ESF_CHECK_ARG(in && out && B > 0 && P > 0 && K > 0 && (long long)B * K < (1LL << 31), "esf_group_mean: null/bad argument");
  group_mean_kernel<<<grid_for((long long)B * K, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(in, B, P, K, out);
  return check_launch("group_mean_kernel");
}

extern "C" int64_t esf_global_mean_scratch_floats(int32_t B, int32_t C) { return (int64_t)B * kGmBlocks * C; }

extern "C" int esf_global_mean(const esf_view* x, float* scratch, float* feat, int32_t feat_stride, int32_t feat_off,
                               void* stream) {
  ESF_CHECK_ARG(view_ok(x) && scratch && feat && feat_stride >= feat_off + x->C, "esf_global_mean: null/bad argument");
  const long long npos = (long long)x->T * x->H * x->W;
  ESF_CHECK_ARG(npos < (1LL << 31), "esf_global_mean: too many positions");
  const View v = to_view(x);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int nblk = (int)std::max(1LL, std::min<long long>(kGmBlocks, npos / 64));
  dim3 grid(nblk, x->B);
  if (x->C % 8 == 0 && x->C / 8 <= 256 && vec8_ok(v)) global_sum_partial_kernel<8><<<grid, 256, 0, s>>>(v, (int)npos, scratch);
  else {
    ESF_CHECK_ARG(x->C <= 256, "esf_global_mean: %d channels need 16-byte addressable rows", x->C);
    global_sum_partial_kernel<1><<<grid, 256, 0, s>>>(v, (int)npos, scratch);
  }
  int rc = check_launch("global_sum_partial_kernel");
  if (rc != ESF_OK) return rc;
  global_mean_finish_kernel<<<dim3(cdiv(x->C, 256), x->B), 256, 0, s>>>(scratch, nblk, x->C, (int)npos, feat, feat_stride,
                                                                       feat_off);
  return check_launch("global_mean_finish_kernel");
}

// Depthwise conv over rows whose channel count was padded to a multiple of 8 by the allocator (engine.Plan.act): the
// kernel runs on c_pad channels with 16-byte vectors (C = 18 -> 24, 162 -> 168 ...), the padding channels get zero
// weights; what lands in the padding of y is never read as data.  The caller vouches that channels [C, c_pad) of x, y
// and res are padding owned by the same allocation.
extern "C" int esf_dwconv_padded(const esf_conv_desc* d, int32_t c_pad, void* stream) {
  ESF_CHECK_ARG(d && view_ok(&d->x) && view_ok(&d->y) && d->w && d->bias, "esf_dwconv_padded: null/bad argument");
  const int C = d->x.C;
  ESF_CHECK_ARG(d->groups == C && d->y.C == C && c_pad % 8 == 0 && c_pad >= C && c_pad < C + 8 && d->x.sW >= c_pad &&
                    d->y.sW >= c_pad && (!d->res.ptr || (d->res.C == C && d->res.sW >= c_pad)),
                "esf_dwconv_padded: not a depthwise conv over rows padded to %d channels", c_pad);
  ESF_CHECK_ARG((d->kW == 3 || d->kW == 5) && d->dT == 1 && d->dH == 1 && d->dW == 1 && (d->sW == 1 || d->sW == 2) &&
                    is16(d->x.dtype) && d->y.dtype == d->x.dtype && d->out_dtype == d->x.dtype &&
                    (!d->res.ptr || d->res.dtype == d->x.dtype),
                "esf_dwconv_padded: unsupported geometry / dtype");
  DirectParams p;
  p.x = to_view(&d->x), p.y = to_view(&d->y);
  p.has_res = d->res.ptr != nullptr;
  p.res = p.has_res ? to_view(&d->res) : p.y;
  p.x.C = p.y.C = p.res.C = c_pad;
  p.c_real = C, p.y_pad = 0;
  p.w = static_cast<const float*>(d->w), p.bias = d->bias;
  p.kT = d->kT, p.kH = d->kH, p.kW = d->kW, p.sT = d->sT, p.sH = d->sH, p.sW = d->sW;
  p.pT = d->pT, p.pH = d->pH, p.pW = d->pW, p.dT = d->dT, p.dH = d->dH, p.dW = d->dW;
  p.groups = c_pad, p.act = d->act, p.out_f32 = 0;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  ESF_CHECK_ARG(vec_ok(p.x, 8) && vec_ok(p.y, 8), "esf_dwconv_padded: rows are not 16-byte addressable");
  const bool done = d->kW == 3 ? launch_dwconv<8, 3>(p, s) : launch_dwconv<8, 5>(p, s);
  if (!done) return set_error(ESF_ERR_UNSUPPORTED, "esf_dwconv_padded: filter too large for shared memory");
  return check_launch("dwconv_kernel");
}

static int conv_direct_impl(const esf_conv_desc* d, int y_pad, void* stream);
extern "C" int esf_conv_direct(const esf_conv_desc* d, void* stream) { return conv_direct_impl(d, 0, stream); }

// Pointwise conv whose OUTPUT rows were padded to y_c_pad (a multiple of 8) channels by the allocator (engine.Plan.act):
// the tiny-channel kernel writes whole 16-byte groups including the padding (zeros).  The caller vouches that channels
// [C, y_c_pad) of y are padding owned by the same allocation; geometries the tiny-channel kernel does not take run as
// esf_conv_direct (the vouch is then simply unused).
extern "C" int esf_pointwise_padded(const esf_conv_desc* d, int32_t y_c_pad, void* stream) {
  ESF_CHECK_ARG(d && view_ok(&d->y), "esf_pointwise_padded: null/bad argument");
  ESF_CHECK_ARG(y_c_pad % 8 == 0 && y_c_pad >= d->y.C && y_c_pad < d->y.C + 8 && d->y.sW >= y_c_pad,
                "esf_pointwise_padded: y rows are not padded to %d channels", y_c_pad);
  return conv_direct_impl(d, y_c_pad, stream);
}

static int conv_direct_impl(const esf_conv_desc* d, int y_pad, void* stream) {
  ESF_CHECK_ARG(d && view_ok(&d->x) && view_ok(&d->y) && d->w && d->bias, "esf_conv_direct: null/bad argument");
  ESF_CHECK_ARG(d->groups >= 1 && d->x.C % d->groups == 0 && d->y.C % d->groups == 0,
                "esf_conv_direct: channels not divisible by groups");
  const int To = (d->x.T + 2 * d->pT - d->dT * (d->kT - 1) - 1) / d->sT + 1;
  const int Ho = (d->x.H + 2 * d->pH - d->dH * (d->kH - 1) - 1) / d->sH + 1;
  const int Wo = (d->x.W + 2 * d->pW - d->dW * (d->kW - 1) - 1) / d->sW + 1;
  ESF_CHECK_ARG(d->y.B == d->x.B && d->y.T == To && d->y.H == Ho && d->y.W == Wo,
                "esf_conv_direct: output view does not match the conv output shape");
  DirectParams p;
  p.x = to_view(&d->x), p.y = to_view(&d->y);
  p.has_res = d->res.ptr != nullptr;
  p.res = p.has_res ? to_view(&d->res) : p.y;
  p.w = static_cast<const float*>(d->w), p.bias = d->bias;
  p.kT = d->kT, p.kH = d->kH, p.kW = d->kW, p.sT = d->sT, p.sH = d->sH, p.sW = d->sW;
  p.pT = d->pT, p.pH = d->pH, p.pW = d->pW, p.dT = d->dT, p.dH = d->dH, p.dW = d->dW;
  p.groups = d->groups, p.act = d->act, p.out_f32 = d->out_dtype == ESF_F32;
  p.c_real = 0, p.y_pad = y_pad;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (p.groups == p.x.C && p.y.C == p.x.C && (d->kW == 3 || d->kW == 5) && d->dT == 1 && d->dH == 1 && d->dW == 1 &&
      (d->sW == 1 || d->sW == 2) && !p.out_f32 && is16(d->x.dtype) && d->y.dtype == d->x.dtype &&
      (!p.has_res || d->res.dtype == d->x.dtype) && (long long)p.y.T * p.y.H * p.y.W < (1LL << 31)) {
    const bool done = d->kW == 3 ? dispatch_dwconv<3>(p, s) : dispatch_dwconv<5>(p, s);
    if (done) return check_launch("dwconv_kernel");
  }
  if (p.groups == 1 && d->kT == 1 && d->kH == 1 && d->kW == 1 && d->sT == 1 && d->sH == 1 && d->sW == 1 && d->pT == 0 &&
      d->pH == 0 && d->pW == 0 && !p.out_f32 && is16(d->x.dtype) && d->y.dtype == d->x.dtype &&
      (!p.has_res || d->res.dtype == d->x.dtype) && (p.x.C < 8 || p.y.C < 8 || p.x.C * p.y.C <= 4096)) {
    const int cin = p.x.C, coutp = (p.y.C + 7) / 8 * 8;
    const size_t smem = (size_t)(cin + 1) * coutp * sizeof(float);
    if (smem <= 48 * 1024) {
      const long long total = (long long)p.y.B * p.y.T * p.y.H * p.y.W;   // one thread per position
      const int vec_out = vec_ok(p.y, 8);
      const unsigned grid = grid_for(total, 256);
      auto dense = [](const View& v) {
        return v.sH == (long long)v.W * v.sW && v.sT == (long long)v.H * v.sH && v.sB == (long long)v.T * v.sT;
      };
      const bool flat = dense(p.x) && dense(p.y) && (!p.has_res || dense(p.res)) &&
                        (long long)p.y.B * p.y.T * p.y.H * p.y.W < (1LL << 31);
      const bool i32 = total < (1LL << 32) - (148LL * 32 * 256);
#define ESF_PW(V)                                                                                         \
  if (flat && i32) pw_small_kernel<V, true, unsigned><<<grid, 256, smem, s>>>(p, vec_out);                \
  else if (i32) pw_small_kernel<V, false, unsigned><<<grid, 256, smem, s>>>(p, vec_out);                  \
  else pw_small_kernel<V, false, long long><<<grid, 256, smem, s>>>(p, vec_out);
      if (cin % 8 == 0 && vec_ok(p.x, 8)) { ESF_PW(8) }
      else if (cin % 4 == 0 && vec_ok(p.x, 4)) { ESF_PW(4) }
      else if (cin % 2 == 0 && vec_ok(p.x, 2)) { ESF_PW(2) }
      else { ESF_PW(1) }
#undef ESF_PW
      return check_launch("pw_small_kernel");
    }
  }
  const long long total = (long long)p.y.B * p.y.T * p.y.H * p.y.W * p.y.C;
  conv_direct_kernel<<<grid_for(total, 256), 256, 0, s>>>(p);
  return check_launch("conv_direct_kernel");
}

extern "C" int esf_pool3d(const esf_view* x, const esf_view* y, int32_t kT, int32_t kH, int32_t kW, int32_t sT,
                          int32_t sH, int32_t sW, int32_t pT, int32_t pH, int32_t pW, int32_t is_avg, int32_t act,
                          void* stream) {
  ESF_CHECK_ARG(view_ok(x) && view_ok(y) && x->C == y->C && x->B == y->B, "esf_pool3d: bad views");
  const int To = (x->T + 2 * pT - kT) / sT + 1, Ho = (x->H + 2 * pH - kH) / sH + 1, Wo = (x->W + 2 * pW - kW) / sW + 1;
  ESF_CHECK_ARG(y->T == To && y->H == Ho && y->W == Wo, "esf_pool3d: output view does not match the pooled shape");
  PoolParams p;
  p.x = to_view(x), p.y = to_view(y);
  p.kT = kT, p.kH = kH, p.kW = kW, p.sT = sT, p.sH = sH, p.sW = sW, p.pT = pT, p.pH = pH, p.pW = pW, p.is_avg = is_avg;
  p.act = act;
  auto width = [](const esf_view* v) {   // widest access every row of the view allows, in 16-bit elements
    const uintptr_t a = reinterpret_cast<uintptr_t>(v->ptr);
    if (a % 16 == 0 && v->sW % 8 == 0 && v->sH % 8 == 0 && v->sT % 8 == 0 && v->sB % 8 == 0) return 8;
    if (a % 4 == 0 && v->sW % 2 == 0 && v->sH % 2 == 0 && v->sT % 2 == 0 && v->sB % 2 == 0) return 2;
    return 1;
  };
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const long long pos = (long long)y->B * To * Ho * Wo;
  const long long items = pos * ((x->C + 7) / 8);
  const bool small = pos * x->C < (1LL << 31) - (148LL * 32 * 256);   // idx + grid stride stays inside 32 bits
  const unsigned grid = grid_for(items, 256);
  const int xv = width(x), yv = width(y);
  {
    const int cv = x->C / 8;
    const long long rows = (long long)y->B * To * Ho;
    if (xv == 8 && yv == 8 && x->C % 8 == 0 && (cv & (cv - 1)) == 0 && !is_avg && act == 0 &&
        rows < (1LL << 31) && x->sT < (1LL << 31) / std::max(1, x->T) && x->sB < (1LL << 40)) {
      int sh = 0;
      while ((1 << sh) < cv) ++sh;
      const int items = Wo * cv;
      const int threads = std::min(256, (items + 31) / 32 * 32);
      pool3d_rows_kernel<<<(unsigned)rows, threads, 0, s>>>(p, sh);
      return check_launch("pool3d_rows_kernel");
    }
  }
#define ESF_POOL(XV, YV)                                                          \
  do {                                                                            \
    if (x->C % 8 == 0) {                                                          \
      if (small) pool3d_kernel<XV, YV, unsigned, false><<<grid, 256, 0, s>>>(p);  \
      else pool3d_kernel<XV, YV, long long, false><<<grid, 256, 0, s>>>(p);       \
    } else {                                                                      \
      if (small) pool3d_kernel<XV, YV, unsigned, true><<<grid, 256, 0, s>>>(p);   \
      else pool3d_kernel<XV, YV, long long, true><<<grid, 256, 0, s>>>(p);        \
    }                                                                             \
  } while (0)
  if (xv == 8 && yv == 8) ESF_POOL(8, 8);
  else if (xv == 8 && yv == 2) ESF_POOL(8, 2);
  else if (xv == 8) ESF_POOL(8, 1);
  else if (xv == 2 && yv >= 2) ESF_POOL(2, 2);
  else if (xv == 2) ESF_POOL(2, 1);
  else if (yv >= 2) ESF_POOL(1, 2);
  else ESF_POOL(1, 1);
#undef ESF_POOL
  return check_launch("pool3d_kernel");
}

extern "C" int64_t esf_eca_scratch_floats(int32_t B, int32_t C) { return (int64_t)B * kEcaBlocksPerClip * C; }

extern "C" int esf_eca_fuse(const esf_view* x_fast, int32_t alpha, const float* eca_w, int32_t eca_k,
                            const float* bn_scale, const float* bn_shift, float* partial,
                            const esf_view* y_slow_slice, void* stream) {
  ESF_CHECK_ARG(view_ok(x_fast) && view_ok(y_slow_slice) && eca_w && bn_scale && bn_shift && partial,
                "esf_eca_fuse: null/bad argument");
  ESF_CHECK_ARG(alpha >= 1 && x_fast->T % alpha == 0, "esf_eca_fuse: T=%d not divisible by alpha=%d", x_fast->T, alpha);
  ESF_CHECK_ARG(y_slow_slice->B == x_fast->B && y_slow_slice->T == x_fast->T / alpha && y_slow_slice->H == x_fast->H &&
                    y_slow_slice->W == x_fast->W && y_slow_slice->C == x_fast->C,
                "esf_eca_fuse: output slice shape mismatch");
  ESF_CHECK_ARG(eca_k % 2 == 1, "esf_eca_fuse: even ECA kernel");
  EcaParams p;
  p.x = to_view(x_fast), p.y = to_view(y_slow_slice);
  p.alpha = alpha, p.eca_w = eca_w, p.eca_k = eca_k, p.bn_scale = bn_scale, p.bn_shift = bn_shift, p.partial = partial;
  p.dense = p.x.sH == (long long)p.x.W * p.x.sW && p.y.sH == (long long)p.y.W * p.y.sW;
  const long long npos = (long long)(x_fast->T / alpha) * x_fast->H * x_fast->W;
  const int nblk = (int)std::max(1LL, std::min<long long>(kEcaBlocksPerClip, npos / 32));
  dim3 grid(nblk, x_fast->B);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int cw = std::min(x_fast->C, kEcaThreads);
  // 16-byte path: any C <= 256 whose rows are 16-byte addressable and at least ceil8(C) wide (C = 60 / 120 / 240 of
  // ShuffleNet as well as the powers of two of the R50 models); the ragged last group is stored element-wise
  const int cgs = (x_fast->C + 7) / 8;
  if (cgs <= 32 && vec8_ok(p.x) && vec8_ok(p.y) && p.x.sW >= cgs * 8 && npos < (1LL << 31)) {
    eca_partial_vec_kernel<<<grid, kEcaThreads, 0, s>>>(p);
    int rc = check_launch("eca_partial_vec_kernel");
    if (rc != ESF_OK) return rc;
    eca_apply_vec_kernel<<<grid, kEcaThreads, 3 * cgs * 8 * sizeof(float), s>>>(p, nblk);
    return check_launch("eca_apply_vec_kernel");
  }
  eca_partial_kernel<<<grid, kEcaThreads, (kEcaThreads / cw) * cw * sizeof(float), s>>>(p);
  int rc = check_launch("eca_partial_kernel");
  if (rc != ESF_OK) return rc;
  eca_apply_kernel<<<grid, kEcaThreads, 2 * x_fast->C * sizeof(float), s>>>(p, nblk);
  return check_launch("eca_apply_kernel");
}

extern "C" int esf_head_pool(const esf_view* x0, const esf_view* x1, float* feat, void* stream) {
  ESF_CHECK_ARG(view_ok(x0) && feat, "esf_head_pool: null/bad argument");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int c1 = (x1 && x1->ptr) ? x1->C : 0;
  const int stride = x0->C + c1;
  auto pool_one = [&](const esf_view* x, int off) {
    const View v = to_view(x);
    const int cgs = x->C / 8;
    int gpb = 32;                                 // narrower blocks until the grid has ~4 blocks per SM
    while (gpb > 4 && (long long)cdiv(cgs, gpb) * x->B < 148 * 4) gpb >>= 1;
    const int last = cgs % gpb;                   // channel groups in the last block must divide 256 threads evenly
    if (x->C % 8 == 0 && (last & (last - 1)) == 0 && vec8_ok(v) && (long long)x->T * x->H * x->W < (1LL << 31))
      head_pool_vec_kernel<<<dim3(cdiv(cgs, gpb), x->B), 256, 0, s>>>(v, feat, stride, off, gpb);
    else
      head_pool_kernel<<<dim3(cdiv(x->C, 64), x->B), 256, 0, s>>>(v, feat, stride, off);
    return check_launch("head_pool_kernel");
  };
  int rc = pool_one(x0, 0);
  if (rc != ESF_OK || c1 == 0) return rc;
  ESF_CHECK_ARG(view_ok(x1) && x1->B == x0->B, "esf_head_pool: bad second pathway view");
  return pool_one(x1, x0->C);
}

extern "C" int esf_head_fc(const float* feat, int32_t B, int32_t Cin, int32_t feat_stride, const float* w,
                           const float* bias, int32_t num_classes, int32_t act, float* out, int32_t out_stride,
                           void* stream) {
  ESF_CHECK_ARG(feat && w && bias && out && B > 0 && Cin > 0 && num_classes > 0, "esf_head_fc: null/bad argument");
  const size_t smem = (size_t)(Cin + num_classes) * sizeof(float);
  ESF_CHECK_ARG(feat_stride >= Cin && out_stride >= num_classes, "esf_head_fc: strides smaller than the row lengths");
  if (B >= 8 || smem > 48 * 1024) {
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    head_fc_tiled_kernel<<<dim3(cdiv(num_classes, 8), cdiv(B, 8)), 256, 0, s>>>(feat, B, Cin, feat_stride, w, bias,
                                                                                 num_classes, act, out, out_stride);
    int rc = check_launch("head_fc_tiled_kernel");
    if (rc != ESF_OK || act != 1) return rc;
    head_softmax_kernel<<<B, 256, 0, s>>>(out, num_classes, out_stride);
    return check_launch("head_softmax_kernel");
  }
  head_fc_kernel<<<B, 256, smem, static_cast<cudaStream_t>(stream)>>>(feat, Cin, feat_stride, w, bias, num_classes, act,
                                                                      out, out_stride);
  return check_launch("head_fc_kernel");
}

static bool same_pos(const esf_view* a, const esf_view* b) {
  return a->B == b->B && a->T == b->T && a->H == b->H && a->W == b->W;
}

extern "C" int esf_shuffle_concat(const esf_view* a, const esf_view* b, int32_t groups, const esf_view* y, void* stream) {
  ESF_CHECK_ARG(view_ok(a) && view_ok(y) && groups >= 1, "esf_shuffle_concat: null/bad argument");
  const int cb = (b && b->ptr) ? b->C : 0;
  ESF_CHECK_ARG(same_pos(a, y) && (cb == 0 || (view_ok(b) && same_pos(b, y))) && a->C + cb == y->C && y->C % groups == 0,
                "esf_shuffle_concat: shape mismatch");
  const long long total = (long long)y->B * y->T * y->H * y->W * y->C;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const View va = to_view(a), vb = cb ? to_view(b) : to_view(a), vy = to_view(y);
  const int flat32 = dense_pos(va) && dense_pos(vb) && dense_pos(vy) && total / 2 < (1LL << 31);
  if (y->C % 8 == 0 && vec_ok(vy, 8))
    shuffle_concat_vec_kernel<8><<<grid_for(total / 8, 256), 256, 0, s>>>(va, vb, cb, groups, vy, flat32);
  else if (y->C % 4 == 0 && vec_ok(vy, 4))
    shuffle_concat_vec_kernel<4><<<grid_for(total / 4, 256), 256, 0, s>>>(va, vb, cb, groups, vy, flat32);
  else if (y->C % 2 == 0 && vec_ok(vy, 2))
    shuffle_concat_vec_kernel<2><<<grid_for(total / 2, 256), 256, 0, s>>>(va, vb, cb, groups, vy, flat32);
  else
    shuffle_concat_kernel<<<grid_for(total, 256), 256, 0, s>>>(va, vb, cb, groups, vy);
  return check_launch("shuffle_concat_kernel");
}

extern "C" int esf_eltwise_add(const esf_view* a, const esf_view* b, const esf_view* y, int32_t act, void* stream) {
  ESF_CHECK_ARG(view_ok(a) && view_ok(b) && view_ok(y) && same_pos(a, y) && same_pos(b, y) && a->C == y->C && b->C == y->C,
                "esf_eltwise_add: null/bad argument");
  const long long total = (long long)y->B * y->T * y->H * y->W * y->C;
  const View va = to_view(a), vb = to_view(b), vy = to_view(y);
  if (y->C % 8 == 0 && vec8_ok(va) && vec8_ok(vb) && vec8_ok(vy) && dense_pos(va) && dense_pos(vb) && dense_pos(vy) &&
      total / 8 < (1LL << 32) - (148LL * 32 * 256)) {
    eltwise_vec8_kernel<0><<<grid_for(total / 8, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        va, vb, nullptr, vy, act, (unsigned)(y->T * y->H * y->W));
    return check_launch("eltwise_vec8_kernel");
  }
  eltwise_add_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(va, vb, vy, act);
  return check_launch("eltwise_add_kernel");
}

extern "C" int esf_channel_scale(const esf_view* x, const float* scale, const esf_view* y, void* stream) {
  ESF_CHECK_ARG(view_ok(x) && view_ok(y) && scale && same_pos(x, y) && x->C == y->C, "esf_channel_scale: null/bad argument");
  const long long total = (long long)y->B * y->T * y->H * y->W * y->C;
  const View vx = to_view(x), vy = to_view(y);
  if (y->C % 8 == 0 && vec8_ok(vx) && vec8_ok(vy) && dense_pos(vx) && dense_pos(vy) &&
      (reinterpret_cast<uintptr_t>(scale) & 15) == 0 && total / 8 < (1LL << 32) - (148LL * 32 * 256)) {
    eltwise_vec8_kernel<1><<<grid_for(total / 8, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        vx, vx, scale, vy, 0, (unsigned)(y->T * y->H * y->W));
    return check_launch("eltwise_vec8_kernel");
  }
  channel_scale_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(vx, scale, vy);
  return check_launch("channel_scale_kernel");
}
