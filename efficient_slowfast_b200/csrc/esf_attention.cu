// Generic CUDA-core fallback of the CMDA slow->fast position attention: softmax_j(q_i . k_j) v_j over all N = T*H*W
// positions of a clip, then gamma * O + x_d, the bn_s2f affine, ReLU, the x alpha nearest temporal upsample and the
// store into the fast pathway's concat slice.
//
// Any head dim, FP32 math straight from the projection rows [x_d | q | k | v]: one warp per query, logits staged in
// shared memory.  Used only where the tcgen05 kernel (csrc/esf_attn_tc.cu) and the FP32 flash kernel
// (csrc/esf_precise.cu) do not apply: d > 128, which in the reference's models only occurs with N <= 392 keys
// (SlowFastShuffleNet s4_fuse, d = 240).  The output is 16-bit, or FP32 for the FP32-accurate plan.
#include <math_constants.h>

#include "esf_common.cuh"
#include "esf_host.h"

namespace esf {

__global__ void __launch_bounds__(128) attn_generic_kernel(const float* __restrict__ proj, int N, int T, int H, int W,
                                                           int d, float gamma, const float* __restrict__ bn_scale,
                                                           const float* __restrict__ bn_shift, int alpha, int f16,
                                                           int out_f32, void* __restrict__ y, long long ysB, long long ysT,
                                                           long long ysH, long long ysW) {
  extern __shared__ float srow[];  // [4 warps][N]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.y;
  const int i = blockIdx.x * 4 + warp;
  if (i >= N) return;
  float* s = srow + warp * N;
  const float* base = proj + (long long)b * N * 4 * d;
  const float* qi = base + (long long)i * 4 * d + d;
  float m = -CUDART_INF_F;
  for (int j = 0; j < N; ++j) {
    const float* kj = base + (long long)j * 4 * d + 2 * d;
    float acc = 0.f;
    for (int c = lane; c < d; c += 32) acc = fmaf(qi[c], kj[c], acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) s[j] = acc;
    m = fmaxf(m, acc);
  }
  __syncwarp();
  float l = 0.f;
  for (int j = 0; j < N; ++j) l += expf(s[j] - m);
  const int HW = H * W;
  const int t = i / HW, hw = i % HW, hh = hw / W, ww = hw % W;
  for (int c = lane; c < d; c += 32) {
    float o = 0.f;
    for (int j = 0; j < N; ++j) o = fmaf(expf(s[j] - m), base[(long long)j * 4 * d + 3 * d + c], o);
    const float a = fmaf(gamma, o / l, base[(long long)i * 4 * d + c]);
    const float v = fmaxf(fmaf(a, bn_scale[c], bn_shift[c]), 0.f);
    for (int r = 0; r < alpha; ++r) {
      const long long at = b * ysB + (long long)(t * alpha + r) * ysT + hh * ysH + ww * ysW + c;
      if (out_f32) static_cast<float*>(y)[at] = v;
      else static_cast<__nv_bfloat16*>(y)[at] = f2h16(v, f16);
    }
  }
}

}  // namespace esf

using namespace esf;

extern "C" int esf_attn_generic(const float* proj, int32_t B, int32_t T, int32_t H, int32_t W, int32_t d, float gamma,
                                const float* bn_scale, const float* bn_shift, int32_t alpha,
                                const esf_view* y_fast_slice, void* stream) {
  ESF_CHECK_ARG(proj && bn_scale && bn_shift && view_ok(y_fast_slice) && d > 0, "esf_attn_generic: null/bad argument");
  const esf_view* y = y_fast_slice;
  ESF_CHECK_ARG(y->B == B && y->T == T * alpha && y->H == H && y->W == W && y->C == d,
                "esf_attn_generic: output slice shape mismatch");
  const int N = T * H * W;
  const size_t smem = (size_t)4 * N * sizeof(float);
  ESF_CHECK_ARG(smem <= 160 * 1024, "esf_attn_generic: N = %d too large for the fallback kernel", N);
  static unsigned char attr_done[kMaxDevices] = {0};
  unsigned char* slot = device_slot(attr_done);
  if (!slot || !*slot) {
    ESF_CUDA(cudaFuncSetAttribute(attn_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    if (slot) *slot = 1;
  }
  attn_generic_kernel<<<dim3(cdiv(N, 4), B), 128, smem, static_cast<cudaStream_t>(stream)>>>(
      proj, N, T, H, W, d, gamma, bn_scale, bn_shift, alpha, y->dtype == ESF_F16, y->dtype == ESF_F32, y->ptr, y->sB,
      y->sT, y->sH, y->sW);
  return check_launch("attn_generic_kernel");
}
