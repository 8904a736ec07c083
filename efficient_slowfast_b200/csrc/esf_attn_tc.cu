// CMDA slow->fast position attention on the 5th-generation tensor cores (tcgen05 + TMEM), single pass, lazy rescale.
//
//   out[i] = relu(bn(gamma * sum_j softmax_j(q_i . k_j) v_j + x_i)),  N = T*H*W keys per clip, no N x N matrix.
//
// Work split: one CTA = 256 query rows of one clip (two 128-row tiles A/B that share every K/V tile), 10 warps:
//   warp 8   TMA producer (Q once, then a `stages`-deep ring of K~ / V^T tiles, 64 keys each)
//   warp 9   MMA issuer: S = Q~ K~^T (M=128, N=64) into double-buffered TMEM tiles, O += P V (M=128, N=DVp)
//   warps 0-3 / 4-7  softmax warpgroups of tile A / B, one query row per thread
// S is computed with the hi/lo split
//   s = q_hi.k_hi + q_lo.k_hi + q_hi.k_lo   (~FP32 logits out of BF16 MMAs; the logits are unscaled and reach 1e2)
// and p = exp2((s - m) log2e) is streamed as a BF16 A-operand through shared memory into the second MMA; O accumulates
// in TMEM.  The running row maximum m is only raised when a key tile exceeds it by more than 8 in the log2 domain (p
// stays <= 256, harmless in FP32 sums / BF16 P); on those rare tiles the owning warp rescales its 32 TMEM lanes of O
// (tcgen05.ld / st) inside the window where no P.V MMA of its tile is in flight.  The tensor pipe is mostly idle by
// construction: the kernel is bound by the MUFU (exp) pipe -- 16 exp/clk/SM (SURVEY.md 8d: exp roofline).
//
// Reference ops replaced: SpatialAttention.forward (wdf_attention_helper.py:33-54) + bn_s2f + ReLU + nearest x alpha
// upsample + concat (custom_video_model_builder.py:142-146).
#include <math_constants.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>

#include "esf_common.cuh"
#include "esf_host.h"

namespace esf {

constexpr int kTcThreads = 352;  // 8 softmax warps + TMA producer + 2 MMA issuers
constexpr int kTcBN = 64;          // keys per tile
constexpr int kTcMaxStages = 6;
constexpr int kTcMaxSteps = 12;
constexpr int kTcSmemLimit = 232448;
constexpr float kTcLog2e = 1.4426950408889634f;

struct __align__(64) AttnTcParams {
  CUtensorMap q_map, k_map, v_map;
  CUtensorMap vlo_map;  // split mode: V_lo^T (same shape as V^T)
  const float* x;  // [B][N][d]
  int B, N, T, H, W, d, alpha;
  float gamma;
  const float* bn_scale;
  const float* bn_shift;
  __nv_bfloat16* y;
  long long ysB, ysT, ysH, ysW;
  int DVp;       // padded value dim (MMA N of the second GEMM): 16 / 32 / 64 / 128
  int nchunks;   // 64-element (or KQ-element when KQ < 64) chunks per Q~/K~ row
  int chunk_el;  // elements per chunk: 32 or 64
  uint32_t sbo, layout_type;
  int nsteps1, nsteps2;
  uint32_t steps1[kTcMaxSteps], steps2[kTcMaxSteps];  // A offset | B offset << 16 (16-byte units, see host code)
  int stages;
  uint32_t q_tile_bytes, k_tile_bytes, v_tile_bytes;
  int f16;  // 16-bit operands (Q~, K~, V^T, P) and the output are IEEE half instead of BF16
  int out_f32;  // the output view is FP32 (FP32-accurate path, esf_precise.cu); strides stay in elements
  // split mode (v1 kernel, FP32-accurate plan): P and V are FP16 PAIRS, O += P_hi V_hi + P_lo V_hi + P_hi V_lo.  P_lo
  // lives 16 KB behind P_hi in shared memory, V_lo^T `v_half` bytes behind V^T inside a stage.
  int split;
  uint32_t v_half;
};

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ void tma_load_3d(void* smem, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::
          "r"(smem_u32(smem)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// SPLIT (compile time: the 16-bit plan's code must not carry the FP32 plan's branches): P and V as FP16 pairs
template <bool SPLIT>
__global__ void __launch_bounds__(kTcThreads, 1) attn_tc_kernel(const __grid_constant__ AttnTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* Qs = smem;                                   // 2 tiles x q_tile_bytes
  uint8_t* Ks = Qs + 2 * p.q_tile_bytes;                // stages x k_tile_bytes
  uint8_t* Vs = Ks + p.stages * p.k_tile_bytes;         // stages x v_tile_bytes
  uint8_t* Ps = Vs + p.stages * p.v_tile_bytes;         // 2 x 16 KB (split mode: 2 x (16 KB P_hi + 16 KB P_lo))
  const uint32_t p_q_bytes = SPLIT ? 32768u : 16384u;
  uint64_t* bars = reinterpret_cast<uint64_t*>(Ps + 2 * p_q_bytes);
  uint64_t* q_full = bars;                   // 1
  uint64_t* kv_full = q_full + 1;            // stages
  uint64_t* kv_empty = kv_full + kTcMaxStages;
  uint64_t* s_full = kv_empty + kTcMaxStages;  // [q][buf]
  uint64_t* s_free = s_full + 4;
  uint64_t* p_full = s_free + 4;             // [q]
  uint64_t* p_free = p_full + 2;
  uint64_t* o_full = p_free + 2;             // [q]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_full + 2);

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.y;
  const int row0 = blockIdx.x * 256;
  const int N = p.N;
  const int nt = (N + kTcBN - 1) / kTcBN;

  if (threadIdx.x == 0) {
    mbar_init(q_full, 1);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&kv_full[s], 1);
      mbar_init(&kv_empty[s], 2);  // one tcgen05.commit from each of the two MMA warps
    }
    for (int i = 0; i < 4; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&s_free[i], 4);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&p_full[i], 4);
      mbar_init(&p_free[i], 1);
      mbar_init(&o_full[i], 1);
    }
    fence_barrier_init();
  }
  if (warp == 8 && lane == 0) {
    prefetch_tmap(&p.q_map);
    prefetch_tmap(&p.k_map);
    prefetch_tmap(&p.v_map);
    if (SPLIT) prefetch_tmap(&p.vlo_map);
  }
  if (warp == 9) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t chunk_bytes_q = 128 * p.chunk_el * 2;  // one chunk of a 128-row Q tile
  const uint32_t chunk_bytes_k = kTcBN * p.chunk_el * 2;

  if (warp == 8) {
    // ------------------------------------------------------------------ TMA producer (all lanes loop, one issues)
    if (elect_one()) {
      mbar_arrive_expect_tx(q_full, 2 * p.q_tile_bytes);
      for (int q = 0; q < 2; ++q)
        for (int ch = 0; ch < p.nchunks; ++ch)
          tma_load_3d(Qs + q * p.q_tile_bytes + ch * chunk_bytes_q, &p.q_map, q_full, ch * p.chunk_el, row0 + q * 128, b);
    }
    __syncwarp();
    int stage = 0;
    uint32_t phase = 0;
    for (int j = 0; j < nt; ++j) {
      mbar_wait(&kv_empty[stage], phase ^ 1, 11);
      if (elect_one()) {
        mbar_arrive_expect_tx(&kv_full[stage], p.k_tile_bytes + p.v_tile_bytes);
        for (int ch = 0; ch < p.nchunks; ++ch)
          tma_load_3d(Ks + stage * p.k_tile_bytes + ch * chunk_bytes_k, &p.k_map, &kv_full[stage], ch * p.chunk_el,
                      j * kTcBN, b);
        tma_load_3d(Vs + stage * p.v_tile_bytes, &p.v_map, &kv_full[stage], j * kTcBN, 0, b);
        if (SPLIT) tma_load_3d(Vs + stage * p.v_tile_bytes + p.v_half, &p.vlo_map, &kv_full[stage], j * kTcBN, 0, b);
      }
      __syncwarp();
      if (++stage == p.stages) {
        stage = 0;
        phase ^= 1;
      }
    }
  } else if (warp == 9 || warp == 10) {
    // ------------------------------------------------------------------ MMA issuers: warp 9 -> tile A, warp 10 -> B
    // One thread issues; the whole warp runs the (warp-uniform) control flow so that descriptors stay in uniform
    // registers.  Two issuing warps because at N = 64 an MMA retires in 32 clk -- faster than one thread can issue.
    const int q = warp - 9;
    const uint32_t idesc_s = make_idesc_16(128, kTcBN, p.f16);
    const uint32_t idesc_o = make_idesc_16(128, p.DVp, p.f16);
    const uint32_t qk_hi = kmajor_desc_hi(p.sbo, p.layout_type);
    const uint32_t pv_hi = kmajor_desc_hi(1024, 2);
    const uint32_t q_lo = kmajor_desc_lo(smem_u32(Qs) + q * p.q_tile_bytes);
    const uint32_t k_lo = kmajor_desc_lo(smem_u32(Ks));
    const uint32_t v_lo = kmajor_desc_lo(smem_u32(Vs));
    const uint32_t p_lo = kmajor_desc_lo(smem_u32(Ps) + q * p_q_bytes);
    const uint32_t k_stage_step = p.k_tile_bytes >> 4, v_stage_step = p.v_tile_bytes >> 4;
    const uint32_t o_tmem = tmem_base + 4 * kTcBN + q * p.DVp;
    auto issue_s = [&](int c, int stage) {
      const int buf = c & 1;  // S tile number c lives in TMEM buffer c & 1
      mbar_wait(&s_free[q * 2 + buf], ((c >> 1) & 1) ^ 1, 12);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t d_tmem = tmem_base + (q * 2 + buf) * kTcBN;
        const uint32_t kb = k_lo + stage * k_stage_step;
#pragma unroll
        for (int i = 0; i < kTcMaxSteps; ++i)
          if (i < p.nsteps2)
            umma_bf16_lohi(d_tmem, q_lo + (p.steps2[i] & 0xffff), qk_hi, kb + (p.steps2[i] >> 16), qk_hi, idesc_s, i != 0);
        umma_commit(&s_full[q * 2 + buf]);
      }
      __syncwarp();
    };
    mbar_wait(q_full, 0, 13);
    tc_fence_after();
    // S runs one key tile ahead of P.V
    int s_stage = 0;  // stage of S tile j + 1
    uint32_t s_phase = 0;
    mbar_wait(&kv_full[s_stage], s_phase, 15);
    tc_fence_after();
    issue_s(0, s_stage);
    for (int j = 0; j < nt; ++j) {
      const int pv_stage = s_stage;
      if (++s_stage == p.stages) {
        s_stage = 0;
        s_phase ^= 1;
      }
      if (j + 1 < nt) {
        mbar_wait(&kv_full[s_stage], s_phase, 16);
        tc_fence_after();
        issue_s(j + 1, s_stage);
      }
      mbar_wait(&p_full[q], j & 1, 17);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t vl = v_lo + pv_stage * v_stage_step;
        umma_bf16_lohi(o_tmem, p_lo, pv_hi, vl, pv_hi, idesc_o, j != 0);
        umma_bf16_lohi(o_tmem, p_lo + 2, pv_hi, vl + 2, pv_hi, idesc_o, 1);
        umma_bf16_lohi(o_tmem, p_lo + 4, pv_hi, vl + 4, pv_hi, idesc_o, 1);
        umma_bf16_lohi(o_tmem, p_lo + 6, pv_hi, vl + 6, pv_hi, idesc_o, 1);
        if (SPLIT) {
          // the two correction products (2^-11 of the main one) go to an accumulator of their own, O2 = O + 2 DVp
          // columns: added to O they would only triple the number of roundings of the big accumulator
          const uint32_t pl2 = p_lo + (16384u >> 4), vl2 = vl + (p.v_half >> 4), o2 = o_tmem + 2 * p.DVp;
#pragma unroll
          for (int k = 0; k < 8; k += 2) umma_bf16_lohi(o2, pl2 + k, pv_hi, vl + k, pv_hi, idesc_o, (j != 0) || (k != 0));  // P_lo V_hi
#pragma unroll
          for (int k = 0; k < 8; k += 2) umma_bf16_lohi(o2, p_lo + k, pv_hi, vl2 + k, pv_hi, idesc_o, 1);                  // P_hi V_lo
        }
        umma_commit(&p_free[q]);
        umma_commit(&kv_empty[pv_stage]);
        if (j == nt - 1) umma_commit(&o_full[q]);
      }
      __syncwarp();
    }
  } else {
    // ------------------------------------------------------------------ softmax warpgroups
    const int q = warp >> 2;
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;  // row inside the 128-row tile
    const int n = row0 + q * 128 + r;   // query position
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
    const bool tail = (N % kTcBN) != 0;
    float m = -CUDART_INF_F;   // running row maximum (raised lazily), natural-log units
    float l = 0.f;             // running sum of p
    uint8_t* prow = Ps + q * p_q_bytes;
    const uint32_t o_addr = lane_addr + 4 * kTcBN + q * p.DVp;
    constexpr float kTau = 5.545177f;  // 8 * ln 2: p = exp(s - m) never exceeds 256
    for (int j = 0; j < nt; ++j) {
      const int buf = j & 1;
      mbar_wait(&s_full[q * 2 + buf], (j >> 1) & 1, 19);
      tc_fence_after();
      float v[64];
      tmem_ld32(lane_addr + (q * 2 + buf) * kTcBN, v);
      tmem_ld32(lane_addr + (q * 2 + buf) * kTcBN + 32, v + 32);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_free[q * 2 + buf]);
      if (tail && j == nt - 1) {
#pragma unroll
        for (int i = 0; i < 64; ++i)
          if (j * kTcBN + i >= N) v[i] = -CUDART_INF_F;
      }
      float mx0 = v[0], mx1 = v[1];
#pragma unroll
      for (int i = 2; i < 64; i += 2) {
        mx0 = fmaxf(mx0, v[i]);
        mx1 = fmaxf(mx1, v[i + 1]);
      }
      const float mx = fmaxf(mx0, mx1);
      const bool raise = mx > m + kTau;  // always true for the first tile (m = -inf)
      const float m_new = raise ? mx : m;
      const float f = raise ? fast_exp2((m - m_new) * kTcLog2e) : 1.f;  // first tile: exp2(-inf) = 0
      m = m_new;
      const float ms = m * kTcLog2e;
#pragma unroll
      for (int i = 0; i < 64; ++i) v[i] = fast_exp2(fmaf(v[i], kTcLog2e, -ms));
      float s0 = 0.f, s1 = 0.f;
#pragma unroll
      for (int i = 0; i < 64; i += 2) {
        s0 += v[i];
        s1 += v[i + 1];
      }
      l = fmaf(l, f, s0 + s1);
      mbar_wait(&p_free[q], (j & 1) ^ 1, 20);  // P.V of the previous key tile is complete: P buffer and O are quiescent
      if (j > 0 && __any_sync(0xffffffffu, raise)) {
        // rare: some row of this warp raised its maximum -> rescale this warp's 32 TMEM lanes of O
        tc_fence_after();
        for (int part = 0; part < (SPLIT ? 2 : 1); ++part)
          for (int c0 = 0; c0 < p.DVp; c0 += 16) {
            float o[16];
            tmem_ld16(o_addr + part * 2 * p.DVp + c0, o);
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) o[jj] *= f;
            tmem_st16(o_addr + part * 2 * p.DVp + c0, o);
          }
        tmem_wait_st();
      }
#pragma unroll
      for (int ck = 0; ck < 8; ++ck) {
        uint4 o;
        o.x = pack16x2(v[8 * ck + 0], v[8 * ck + 1], p.f16);
        o.y = pack16x2(v[8 * ck + 2], v[8 * ck + 3], p.f16);
        o.z = pack16x2(v[8 * ck + 4], v[8 * ck + 5], p.f16);
        o.w = pack16x2(v[8 * ck + 6], v[8 * ck + 7], p.f16);
        *reinterpret_cast<uint4*>(prow + swz(r * 128 + ck * 16, 7)) = o;
        if (SPLIT) {   // P_lo = fp16(p - P_hi): the pair carries p to 2^-22
          const uint32_t hh[4] = {o.x, o.y, o.z, o.w};
          uint32_t ll[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 h2 = unpack16x2(hh[e], p.f16);
            ll[e] = pack16x2(v[8 * ck + 2 * e] - h2.x, v[8 * ck + 2 * e + 1] - h2.y, p.f16);
          }
          *reinterpret_cast<uint4*>(prow + 16384 + swz(r * 128 + ck * 16, 7)) = make_uint4(ll[0], ll[1], ll[2], ll[3]);
        }
      }
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[q]);
    }
    // epilogue: O / l, gamma * O + x, BN, ReLU, x alpha temporal replication
    mbar_wait(&o_full[q], 0, 21);
    tc_fence_after();
    const float inv = 1.f / l;
    const int HW = p.H * p.W;
    const bool valid = n < N;
    const int t = valid ? n / HW : 0, hw = valid ? n % HW : 0, hh = hw / p.W, ww = hw % p.W;
    __nv_bfloat16* yb = p.y + b * p.ysB + hh * p.ysH + ww * p.ysW;
    const float* xr = p.x + ((long long)b * N + (valid ? n : 0)) * p.d;
    const bool vec_ok = (p.d % 8 == 0) && ((reinterpret_cast<uintptr_t>(p.y) & 15) == 0) && (p.ysW % 8 == 0) &&
                        (p.ysH % 8 == 0) && (p.ysT % 8 == 0) && (p.ysB % 8 == 0);
    for (int c0 = 0; c0 < p.DVp; c0 += 16) {
      float o[16];
      tmem_ld16(lane_addr + 4 * kTcBN + q * p.DVp + c0, o);
      if (SPLIT) {
        float o2[16];
        tmem_ld16(lane_addr + 4 * kTcBN + 2 * p.DVp + q * p.DVp + c0, o2);
#pragma unroll
        for (int jj = 0; jj < 16; ++jj) o[jj] += o2[jj];
      }
      if (!valid) continue;
#pragma unroll
      for (int jj = 0; jj < 16; ++jj) {
        const int ch = c0 + jj;
        if (ch < p.d) {
          const float a = fmaf(p.gamma, o[jj] * inv, xr[ch]);
          o[jj] = fmaxf(fmaf(a, __ldg(p.bn_scale + ch), __ldg(p.bn_shift + ch)), 0.f);
        }
      }
      if (p.out_f32) {
        for (int rep = 0; rep < p.alpha; ++rep) {
          float* yf = reinterpret_cast<float*>(p.y) + b * p.ysB + hh * p.ysH + ww * p.ysW +
                      (long long)(t * p.alpha + rep) * p.ysT + c0;
#pragma unroll
          for (int jj = 0; jj < 16; ++jj)
            if (c0 + jj < p.d) yf[jj] = o[jj];
        }
        continue;
      }
      for (int rep = 0; rep < p.alpha; ++rep) {
        __nv_bfloat16* yp = yb + (long long)(t * p.alpha + rep) * p.ysT + c0;
        if (vec_ok) {
#pragma unroll
          for (int h8 = 0; h8 < 2; ++h8) {
            if (c0 + h8 * 8 < p.d) {
              uint4 pk;
              pk.x = pack16x2(o[h8 * 8 + 0], o[h8 * 8 + 1], p.f16);
              pk.y = pack16x2(o[h8 * 8 + 2], o[h8 * 8 + 3], p.f16);
              pk.z = pack16x2(o[h8 * 8 + 4], o[h8 * 8 + 5], p.f16);
              pk.w = pack16x2(o[h8 * 8 + 6], o[h8 * 8 + 7], p.f16);
              *reinterpret_cast<uint4*>(yp + h8 * 8) = pk;
            }
          }
        } else {
#pragma unroll
          for (int jj = 0; jj < 16; ++jj)
            if (c0 + jj < p.d) yp[jj] = f2h16(o[jj], p.f16);
        }
      }
    }
    tc_fence_before();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ================================================================================================ v2 (d <= 32)
// Same algorithm with 16 softmax warps (4 per scheduler instead of 2 -- the v1 profile is latency bound: XU pipe 53 %,
// issue slots 39 %): every query row is handled by TWO threads, one per 32-key half of each 64-key tile.  The two
// halves are independent split-K streams with their own running maximum and their own TMEM accumulator O[q][h]; the
// row sums come out of the P.V MMA itself (V^T has a row of ones), so the hot loop is FFMA + MUFU.EX2 + 1/2 F2FP +
// 1/2 FMNMX3 per element.  The epilogue merges the halves: O = (O0 f0 + O1 f1) / (l0 f0 + l1 f1), f_h = exp(m_h - M).
//
// The loop is shaped to keep the MUFU pipe fed (the only roofline this kernel has):
//   * the exponentials of a tile are computed speculatively with the CURRENT running maximum, interleaved with the
//     tile-maximum reduction instead of after it; only when some row of the warp exceeds its maximum by more than tau
//     the values are rescaled by exp2(m_old - m_new) -- or, if they may have overflowed (first tile), the scores are
//     re-read from TMEM and the tile is replayed with the raised maximum;
//   * P never touches shared memory: it is written to TMEM (tcgen05.st) and the P.V MMA takes its A operand from
//     there, which removes the swizzled st.shared, the generic->async proxy fence and their address arithmetic;
// Two things that were measured and did NOT help (so the kernel is issue/latency bound, not MUFU-throughput bound):
// fetching the scores of tile j+1 before P of tile j is stored (-25 %), evaluating 1/8 .. 3/8 of the exponentials
// with a polynomial on the FMA pipe (-5 .. -25 %), and computing the tile maximum first so that the S buffer can be
// handed back to the MMA warp before the exponentials (-2 .. -4 %), and a FlashAttention-3 style ping-pong of the two
// key halves through named barriers (-2 .. -17 %: the non-MUFU phase of a tile is longer than its MUFU phase).
// What DID help after instrumenting the loop with clock64 (-DESF_ATTN_TIMING): the softmax warps found S_{j+1} missing
// on 87 % of the tiles (~200 of ~1500 cycles) because one warp issued both MMAs and could only issue S_{j+1} after it
// had waited for both halves of P_{j-1}; a Q.K^T issuer warp of its own removed that wait (-4 .. -8 %).
// The FMA-pipe exponential was repeated with packed sm_100 arithmetic (FFMA2 / FADD2.RM, 5.5 issue slots per element
// instead of ~8, on 1 .. 4 of every 8 element pairs): correct (kernel tests green at 2/8 and 4/8) but no faster --
// d = 8: 3.26 / 3.16 / 3.07 / 3.31 / 3.05 Texp/s at 0 .. 4/8, d = 32: 2.97 / 2.96 / 2.93 / 2.82 / 2.61 (8 clips,
// N = 25 088).  The scale FFMA of every pair is an FFMA2 since then; the polynomial was removed, MUFU only.
// TMEM columns: S[q][buf] 4 x 64 | O[q][h] 4 x DVp (<= 48) | P[q][h] 4 x 16  = 512.
// 16 softmax warps + TMA producer + Q.K^T issuer + 2 P.V issuers.  20 warps: ptxas sizes the register file for the
// block rounded up to 128 threads, so 21 warps would cap the softmax threads at 80 registers (spills).
constexpr int kV2Threads = 640;
constexpr int kV2PCol = 448;     // first TMEM column of P
// Tried and dropped: issue the tcgen05.st of P, fetch the next scores, and complete the hand-over (wait::st, fence,
// arrive p_full) half way through the next tile's exponentials, so that the ~200 cycles of store latency are covered
// by MUFU work.  Measured with the dedicated Q.K^T issuer in place: correct, but 12 % SLOWER (d = 8: 3.56 -> 3.12
// Texp/s, d = 32: 3.25 -> 2.88) -- the P.V MMA then finishes after the next P is ready, and the sync in the middle of
// the MUFU stream lets the pipe drain.  With a second P buffer still 9 % slower at d = 8 (2.993 -> 3.267 ms, 16 clips).
// Also tried and dropped: P aliased onto the S tile it was computed from (FlashAttention-4 style; consecutive P tiles then
// live in different TMEM buffers, the S buffer is released by the P.V commits and p_free is only consulted before an O
// rescale).  No measurable gain (d = 8: 0.812 vs 0.814 ms, d = 32: 0.863 vs 0.860 ms at 4 clips) and the interaction
// with the replay / rescale path was not yet right (one kernel test failed at 4x logits), so it is not in the tree.

// Also measured, correct and removed again (profiles/r2_attention_experiments.md):
//   * a second P buffer per (query tile, half) (d < 32: TMEM has the columns), so that the P store of tile j need not
//     wait for the P.V MMA of tile j - 1, and an independent Q.K^T issue of the two query tiles instead of lock step:
//     no change, d = 8 2.993 / 3.002 / 2.980 / 2.989 ms, d = 32 3.214 / 3.212 / 3.219 / 3.217 ms (16 clips,
//     N = 25 088; neither, P, QK, both).  The waits they remove (ncu: 4.7 % + 6 % of the softmax warps' samples) are
//     not what bounds the loop.  As run-time flags of this kernel they also cost the default path 4 - 6 % (88 instead
//     of 96 registers, d = 8: 11.04 -> 11.68 ms, d = 32: 12.23 -> 12.68 ms at batch 64).
//   * a software-pipelined softmax loop (the exponentials of tile j + 1 issued before tile j is packed, stored and
//     handed over; two tiles of values live, so the softmax warps took 112 registers from the control warps with
//     setmaxnreg): 3 % slower (d = 8: 2.832 -> 2.913 ms, d = 32: 3.112 -> 3.192 ms, 16 clips).
template <bool F16>
__global__ void __launch_bounds__(kV2Threads, 1) attn_tc_v2_kernel(const __grid_constant__ AttnTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* Qs = smem;
  uint8_t* Ks = Qs + 2 * p.q_tile_bytes;
  uint8_t* Vs = Ks + p.stages * p.k_tile_bytes;
  float* mx_sh = reinterpret_cast<float*>(Vs + p.stages * p.v_tile_bytes);  // [q][h][128] running maxima for the final merge
  uint64_t* bars = reinterpret_cast<uint64_t*>(mx_sh + 2 * 2 * 128);
  uint64_t* q_full = bars;
  uint64_t* kv_full = q_full + 1;
  uint64_t* kv_empty = kv_full + kTcMaxStages;
  uint64_t* s_full = kv_empty + kTcMaxStages;  // [q][buf]
  uint64_t* s_free = s_full + 4;
  uint64_t* p_full = s_free + 4;               // [q][h] (8 slots, 4 used)
  uint64_t* p_free = p_full + 8;
  uint64_t* o_full = p_free + 8;               // [q]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_full + 2);

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.y;
  const int row0 = blockIdx.x * 256;
  const int N = p.N;
  const int nt = (N + kTcBN - 1) / kTcBN;

  if (threadIdx.x == 0) {
    mbar_init(q_full, 1);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&kv_full[s], 1);
      mbar_init(&kv_empty[s], 2);
    }
    for (int i = 0; i < 4; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&s_free[i], 8);   // 8 softmax warps read every S tile
    }
    for (int i = 0; i < 8; ++i) {
      mbar_init(&p_full[i], 4);
      mbar_init(&p_free[i], 1);
    }
    mbar_init(&o_full[0], 1);
    mbar_init(&o_full[1], 1);
    fence_barrier_init();
  }
  if (warp == 16 && lane == 0) {
    prefetch_tmap(&p.q_map);
    prefetch_tmap(&p.k_map);
    prefetch_tmap(&p.v_map);
  }
  if (warp == 17) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 16) {
    // ------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      mbar_arrive_expect_tx(q_full, 2 * p.q_tile_bytes);
      for (int q = 0; q < 2; ++q) tma_load_3d(Qs + q * p.q_tile_bytes, &p.q_map, q_full, 0, row0 + q * 128, b);
    }
    __syncwarp();
    int stage = 0;
    uint32_t phase = 0;
    for (int j = 0; j < nt; ++j) {
      mbar_wait(&kv_empty[stage], phase ^ 1, 31);
      if (elect_one()) {
        mbar_arrive_expect_tx(&kv_full[stage], p.k_tile_bytes + p.v_tile_bytes);
        tma_load_3d(Ks + stage * p.k_tile_bytes, &p.k_map, &kv_full[stage], 0, j * kTcBN, b);
        tma_load_3d(Vs + stage * p.v_tile_bytes, &p.v_map, &kv_full[stage], j * kTcBN, 0, b);
      }
      __syncwarp();
      if (++stage == p.stages) {
        stage = 0;
        phase ^= 1;
      }
    }
  } else if (warp == 17) {
    // ------------------------------------------------------------------ Q.K^T issuer (both query tiles)
    // Separate from the P.V issuers: with one warp doing both, S_{j+1} could only be issued after that warp had waited
    // for BOTH halves of P_{j-1}, and the softmax warps found it missing on 87 % of the tiles (~200 cycles each).
    // Truncating the step list (timing only) showed five of the six d = 32 MMAs per tile cost 6.8 % of the launch.
    const uint32_t idesc_s = make_idesc_16(128, kTcBN, F16);
    const uint32_t qk_hi = kmajor_desc_hi(p.sbo, p.layout_type);
    const uint32_t q_lo0 = kmajor_desc_lo(smem_u32(Qs));
    const uint32_t q_step = p.q_tile_bytes >> 4;
    const uint32_t k_lo = kmajor_desc_lo(smem_u32(Ks));
    const uint32_t k_stage_step = p.k_tile_bytes >> 4;
    mbar_wait(q_full, 0, 33);
    tc_fence_after();
    // round 1's loop, verbatim (the two query tiles in lock step)
    int stage = 0;
    uint32_t phase = 0;
    for (int c = 0; c < nt; ++c) {
      const int buf = c & 1;
      mbar_wait(&kv_full[stage], phase, 34);
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        mbar_wait(&s_free[q * 2 + buf], ((c >> 1) & 1) ^ 1, 32);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t d_tmem = tmem_base + (q * 2 + buf) * kTcBN;
          const uint32_t kb = k_lo + stage * k_stage_step;
          const uint32_t q_lo = q_lo0 + q * q_step;
#pragma unroll
          for (int i = 0; i < 6; ++i)
            if (i < p.nsteps2)
              umma_bf16_lohi(d_tmem, q_lo + (p.steps2[i] & 0xffff), qk_hi, kb + (p.steps2[i] >> 16), qk_hi, idesc_s, i != 0);
          umma_commit(&s_full[q * 2 + buf]);
        }
        __syncwarp();
      }
      if (++stage == p.stages) {
        stage = 0;
        phase ^= 1;
      }
    }
  } else if (warp == 18 || warp == 19) {
    // ------------------------------------------------------------------ P.V issuers (one per query tile)
    const int q = warp - 18;
    const uint32_t idesc_o = make_idesc_16(128, p.DVp, F16);
    const uint32_t pv_hi = kmajor_desc_hi(1024, 2);
    const uint32_t v_lo = kmajor_desc_lo(smem_u32(Vs));
    const uint32_t v_stage_step = p.v_tile_bytes >> 4;
    int stage = 0;
    uint32_t phase = 0;
    for (int j = 0; j < nt; ++j) {
      mbar_wait(&kv_full[stage], phase, 35);   // already complete (S_j was computed from this stage): visibility only
      const uint32_t vl = v_lo + stage * v_stage_step;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        mbar_wait(&p_full[q * 2 + h], j & 1, 36);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t o_tmem = tmem_base + 4 * kTcBN + (q * 2 + h) * p.DVp;
          const uint32_t p_tmem = tmem_base + kV2PCol + (q * 2 + h) * 16;
          umma_f16_ts(o_tmem, p_tmem, vl + 4 * h, pv_hi, idesc_o, j != 0);      // keys 32h .. 32h+15
          umma_f16_ts(o_tmem, p_tmem + 8, vl + 4 * h + 2, pv_hi, idesc_o, 1);  // keys 32h+16 .. 32h+31
          umma_commit(&p_free[q * 2 + h]);
          if (h == 1) {
            umma_commit(&kv_empty[stage]);
            if (j == nt - 1) umma_commit(&o_full[q]);
          }
        }
        __syncwarp();
      }
      if (++stage == p.stages) {
        stage = 0;
        phase ^= 1;
      }
    }
  } else {
    // ------------------------------------------------------------------ softmax: warp = q * 8 + h * 4 + quarter
    const int q = warp >> 3;
    const int h = (warp >> 2) & 1;
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const int n = row0 + q * 128 + r;
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
    const uint32_t o_addr = lane_addr + 4 * kTcBN + (q * 2 + h) * p.DVp;
    const uint32_t p_addr = lane_addr + kV2PCol + (q * 2 + h) * 16;
    const bool tail = (N % kTcBN) != 0;
    float m = -CUDART_INF_F;
    // 12 * ln 2: p = exp(s - m) stays <= 4096, inside FP16 and harmless in the FP32 sums; a larger window means
    // fewer raise events and keeps small probabilities further away from the FP16 subnormals
    constexpr float kTau = 8.317766f;
    float v[32];
    mbar_wait(&s_full[q * 2], 0, 37);
    tc_fence_after();
    tmem_ld32_nowait(lane_addr + (q * 2) * kTcBN + 32 * h, v);
    tmem_wait_ld();
    tmem_ld32_acquire(v);
#ifdef ESF_ATTN_TIMING
    long long tph[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long tlast = clock64();
#define ESF_TICK(k) { const long long tn = clock64(); tph[k] += tn - tlast; tlast = tn; }
#else
#define ESF_TICK(k)
#endif
    for (int j = 0; j < nt; ++j) {
      const int buf = j & 1;
      const uint32_t s_addr = lane_addr + (q * 2 + buf) * kTcBN + 32 * h;
      const bool last_tail = tail && j == nt - 1;
      if (last_tail) {
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (j * kTcBN + 32 * h + i >= N) v[i] = -CUDART_INF_F;
      }
      // speculative pass with the current maximum; the tile maximum rides along
      float ms = (m == -CUDART_INF_F) ? 0.f : m * kTcLog2e;
      float mx0 = -CUDART_INF_F, mx1 = -CUDART_INF_F;
      ESF_TICK(0)   // tail mask + ping-pong wait
      const float2 ms2 = make_float2(-ms, -ms), c2 = make_float2(kTcLog2e, kTcLog2e);
#pragma unroll
      for (int i = 0; i < 32; i += 4) {
        mx0 = fmaxf(fmaxf(mx0, v[i]), v[i + 1]);
        mx1 = fmaxf(fmaxf(mx1, v[i + 2]), v[i + 3]);
#pragma unroll
        for (int e = 0; e < 4; e += 2) {
          float2 x = __ffma2_rn(make_float2(v[i + e], v[i + e + 1]), c2, ms2);
          x.x = fast_exp2(x.x);
          x.y = fast_exp2(x.y);
          v[i + e] = x.x;
          v[i + e + 1] = x.y;
        }
      }
      const float mx = fmaxf(mx0, mx1);
      asm volatile("" ::"f"(v[31]), "f"(mx));
      ESF_TICK(1)   // exponentials + tile maximum
      // raise lazily; a half tile that is entirely masked (tail) must not raise from -inf to -inf
      const bool raise = mx > m + kTau;
      const bool any_raise = __any_sync(0xffffffffu, raise);
      float f = 1.f;
      if (any_raise) {
        const float m_new = raise ? mx : m;
        f = raise ? fast_exp2((m - m_new) * kTcLog2e) : 1.f;  // first tile: exp2(-inf) = 0
        // exp2(x - m_new) = exp2(x - m) * f: the speculative values only need scaling, unless they may have
        // overflowed FP32 (always on the first tile, where m = -inf): then the tile is replayed from TMEM
        const bool big = raise && !((mx - m) * kTcLog2e < 100.f);
        m = m_new;
        if (__any_sync(0xffffffffu, big)) {
          tmem_ld32_nowait(s_addr, v);
          tmem_wait_ld();
          tmem_ld32_acquire(v);
          if (last_tail) {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (j * kTcBN + 32 * h + i >= N) v[i] = -CUDART_INF_F;
          }
          ms = (m == -CUDART_INF_F) ? 0.f : m * kTcLog2e;
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = fast_exp2(fmaf(v[i], kTcLog2e, -ms));
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] *= f;
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_free[q * 2 + buf]);
      ESF_TICK(2)   // raise handling + s_free arrive
      uint32_t pk[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) pk[i] = pack16x2(v[2 * i], v[2 * i + 1], F16);
      asm volatile("" ::"r"(pk[15]));
      ESF_TICK(3)   // pack
      mbar_wait(&p_free[q * 2 + h], (j & 1) ^ 1, 38);   // previous use consumed
      tc_fence_after();
      ESF_TICK(4)   // wait p_free
      if (j > 0 && any_raise) {
        // O may only be touched while no P.V MMA of this (q, h) is in flight
        for (int c0 = 0; c0 < p.DVp; c0 += 16) {
          float o[16];
          tmem_ld16(o_addr + c0, o);
#pragma unroll
          for (int jj = 0; jj < 16; ++jj) o[jj] *= f;
          tmem_st16(o_addr + c0, o);
        }
      }
      tmem_st16_b32(p_addr, pk);
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[q * 2 + h]);
      ESF_TICK(5)   // O rescale + P store + p_full arrive
      if (j + 1 < nt) {
        mbar_wait(&s_full[q * 2 + (buf ^ 1)], ((j + 1) >> 1) & 1, 37);
        tc_fence_after();
        ESF_TICK(6)   // wait s_full
        tmem_ld32_nowait(lane_addr + (q * 2 + (buf ^ 1)) * kTcBN + 32 * h, v);
        tmem_wait_ld();
        tmem_ld32_acquire(v);
        ESF_TICK(7)   // tcgen05.ld of the next scores
      }
    }
#ifdef ESF_ATTN_TIMING
    if (blockIdx.x == 3 && blockIdx.y == 0 && lane == 0)
      printf("warp %2d q%d h%d: pp-wait %lld  exp %lld  raise %lld  pack %lld  p_free %lld  Pstore %lld  s_full %lld  ld %lld  (cycles/tile, nt %d)\n",
             warp, q, h, tph[0] / nt, tph[1] / nt, tph[2] / nt, tph[3] / nt, tph[4] / nt, tph[5] / nt, tph[6] / nt, tph[7] / nt, nt);
#endif
    // ---- merge the two halves of every row and write the output
    mx_sh[(q * 2 + h) * 128 + r] = m;
    asm volatile("bar.sync %0, 256;" ::"r"(q + 1) : "memory");   // the 8 warps of this query tile
    const float m0 = mx_sh[(q * 2 + 0) * 128 + r], m1 = mx_sh[(q * 2 + 1) * 128 + r];
    const float M = fmaxf(m0, m1);
    const float f0 = (m0 == -CUDART_INF_F) ? 0.f : fast_exp2((m0 - M) * kTcLog2e);
    const float f1 = (m1 == -CUDART_INF_F) ? 0.f : fast_exp2((m1 - M) * kTcLog2e);
    mbar_wait(&o_full[q], 0, 39);
    tc_fence_after();
    const uint32_t o0 = lane_addr + 4 * kTcBN + (q * 2 + 0) * p.DVp, o1 = o0 + p.DVp;
    // row sum l = column d of both accumulators
    float t0[8], t1[8];
    const int lc = p.d & ~7;
    tmem_ld8(o0 + lc, t0);
    tmem_ld8(o1 + lc, t1);
    float l = 0.f;
#pragma unroll
    for (int jj = 0; jj < 8; ++jj)
      if (lc + jj == p.d) l = t0[jj] * f0 + t1[jj] * f1;
    const float inv = 1.f / l;
    const int HW = p.H * p.W;
    const bool valid = n < N;
    const int t = valid ? n / HW : 0, hw = valid ? n % HW : 0, hh = hw / p.W, ww = hw % p.W;
    __nv_bfloat16* yb = p.y + b * p.ysB + hh * p.ysH + ww * p.ysW;
    const float* xr = p.x + ((long long)b * N + (valid ? n : 0)) * p.d;
    const bool vec_ok = (p.d % 8 == 0) && ((reinterpret_cast<uintptr_t>(p.y) & 15) == 0) && (p.ysW % 8 == 0) &&
                        (p.ysH % 8 == 0) && (p.ysT % 8 == 0) && (p.ysB % 8 == 0);
    // half h of the row's thread pair writes the channel chunks c0 = 8 * (2 * i + h)
    for (int c0 = 8 * h; c0 < p.d; c0 += 16) {
      tmem_ld8(o0 + c0, t0);
      tmem_ld8(o1 + c0, t1);
      if (!valid) continue;
      float o[8];
#pragma unroll
      for (int jj = 0; jj < 8; ++jj) {
        const int ch = c0 + jj;
        o[jj] = 0.f;
        if (ch < p.d) {
          const float a = fmaf(p.gamma, (t0[jj] * f0 + t1[jj] * f1) * inv, xr[ch]);
          o[jj] = fmaxf(fmaf(a, __ldg(p.bn_scale + ch), __ldg(p.bn_shift + ch)), 0.f);
        }
      }
      if (p.out_f32) {
        for (int rep = 0; rep < p.alpha; ++rep) {
          float* yf = reinterpret_cast<float*>(p.y) + b * p.ysB + hh * p.ysH + ww * p.ysW +
                      (long long)(t * p.alpha + rep) * p.ysT + c0;
#pragma unroll
          for (int jj = 0; jj < 8; ++jj)
            if (c0 + jj < p.d) yf[jj] = o[jj];
        }
        continue;
      }
      for (int rep = 0; rep < p.alpha; ++rep) {
        __nv_bfloat16* yp = yb + (long long)(t * p.alpha + rep) * p.ysT + c0;
        if (vec_ok) {
          uint4 pk;
          pk.x = pack16x2(o[0], o[1], F16);
          pk.y = pack16x2(o[2], o[3], F16);
          pk.z = pack16x2(o[4], o[5], F16);
          pk.w = pack16x2(o[6], o[7], F16);
          *reinterpret_cast<uint4*>(yp) = pk;
        } else {
#pragma unroll
          for (int jj = 0; jj < 8; ++jj)
            if (c0 + jj < p.d) yp[jj] = f2h16(o[jj], F16);
        }
      }
    }
    tc_fence_before();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 17) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------ packing
struct TcGeom {
  int DVp, KQ, chunk_el, nchunks, mode;  // mode 0: d <= 8 (4 x 8 segments), 1: hi|lo halves, 2: unsplit
  int v2;                                // d <= 32: half-row kernel; V^T carries a row of ones at index d (row sums)
};
static bool tc_geom(int d, TcGeom* g) {
  if (d <= 0 || d > 128) return false;
  const int dv2 = d < 16 ? 16 : (d < 32 ? 32 : 48);   // room for the ones row
  if (d <= 8) *g = {dv2, 32, 32, 1, 0, 1};
  else if (d <= 16) *g = {dv2, 32, 32, 1, 1, 1};
  else if (d <= 32) *g = {dv2, 64, 64, 1, 1, 1};
  else if (d <= 64) *g = {64, 128, 64, 2, 1, 0};
  else *g = {128, 128, 64, 2, 2, 0};
  return true;
}
struct TcLayout {
  long long q_off, k_off, v_off, x_off, total;
  int Npad;
};
static TcLayout tc_layout(int B, int N, int d, const TcGeom& g) {
  auto al = [](long long v) { return (v + 1023) & ~1023LL; };
  TcLayout L;
  L.Npad = (N + 7) & ~7;
  const long long rows = (long long)B * N;
  L.q_off = 0;
  L.k_off = al(L.q_off + rows * g.KQ * 2);
  L.v_off = al(L.k_off + rows * g.KQ * 2);
  L.x_off = al(L.v_off + (long long)B * g.DVp * L.Npad * 2);
  L.total = al(L.x_off + rows * d * 4);
  return L;
}

// hi / lo split of an FP32 value into two 16-bit numbers of the plan's storage format: v ~= hi + lo
__device__ __forceinline__ __nv_bfloat16 h_hi(float v, int f16) { return f2h16(v, f16); }
__device__ __forceinline__ __nv_bfloat16 h_lo(float v, int f16) { return f2h16(v - h162f(f2h16(v, f16), f16), f16); }

// proj rows are [x_d | q | k | v] (d each, FP32).  One block stages R consecutive rows of one clip in shared memory
// (coalesced loads) and writes Q~/K~ rows, x_d rows and the TRANSPOSED value tile V^T[j][n0..n0+R) from there, so every
// global access is coalesced.
// Template parameters: the geometry of the head dims of the R50 / efficient models at compile time (D = 0: everything
// from the run-time arguments) -- the index arithmetic of every phase is divisions and remainders by these numbers, and
// with run-time divisors the kernel was bound by integer instructions (2.1 TB/s).
template <int D, int KQc, int DVc, int MODEc, int Rc>
__global__ void __launch_bounds__(256) attn_tc_pack_kernel(const float* __restrict__ proj, int N, int Npad, int d_rt,
                                                           int KQ_rt, int DVp_rt, int mode_rt, int R_rt, int f16,
                                                           int ones_row, __nv_bfloat16* __restrict__ Q,
                                                           __nv_bfloat16* __restrict__ K, __nv_bfloat16* __restrict__ VT,
                                                           float* __restrict__ X) {
  extern __shared__ float tile[];  // [R][4d + 1]
  const int d = D ? D : d_rt, KQ = D ? KQc : KQ_rt, DVp = D ? DVc : DVp_rt, mode = D ? MODEc : mode_rt;
  const int R = D ? Rc : R_rt;
  const int b = blockIdx.y;
  const int n0 = blockIdx.x * R;
  const int rows = min(R, N - n0);
  const int W4 = 4 * d, pitch = W4 + 1;
  const float* src = proj + ((long long)b * N + n0) * W4;
  if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {   // 16-byte loads (rows are 16 d bytes)
    for (int i = threadIdx.x; i < rows * d; i += blockDim.x) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(src) + i);
      float* t = tile + (i / d) * pitch + (i % d) * 4;
      t[0] = v.x, t[1] = v.y, t[2] = v.z, t[3] = v.w;
    }
  } else {
    for (int i = threadIdx.x; i < rows * W4; i += blockDim.x) tile[(i / W4) * pitch + (i % W4)] = src[i];
  }
  __syncthreads();
  // Q~ / K~: one thread = 8 consecutive elements of a row (one 16-byte store each)
  __nv_bfloat16* qd = Q + ((long long)b * N + n0) * KQ;
  __nv_bfloat16* kd = K + ((long long)b * N + n0) * KQ;
  auto qk_elem = [&](const float* pr, int e, __nv_bfloat16& qv, __nv_bfloat16& kv) {
    qv = f2h16(0.f, f16), kv = qv;
    if (mode == 0) {
      const int seg = e >> 3, jj = e & 7;
      if (jj < d && seg < 3) {
        const float q = pr[d + jj], k = pr[2 * d + jj];
        qv = seg == 1 ? h_lo(q, f16) : h_hi(q, f16);
        kv = seg == 2 ? h_lo(k, f16) : h_hi(k, f16);
      }
    } else if (mode == 1) {
      const int half = KQ >> 1;
      const int part = e / half, jj = e % half;
      if (jj < d) {
        const float q = pr[d + jj], k = pr[2 * d + jj];
        qv = part ? h_lo(q, f16) : h_hi(q, f16);
        kv = part ? h_lo(k, f16) : h_hi(k, f16);
      }
    } else if (e < d) {
      qv = h_hi(pr[d + e], f16);
      kv = h_hi(pr[2 * d + e], f16);
    }
  };
  auto bits = [](__nv_bfloat16 a, __nv_bfloat16 b2) {
    return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b2) << 16);
  };
  // pair (e, e + 1) of a Q~ / K~ row as one packed word each: one F2FP per hi pair, unpack + two FADD + one F2FP per lo
  // pair (the element-wise form below converts and shifts every half on its own; ncu, round 2: 61 - 74 % of the issue
  // slots busy at 2.9 - 4.5 TB/s)
  auto qk_pair = [&](const float* pr, int e, uint32_t& qw, uint32_t& kw) {
    qw = kw = 0u;
    int part_q = 0, part_k = 0, jj = -1;       // part: 0 hi, 1 lo;  jj: first channel of the pair (-1: zero padding)
    if (mode == 0) {
      const int seg = e >> 3;
      if (seg < 3 && (e & 7) < d) jj = e & 7, part_q = seg == 1, part_k = seg == 2;
    } else if (mode == 1) {
      const int half = KQ >> 1;
      const int part = e / half;
      if (e % half < d) jj = e % half, part_q = part_k = part;
    } else if (e < d) {
      jj = e;
    }
    if (jj < 0) return;
    const float q0 = pr[d + jj], q1 = pr[d + jj + 1], k0 = pr[2 * d + jj], k1 = pr[2 * d + jj + 1];
    qw = pack16x2(q0, q1, f16);
    kw = pack16x2(k0, k1, f16);
    if (part_q) {
      const float2 h = unpack16x2(qw, f16);
      qw = pack16x2(q0 - h.x, q1 - h.y, f16);
    }
    if (part_k) {
      const float2 h = unpack16x2(kw, f16);
      kw = pack16x2(k0 - h.x, k1 - h.y, f16);
    }
  };
  if (KQ % 8 == 0 && d % 2 == 0) {
    const int g8 = KQ >> 3;
    for (int i = threadIdx.x; i < rows * g8; i += blockDim.x) {
      const int r = i / g8, e0 = (i % g8) * 8;
      const float* pr = tile + r * pitch;
      uint32_t qw[4], kw[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) qk_pair(pr, e0 + 2 * e, qw[e], kw[e]);
      *reinterpret_cast<uint4*>(qd + (long long)r * KQ + e0) = make_uint4(qw[0], qw[1], qw[2], qw[3]);
      *reinterpret_cast<uint4*>(kd + (long long)r * KQ + e0) = make_uint4(kw[0], kw[1], kw[2], kw[3]);
    }
  } else if (KQ % 8 == 0) {
    const int g8 = KQ >> 3;
    for (int i = threadIdx.x; i < rows * g8; i += blockDim.x) {
      const int r = i / g8, e0 = (i % g8) * 8;
      const float* pr = tile + r * pitch;
      __nv_bfloat16 qv[8], kv[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) qk_elem(pr, e0 + e, qv[e], kv[e]);
      *reinterpret_cast<uint4*>(qd + (long long)r * KQ + e0) =
          make_uint4(bits(qv[0], qv[1]), bits(qv[2], qv[3]), bits(qv[4], qv[5]), bits(qv[6], qv[7]));
      *reinterpret_cast<uint4*>(kd + (long long)r * KQ + e0) =
          make_uint4(bits(kv[0], kv[1]), bits(kv[2], kv[3]), bits(kv[4], kv[5]), bits(kv[6], kv[7]));
    }
  } else {
    for (int i = threadIdx.x; i < rows * KQ; i += blockDim.x) {
      __nv_bfloat16 qv, kv;
      qk_elem(tile + (i / KQ) * pitch, i % KQ, qv, kv);
      qd[i] = qv;
      kd[i] = kv;
    }
  }
  // x_d
  float* xd = X + ((long long)b * N + n0) * d;
  if (d % 4 == 0) {
    const int g4 = d >> 2;
    for (int i = threadIdx.x; i < rows * g4; i += blockDim.x) {
      const float* pr = tile + (i / g4) * pitch + (i % g4) * 4;
      *reinterpret_cast<float4*>(xd + (long long)i * 4) = make_float4(pr[0], pr[1], pr[2], pr[3]);
    }
  } else {
    for (int i = threadIdx.x; i < rows * d; i += blockDim.x) xd[i] = tile[(i / d) * pitch + (i % d)];
  }
  // V^T (rows j >= d and the columns n >= N of the padded row stay zero): one thread = 8 consecutive keys of one row
  const int r8n = R >> 3;
  for (int i = threadIdx.x; i < DVp * r8n; i += blockDim.x) {
    const int j = i / r8n, r0 = (i % r8n) * 8;
    if (n0 + r0 >= Npad) continue;
    __nv_bfloat16 v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int r = r0 + e;
      float x = (j < d && r < rows) ? tile[r * pitch + 3 * d + j] : 0.f;
      if (ones_row && j == d && r < rows) x = 1.f;   // sum_j p_ij comes out of the P.V MMA as column d of O
      v[e] = f2h16(x, f16);
    }
    *reinterpret_cast<uint4*>(VT + ((long long)b * DVp + j) * Npad + n0 + r0) =
        make_uint4(bits(v[0], v[1]), bits(v[2], v[3]), bits(v[4], v[5]), bits(v[6], v[7]));
  }
}

struct AttnTcOp : esf_op {
  AttnTcParams params;
  dim3 grid;
  int smem_bytes = 0;
  int v2 = 0;
  int launch(cudaStream_t stream) override {
    if (v2) {
      if (params.f16) attn_tc_v2_kernel<true><<<grid, kV2Threads, smem_bytes, stream>>>(params);
      else attn_tc_v2_kernel<false><<<grid, kV2Threads, smem_bytes, stream>>>(params);
      return check_launch("attn_tc_v2_kernel");
    }
    if (params.split) attn_tc_kernel<true><<<grid, kTcThreads, smem_bytes, stream>>>(params);
    else attn_tc_kernel<false><<<grid, kTcThreads, smem_bytes, stream>>>(params);
    return check_launch("attn_tc_kernel");
  }
};

static int encode3(CUtensorMap* m, int f16, void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t s1_bytes,
                   uint64_t s2_bytes, uint32_t b0, uint32_t b1, CUtensorMapSwizzle sw, const char* what) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return set_error(ESF_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {s1_bytes, s2_bytes};
  cuuint32_t box[3] = {b0, b1, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(m, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, dims, strides,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(ESF_ERR_CUDA, "cuTensorMapEncodeTiled(%s) failed with %d", what, (int)r);
  return ESF_OK;
}

}  // namespace esf

using namespace esf;

extern "C" int64_t esf_attn_tc_pack_bytes(int32_t B, int32_t N, int32_t d) {
  TcGeom g;
  if (B <= 0 || N <= 0 || !tc_geom(d, &g)) return set_error(ESF_ERR_UNSUPPORTED, "esf_attn_tc: unsupported head dim %d", d);
  return tc_layout(B, N, d, g).total;
}

extern "C" int esf_attn_tc_pack(const float* proj, int32_t B, int32_t N, int32_t d, int32_t dtype, void* packed,
                                void* stream) {
  ESF_CHECK_ARG(proj && packed && B > 0 && N > 0 && is16(dtype), "esf_attn_tc_pack: null/bad argument");
  TcGeom g;
  if (!tc_geom(d, &g)) return set_error(ESF_ERR_UNSUPPORTED, "esf_attn_tc_pack: unsupported head dim %d", d);
  const TcLayout L = tc_layout(B, N, d, g);
  char* base = static_cast<char*>(packed);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int R = 256;
  while (R > 8 && (size_t)R * (4 * d + 1) * sizeof(float) > 40 * 1024) R >>= 1;
  const size_t smem = (size_t)R * (4 * d + 1) * sizeof(float);
  dim3 grid(cdiv(L.Npad, R), B);
#define ESF_PACK_ARGS                                                                                          \
  proj, N, L.Npad, d, g.KQ, g.DVp, g.mode, R, dtype == ESF_F16, g.v2, reinterpret_cast<__nv_bfloat16*>(base + L.q_off),  \
      reinterpret_cast<__nv_bfloat16*>(base + L.k_off), reinterpret_cast<__nv_bfloat16*>(base + L.v_off),       \
      reinterpret_cast<float*>(base + L.x_off)
  // compile-time geometry for the head dims of the shipped models (must agree with tc_geom and R above)
  if (d == 8 && g.KQ == 32 && g.DVp == 16 && g.mode == 0 && R == 256)
    attn_tc_pack_kernel<8, 32, 16, 0, 256><<<grid, 256, smem, s>>>(ESF_PACK_ARGS);
  else if (d == 32 && g.KQ == 64 && g.DVp == 48 && g.mode == 1 && R == 64)
    attn_tc_pack_kernel<32, 64, 48, 1, 64><<<grid, 256, smem, s>>>(ESF_PACK_ARGS);
  else if (d == 64 && g.KQ == 128 && g.DVp == 64 && g.mode == 1 && R == 32)
    attn_tc_pack_kernel<64, 128, 64, 1, 32><<<grid, 256, smem, s>>>(ESF_PACK_ARGS);
  else if (d == 128 && g.KQ == 128 && g.DVp == 128 && g.mode == 2 && R == 16)
    attn_tc_pack_kernel<128, 128, 128, 2, 16><<<grid, 256, smem, s>>>(ESF_PACK_ARGS);
  else
    attn_tc_pack_kernel<0, 0, 0, 0, 0><<<grid, 256, smem, s>>>(ESF_PACK_ARGS);
#undef ESF_PACK_ARGS
  return check_launch("attn_tc_pack_kernel");
}

static int attn_tc_create_impl(const void* packed, const void* v_lo, int32_t B, int32_t T, int32_t H, int32_t W, int32_t d,
                               float gamma, const float* bn_scale, const float* bn_shift, int32_t alpha,
                               const esf_view* y_fast_slice, esf_op** out);

extern "C" int esf_attn_tc_create(const void* packed, int32_t B, int32_t T, int32_t H, int32_t W, int32_t d,
                                  float gamma, const float* bn_scale, const float* bn_shift, int32_t alpha,
                                  const esf_view* y_fast_slice, esf_op** out) {
  return attn_tc_create_impl(packed, nullptr, B, T, H, W, d, gamma, bn_scale, bn_shift, alpha, y_fast_slice, out);
}

// ---- split mode (FP32-accurate plan): P and V as FP16 pairs ------------------------------------------------------------
// V_lo^T has the layout of V^T inside `packed` ([B][DVp][Npad] FP16): v_lo = fp16(v - fp16(v)), zeros in the ones row.
__global__ void __launch_bounds__(256) attn_tc_vlo_kernel(const float* __restrict__ proj, int N, int Npad, int d, int DVp,
                                                          __half* __restrict__ vlo) {
  const int b = blockIdx.y;
  const long long total = (long long)DVp * Npad;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(i / Npad), n = (int)(i % Npad);
    float lo = 0.f;
    if (j < d && n < N) {
      const float v = proj[((long long)b * N + n) * 4 * d + 3 * d + j];
      lo = v - __half2float(__float2half_rn(v));
    }
    vlo[(long long)b * total + i] = __float2half_rn(lo);
  }
}

extern "C" int64_t esf_attn_tc_vlo_bytes(int32_t B, int32_t N, int32_t d) {
  TcGeom g;
  if (B <= 0 || N <= 0 || !tc_geom(d, &g)) return set_error(ESF_ERR_ARG, "esf_attn_tc_vlo_bytes: bad argument");
  return (int64_t)B * g.DVp * ((N + 7) & ~7) * 2;
}

extern "C" int esf_attn_tc_pack_vlo(const float* proj, int32_t B, int32_t N, int32_t d, void* v_lo, void* stream) {
  ESF_CHECK_ARG(proj && v_lo && B > 0 && N > 0, "esf_attn_tc_pack_vlo: null/bad argument");
  TcGeom g;
  if (!tc_geom(d, &g)) return set_error(ESF_ERR_UNSUPPORTED, "esf_attn_tc_pack_vlo: unsupported head dim %d", d);
  const int Npad = (N + 7) & ~7;
  const long long total = (long long)g.DVp * Npad;
  dim3 grid((unsigned)std::min<long long>((total + 255) / 256, 148 * 8), B);
  attn_tc_vlo_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(proj, N, Npad, d, g.DVp, static_cast<__half*>(v_lo));
  return check_launch("attn_tc_vlo_kernel");
}

extern "C" int esf_attn_tc_create_split(const void* packed, const void* v_lo, int32_t B, int32_t T, int32_t H, int32_t W,
                                        int32_t d, float gamma, const float* bn_scale, const float* bn_shift,
                                        int32_t alpha, const esf_view* y_fast_slice, esf_op** out) {
  ESF_CHECK_ARG(v_lo != nullptr, "esf_attn_tc_create_split: v_lo is null");
  ESF_CHECK_ARG(y_fast_slice && y_fast_slice->dtype == ESF_F32, "esf_attn_tc_create_split: the output view must be FP32");
  ESF_CHECK_ARG(d <= 64, "esf_attn_tc_create_split: head dim %d > 64 has no hi/lo logit split (use esf_p32_attention)", d);
  return attn_tc_create_impl(packed, v_lo, B, T, H, W, d, gamma, bn_scale, bn_shift, alpha, y_fast_slice, out);
}

static int attn_tc_create_impl(const void* packed, const void* v_lo, int32_t B, int32_t T, int32_t H, int32_t W, int32_t d,
                               float gamma, const float* bn_scale, const float* bn_shift, int32_t alpha,
                               const esf_view* y_fast_slice, esf_op** out) {
  ESF_CHECK_ARG(packed && bn_scale && bn_shift && view_ok(y_fast_slice) && out, "esf_attn_tc_create: null/bad argument");
  // an FP32 output view selects the FP32-accurate path: the packed operands are then FP16 (esf_attn_tc_pack dtype F16)
  ESF_CHECK_ARG(is16(y_fast_slice->dtype) || y_fast_slice->dtype == ESF_F32,
                "esf_attn_tc_create: output must be BF16, F16 or F32");
  TcGeom g;
  if (!tc_geom(d, &g)) return set_error(ESF_ERR_UNSUPPORTED, "esf_attn_tc_create: unsupported head dim %d", d);
  const esf_view* y = y_fast_slice;
  ESF_CHECK_ARG(y->B == B && y->T == T * alpha && y->H == H && y->W == W && y->C == d,
                "esf_attn_tc_create: output slice (%d,%d,%d,%d,%d) != (%d,%d,%d,%d,%d)", y->B, y->T, y->H, y->W, y->C,
                B, T * alpha, H, W, d);
  const int N = T * H * W;
  const TcLayout L = tc_layout(B, N, d, g);
  char* base = static_cast<char*>(const_cast<void*>(packed));
  AttnTcOp* op = new (std::nothrow) AttnTcOp();
  if (!op) return set_error(ESF_ERR_ARG, "out of host memory");
  AttnTcParams& p = op->params;
  memset(&p, 0, sizeof(p));
  p.x = reinterpret_cast<const float*>(base + L.x_off);
  p.B = B, p.N = N, p.T = T, p.H = H, p.W = W, p.d = d, p.alpha = alpha, p.gamma = gamma;
  p.bn_scale = bn_scale, p.bn_shift = bn_shift;
  p.y = static_cast<__nv_bfloat16*>(y->ptr);
  p.ysB = y->sB, p.ysT = y->sT, p.ysH = y->sH, p.ysW = y->sW;
  p.DVp = g.DVp, p.nchunks = g.nchunks, p.chunk_el = g.chunk_el;
  p.f16 = y->dtype == ESF_F16 || y->dtype == ESF_F32;
  p.out_f32 = y->dtype == ESF_F32;
  const int RB = g.chunk_el * 2;
  p.sbo = 8 * RB;
  p.layout_type = RB == 128 ? 2 : 4;
  // a step = (offset of the A operand inside a Q tile) | (offset of the B operand inside a K tile) << 16, both in
  // 16-byte units (what gets added to the start-address field of the smem descriptors)
  const uint32_t cq16 = (128u * g.chunk_el * 2) >> 4, ck16 = ((uint32_t)kTcBN * g.chunk_el * 2) >> 4;
  auto step = [&](int ac, int ak, int bc, int bk) { return (uint32_t)((ac * cq16 + ak * 2) | ((bc * ck16 + bk * 2) << 16)); };
  int n1 = 0, n2 = 0;
  if (g.mode == 0) {
    // q~ = [q_hi q_lo | q_hi 0], k~ = [k_hi k_hi | k_lo 0]: step 0 = (q_hi+q_lo).k_hi, step 1 = q_hi.k_lo
    p.steps1[n1++] = step(0, 0, 0, 0);
    p.steps2[n2++] = step(0, 0, 0, 0);
    p.steps2[n2++] = step(0, 1, 0, 1);
  } else if (g.mode == 1) {
    const int half = g.KQ / 2;            // elements of the hi (and of the lo) part
    const int hs = half / 16;             // K steps per part
    auto loc = [&](int part, int k, int* chunk, int* koff) {  // K step k of part -> (chunk, 32 B offset in chunk)
      const int el = part * half + k * 16;
      *chunk = el / g.chunk_el;
      *koff = (el % g.chunk_el) / 16;
    };
    for (int k = 0; k < hs; ++k) {
      int ac, ak, bc, bk;
      loc(0, k, &ac, &ak), loc(0, k, &bc, &bk);
      p.steps1[n1++] = step(ac, ak, bc, bk);
      p.steps2[n2++] = step(ac, ak, bc, bk);  // hi.hi
    }
    for (int k = 0; k < hs; ++k) {
      int ac, ak, bc, bk;
      loc(1, k, &ac, &ak), loc(0, k, &bc, &bk);
      p.steps2[n2++] = step(ac, ak, bc, bk);  // lo.hi
    }
    for (int k = 0; k < hs; ++k) {
      int ac, ak, bc, bk;
      loc(0, k, &ac, &ak), loc(1, k, &bc, &bk);
      p.steps2[n2++] = step(ac, ak, bc, bk);  // hi.lo
    }
  } else {
    for (int k = 0; k < g.KQ / 16; ++k) {
      const int c = (k * 16) / g.chunk_el, ko = ((k * 16) % g.chunk_el) / 16;
      p.steps1[n1++] = step(c, ko, c, ko);
      p.steps2[n2++] = step(c, ko, c, ko);
    }
  }
  p.nsteps1 = n1, p.nsteps2 = n2;
  p.q_tile_bytes = 128 * g.KQ * 2;
  p.k_tile_bytes = kTcBN * g.KQ * 2;
  p.v_tile_bytes = g.DVp * 128;
  op->v2 = g.v2;
  if (v_lo) {   // split mode runs on the one-row-per-thread kernel (row sums in FP32 registers, P through shared memory)
    p.split = 1;
    p.v_half = p.v_tile_bytes;
    p.v_tile_bytes *= 2;
    op->v2 = 0;
  }
  // v1 streams P through 2 x 16 KB of shared memory; v2 keeps P in TMEM and needs 2 KB for the split-K maxima
  const int fixed = 1024 + 2 * (int)p.q_tile_bytes + 512 + (op->v2 ? 2048 : 2 * (p.split ? 32768 : 16384));
  int stages = (kTcSmemLimit - fixed) / (int)(p.k_tile_bytes + p.v_tile_bytes);
  p.stages = std::max(2, std::min(stages, kTcMaxStages));
  op->smem_bytes = fixed + p.stages * (int)(p.k_tile_bytes + p.v_tile_bytes);
  op->grid = dim3(cdiv(N, 256), B);
  const CUtensorMapSwizzle sw = RB == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  int rc = encode3(&p.q_map, p.f16, base + L.q_off, g.KQ, N, B, (uint64_t)g.KQ * 2, (uint64_t)N * g.KQ * 2, g.chunk_el, 128, sw,
                   "attention Q");
  if (rc == ESF_OK)
    rc = encode3(&p.k_map, p.f16, base + L.k_off, g.KQ, N, B, (uint64_t)g.KQ * 2, (uint64_t)N * g.KQ * 2, g.chunk_el, kTcBN, sw,
                 "attention K");
  if (rc == ESF_OK)
    rc = encode3(&p.v_map, p.f16, base + L.v_off, N, g.DVp, B, (uint64_t)L.Npad * 2, (uint64_t)g.DVp * L.Npad * 2, kTcBN, g.DVp,
                 CU_TENSOR_MAP_SWIZZLE_128B, "attention V^T");
  if (rc == ESF_OK && v_lo)
    rc = encode3(&p.vlo_map, p.f16, const_cast<void*>(v_lo), N, g.DVp, B, (uint64_t)L.Npad * 2, (uint64_t)g.DVp * L.Npad * 2,
                 kTcBN, g.DVp, CU_TENSOR_MAP_SWIZZLE_128B, "attention V_lo^T");
  if (rc == ESF_OK && !v_lo) p.vlo_map = p.v_map;   // fully initialised parameter block
  if (rc == ESF_OK) {
    static unsigned char attr_done[kMaxDevices] = {0};   // kernel attributes are per device
    unsigned char* slot = device_slot(attr_done);
    if (!slot || !*slot) {
      cudaError_t e = cudaFuncSetAttribute(attn_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmemLimit);
      if (e == cudaSuccess)
        e = cudaFuncSetAttribute(attn_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmemLimit);
      if (e == cudaSuccess)
        e = cudaFuncSetAttribute(attn_tc_v2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmemLimit);
      if (e == cudaSuccess)
        e = cudaFuncSetAttribute(attn_tc_v2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmemLimit);
      if (e != cudaSuccess) rc = set_error(ESF_ERR_CUDA, "cudaFuncSetAttribute(attn_tc) failed: %s", cudaGetErrorString(e));
      else if (slot) *slot = 1;
    }
  }
  if (rc != ESF_OK) {
    delete op;
    return rc;
  }
  *out = op;
  return ESF_OK;
}
