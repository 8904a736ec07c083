// Dense Conv3d (+ folded BatchNorm, + residual, + ReLU) as a persistent, warp-specialised implicit GEMM on the
// 5th-generation tensor cores:  D[m, n] = sum_{tap, c} X[pos(m) + tap, c] * Wp[n, tap, c]
//
//   M  = a box of (bw x bh x bt x bb) <= 128 output positions of the channels-last (B,T,H,W,C) activation,
//   N  = n_tile output channels (16..256),  K = taps x input-channel chunks of kc in {16,32,64} elements.
//
//   warp 16     TMA producer: one 5-D box load per (tap, chunk) of the activation -- the filter tap is a coordinate
//               offset, zero padding is TMA out-of-bounds fill, a strided conv reads one tensor map per stride phase
//               -- plus a 2-D load of the packed weights; `stages`-deep mbarrier ring.
//   warp 17     MMA issuer: one elected thread issues tcgen05.mma (M=128, N=n_tile, K=16) into one of two TMEM
//               accumulators; tcgen05.commit releases smem stages / publishes the accumulator.
//   warps 0-15  epilogue: tcgen05.ld -> + bias (+ residual tile fetched by TMA) -> ReLU -> 16-bit/FP32 -> swizzled smem
//               -> TMA store straight into the (possibly channel-sliced) destination, i.e. concat is free.  Sixteen
//               warps (four per TMEM lane quarter, a quarter of the slab's columns each) because 1x1x1 expansions are
//               bound by this path, not by the MMAs.
//   warp 18     residual producer: TMA-loads the residual tile of each output slab into the staging buffer the
//               epilogue will overwrite in place, `obufs - 1` slabs ahead of its consumer.
//
// Reference ops replaced: see include/esf.h (esf_conv_igemm_create).
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <vector>

#include "esf_common.cuh"
#include "esf_host.h"

namespace esf {

constexpr int kEpiWarps = 16;
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kProducerWarp = 16;
constexpr int kMmaWarp = 17;
constexpr int kResWarp = 18;
constexpr int kThreads = 19 * 32;
constexpr int kMaxStages = 8;
constexpr int kMaxAMaps = 8;
constexpr int kMaxTaps = 64;
constexpr int kAStageBytes = 16384;   // 128 rows x 128 B
constexpr int kOutStageBytes = 16384; // 128 rows x 128 B
constexpr int kMaxOutBufs = 8;
constexpr int kTmemCols = 512;
constexpr int kSmemLimit = 232448;    // 227 KB

struct __align__(64) IgemmParams {
  CUtensorMap a_maps[kMaxAMaps];
  CUtensorMap b_map;
  CUtensorMap out_map;
  CUtensorMap res_map;
  int4 taps[kMaxTaps];  // x: a_map index, y/z/w: coordinate offsets along W/H/T in that map
  int num_taps, kchunks, kc;
  int n_tile, n_tiles;
  int bw, bh, bt, bb;  // output box of one M tile
  int tw, th, tt, tb;  // boxes per dimension
  int rows;            // bw*bh*bt*bb
  int stages;
  uint32_t a_bytes, b_bytes, b_stride;  // TMA bytes per stage / smem stride of a B stage
  uint32_t sbo, layout_type;            // UMMA descriptor fields for the A/B swizzle mode
  uint32_t res_bytes;
  const float* bias;
  int act, has_res, out_f32, f16;  // f16: 16-bit operands / outputs are IEEE half instead of BF16
  int slab_cols;      // output columns per TMA store slab
  uint32_t out_swz;   // swizzle mask of the staging rows (7 / 3 / 1)
  int num_tiles;
  // "column blocks" (banded stem GEMM): an extra tile index that shifts the innermost coordinate of the
  // activation loads and of the output stores; ncb == 1 and zero strides for ordinary convolutions
  int ncb, a_cb_stride, out_cb_w;  // out_cb_w: W-coordinate step of the output store per column block
  int obufs;                       // depth of the output/residual staging ring (3..kMaxOutBufs)
  // W-folded GEMMs (thin-channel layers): innermost start coordinate of the activation loads, and -- when the output
  // (residual) is a channel slice -- the (w, c) decomposition of an output column n = w_in_block * cout + c
  int a_c_base, fold_wb, out_fold_cout, res_fold_cout;
  // per-clip weights (Non-local block: the "weight" matrix of a clip is its own phi / g^T rows): the packed weight
  // matrices of all clips are stacked along n, b_clip_rows rows each, and an M tile never spans two clips (bb = 1)
  int b_clip_rows;
  uint32_t dv_mul[5], dv_shr[5];   // magic numbers of the divisions by n_tiles, ncb, tw, th, tt (finish_op)
};

struct TileCoord {
  int n_idx, cb, w0, h0, t0, b0;
};
// x / d for 0 <= x < 2^31 by a multiply-high and a shift (m = ceil(2^(31 + ceil(log2 d)) / d), the usual magic-number
// division): the five run-time divisions of a tile index were a ~1000-cycle dependent chain on the critical path of
// every tile (the TMA-store leader, the producer and the residual warp all decompose the index).
__device__ __forceinline__ int fast_div(int x, uint32_t mul, uint32_t shr) {
  return mul ? (int)(__umulhi((uint32_t)x, mul) >> shr) : x;
}
__device__ __forceinline__ TileCoord tile_coord(const IgemmParams& p, int tile) {
  TileCoord c;
  int m = fast_div(tile, p.dv_mul[0], p.dv_shr[0]);
  c.n_idx = tile - m * p.n_tiles;
  int q = fast_div(m, p.dv_mul[1], p.dv_shr[1]);
  c.cb = m - q * p.ncb;
  m = q;
  q = fast_div(m, p.dv_mul[2], p.dv_shr[2]);
  c.w0 = (m - q * p.tw) * p.bw;
  m = q;
  q = fast_div(m, p.dv_mul[3], p.dv_shr[3]);
  c.h0 = (m - q * p.th) * p.bh;
  m = q;
  q = fast_div(m, p.dv_mul[4], p.dv_shr[4]);
  c.t0 = (m - q * p.tt) * p.bt;
  c.b0 = q * p.bb;
  return c;
}

// staging rows are addressed in the shared state space (32-bit addresses, LDS / STS) -- generic 64-bit pointers cost
// two extra integer instructions per access and a generic-to-shared resolution on the epilogue's critical path
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__device__ __forceinline__ void epi_bar_sync(int id) { asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(kEpiThreads) : "memory"); }

// One epilogue thread: NC accumulator columns of its row for one output slab.  `row` points at the thread's staging row,
// `inner` is the byte offset of its first column inside the row and `x` the row's swizzle XOR term.
template <int NC, bool F16>
__device__ __forceinline__ void epi_process16(uint32_t taddr, const float* __restrict__ bias, uint32_t row, uint32_t inner,
                                              uint32_t x, bool has_res, int act, bool row_valid) {
  float v[NC], b[NC];
  uint4 rr[NC / 8];
#pragma unroll
  for (int c = 0; c < NC / 4; ++c) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(bias) + c);
    b[4 * c] = t.x, b[4 * c + 1] = t.y, b[4 * c + 2] = t.z, b[4 * c + 3] = t.w;
  }
  if (has_res) {
#pragma unroll
    for (int c = 0; c < NC / 8; ++c) rr[c] = lds128(row + ((inner + c * 16) ^ x));
  }
  tmem_ld<NC>(taddr, v);
#pragma unroll
  for (int j = 0; j < NC; ++j) v[j] += b[j];
  if (has_res) {
#pragma unroll
    for (int c = 0; c < NC / 8; ++c) {
      const uint32_t u[4] = {rr[c].x, rr[c].y, rr[c].z, rr[c].w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 f = unpack16x2(u[e], F16);
        v[8 * c + 2 * e] += f.x;
        v[8 * c + 2 * e + 1] += f.y;
      }
    }
  }
  const float lo = act ? 0.f : -INFINITY;
#pragma unroll
  for (int j = 0; j < NC; ++j) v[j] = fmaxf(v[j], lo);
  if (act == 2) {
#pragma unroll
    for (int j = 0; j < NC; ++j) v[j] = fminf(v[j], 6.f);
  }
  if (row_valid) {
#pragma unroll
    for (int c = 0; c < NC / 8; ++c) {
      uint4 o;
      o.x = pack16x2(v[8 * c + 0], v[8 * c + 1], F16);
      o.y = pack16x2(v[8 * c + 2], v[8 * c + 3], F16);
      o.z = pack16x2(v[8 * c + 4], v[8 * c + 5], F16);
      o.w = pack16x2(v[8 * c + 6], v[8 * c + 7], F16);
      sts128(row + ((inner + c * 16) ^ x), o);
    }
  }
}

// FP32 destination (attention projections): 8 columns per thread, no residual.
__device__ __forceinline__ void epi_process32(uint32_t taddr, const float* __restrict__ bias, uint32_t row, uint32_t inner,
                                              uint32_t x, int act, bool row_valid) {
  float v[8];
  tmem_ld<8>(taddr, v);
#pragma unroll
  for (int j = 0; j < 8; ++j) v[j] = apply_act(v[j] + __ldg(bias + j), act);
  if (row_valid) {
    sts128(row + (inner ^ x), make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3])));
    sts128(row + ((inner + 16) ^ x),
           make_uint4(__float_as_uint(v[4]), __float_as_uint(v[5]), __float_as_uint(v[6]), __float_as_uint(v[7])));
  }
}

struct EpiCtx {
  uint8_t* smem_out;
  uint64_t *tmem_full, *tmem_empty, *res_full, *buf_free;
  uint32_t tmem_base;
  int warp, lane;
};

// The tile loop of the 16 epilogue warps (see the kernel header): TMEM -> + bias (+ residual) -> activation -> staging
// smem -> TMA store.
template <int CPT, bool F16, bool F32OUT>
__device__ __forceinline__ void epilogue_loop(const IgemmParams& p, const EpiCtx& ec) {
  const int warp = ec.warp, lane = ec.lane;
  const int act = p.act;
  const int q = warp & 3;       // TMEM lane quarter this warp may access
  const int part = warp >> 2;   // which share of the slab's columns
  const int r = q * 32 + lane;
  const bool row_valid = r < p.rows;
  const bool leader = threadIdx.x == 0;
  const int slabs = p.n_tile / p.slab_cols;
  constexpr int cpt = CPT;  // columns per thread per slab
  const bool active = part * cpt < p.slab_cols;
  constexpr int oes = F32OUT ? 4 : 2;
  const uint32_t rowoff = r * p.slab_cols * oes;
  const uint32_t inner = part * cpt * oes;
  const uint32_t x = ((rowoff >> 7) & p.out_swz) << 4;
  const int R = p.obufs;
  const bool has_res = p.has_res != 0;
  const uint32_t stage_base = smem_u32(ec.smem_out);
  int buf = 0, use = 0, prev_buf = 0;
  bool first = true;
  int iter = 0;
  // Per-tile integer work of the 512 epilogue threads is what bounds the small-N layers (ncu, 1x1x1 64->32 @56^2: 309
  // instructions per warp and tile, half of them the six divisions of tile_coord; 89 % of all instructions of the
  // kernel): only the leader needs the tile's coordinates (for the TMA store), everybody else just its N tile, which
  // is carried incrementally.
  const int n_step = gridDim.x % p.n_tiles;
  int n_idx = blockIdx.x % p.n_tiles;
  for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++iter) {
    TileCoord tc;
    if (leader) tc = tile_coord(p, tile);
    const int acc = iter & 1;
    const uint32_t acc_phase = (iter >> 1) & 1;
    mbar_wait(&ec.tmem_full[acc], acc_phase, 4);
    tc_fence_after();
    for (int s = 0; s < slabs; ++s) {
      uint8_t* stage_buf = ec.smem_out + buf * kOutStageBytes;
      if (has_res) mbar_wait(&ec.res_full[buf], use & 1, 5);
      if (active) {
        const int col = s * p.slab_cols + part * cpt;
        const uint32_t taddr = ec.tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * p.n_tile + col;
        const float* bias = p.bias + n_idx * p.n_tile + col;
        const uint32_t row = stage_base + buf * kOutStageBytes + rowoff;
        if constexpr (F32OUT) epi_process32(taddr, bias, row, inner, x, act, row_valid);
        else epi_process16<CPT, F16>(taddr, bias, row, inner, x, has_res, act, row_valid);
      }
      if (s == slabs - 1) {  // accumulator fully drained: hand the TMEM buffer back to the MMA warp
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&ec.tmem_empty[acc]);
      }
      fence_proxy_async_smem();
      // One barrier per slab is enough with a ring of >= 3 buffers: a thread that runs ahead writes buffer
      // (g + 1) % R, whose previous store (g + 1 - R <= g - 2) the leader saw finish reading before it arrived here.
      epi_bar_sync(1);
      if (leader) {
        int c = tc.n_idx * p.n_tile + s * p.slab_cols, w = tc.w0 + tc.cb * p.out_cb_w;
        if (p.out_fold_cout) {
          w = tc.cb * p.fold_wb + c / p.out_fold_cout;
          c = c % p.out_fold_cout;
        }
        tma_store_5d(&p.out_map, stage_buf, c, w, tc.h0, tc.t0, tc.b0);
        tma_store_commit();
        tma_store_wait_read<1>();  // every store before this one has finished reading its staging buffer
        if (has_res && !first) mbar_arrive(&ec.buf_free[prev_buf]);
      }
      first = false;
      prev_buf = buf;
      if (++buf == R) {
        buf = 0;
        ++use;
      }
    }
    n_idx += n_step;
    if (n_idx >= p.n_tiles) n_idx -= p.n_tiles;
  }
  if (leader) tma_store_wait_all<0>();
}

__global__ void __launch_bounds__(kThreads, 1) igemm_kernel(const __grid_constant__ IgemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem_a + p.stages * kAStageBytes;
  uint8_t* smem_out = smem_b + p.stages * p.b_stride;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem_out + p.obufs * kOutStageBytes);
  uint64_t* empty_bar = full_bar + kMaxStages;
  uint64_t* tmem_full = empty_bar + kMaxStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* res_full = tmem_empty + 2;
  uint64_t* buf_free = res_full + kMaxOutBufs;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(buf_free + kMaxOutBufs);

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], kEpiWarps);  // one arrival per epilogue warp
    }
    for (int a = 0; a < p.obufs; ++a) {
      mbar_init(&res_full[a], 1);
      mbar_init(&buf_free[a], 1);
    }
    fence_barrier_init();
  }
  if (warp == kProducerWarp && lane == 0) {
    prefetch_tmap(&p.a_maps[0]);
    prefetch_tmap(&p.b_map);
    prefetch_tmap(&p.out_map);
    if (p.has_res) prefetch_tmap(&p.res_map);
  }
  if (warp == kMmaWarp) {
    tmem_alloc(tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int num_kb = p.num_taps * p.kchunks;

  if (warp == kProducerWarp) {
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      const TileCoord tc = tile_coord(p, tile);
      for (int tap = 0; tap < p.num_taps; ++tap) {
        const int4 tp = p.taps[tap];
        for (int ch = 0; ch < p.kchunks; ++ch) {
          mbar_wait(&empty_bar[stage], phase ^ 1, 1);
          if (elect_one()) {
            mbar_arrive_expect_tx(&full_bar[stage], p.a_bytes + p.b_bytes);
            tma_load_5d(smem_a + stage * kAStageBytes, &p.a_maps[tp.x], &full_bar[stage],
                        p.a_c_base + tc.cb * p.a_cb_stride + ch * p.kc, tc.w0 + tp.y, tc.h0 + tp.z, tc.t0 + tp.w, tc.b0);
            tma_load_2d(smem_b + stage * p.b_stride, &p.b_map, &full_bar[stage],
                        (tap * p.kchunks + ch) * p.kc, tc.n_idx * p.n_tile + tc.b0 * p.b_clip_rows);
          }
          __syncwarp();
          if (++stage == p.stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == kMmaWarp) {
    {
      // the issuing thread is a serial instruction stream: keep it to two adds per MMA (descriptor lo words)
      const uint32_t idesc = make_idesc_16(128, p.n_tile, p.f16);
      const uint32_t desc_hi = kmajor_desc_hi(p.sbo, p.layout_type);
      const uint32_t a_lo0 = kmajor_desc_lo(smem_u32(smem_a)), b_lo0 = kmajor_desc_lo(smem_u32(smem_b));
      const uint32_t a_step = kAStageBytes >> 4, b_step = p.b_stride >> 4;
      const int ksteps = p.kc >> 4;
      int stage = 0;
      uint32_t phase = 0;
      uint32_t a_lo = a_lo0, b_lo = b_lo0;
      int iter = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++iter) {
        const int acc = iter & 1;
        const uint32_t acc_phase = (iter >> 1) & 1;
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1, 2);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * p.n_tile;
        uint32_t accum = 0;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase, 3);
          tc_fence_after();
          if (elect_one()) {
            if (ksteps == 4) {
              umma_bf16_lohi(d_tmem, a_lo, desc_hi, b_lo, desc_hi, idesc, accum);
              umma_bf16_lohi(d_tmem, a_lo + 2, desc_hi, b_lo + 2, desc_hi, idesc, 1);
              umma_bf16_lohi(d_tmem, a_lo + 4, desc_hi, b_lo + 4, desc_hi, idesc, 1);
              umma_bf16_lohi(d_tmem, a_lo + 6, desc_hi, b_lo + 6, desc_hi, idesc, 1);
            } else {
              umma_bf16_lohi(d_tmem, a_lo, desc_hi, b_lo, desc_hi, idesc, accum);
              if (ksteps == 2) umma_bf16_lohi(d_tmem, a_lo + 2, desc_hi, b_lo + 2, desc_hi, idesc, 1);
            }
            umma_commit(&empty_bar[stage]);
            if (kb == num_kb - 1) umma_commit(&tmem_full[acc]);
          }
          __syncwarp();
          accum = 1;
          a_lo += a_step;
          b_lo += b_step;
          if (++stage == p.stages) {
            stage = 0;
            phase ^= 1;
            a_lo = a_lo0;
            b_lo = b_lo0;
          }
        }
      }
    }
  } else if (warp == kResWarp) {
    // residual tile of this CTA's k-th slab -> staging buffer k % R, as soon as the store that last used the buffer
    // has read it: the DRAM latency of the (HBM-bound) residual stream and the coordinate arithmetic stay off the
    // epilogue's critical path
    if (p.has_res) {
      const int slabs = p.n_tile / p.slab_cols;
      const int R = p.obufs;
      int buf = 0, use = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        const TileCoord tc = tile_coord(p, tile);
        for (int s = 0; s < slabs; ++s) {
          if (use > 0) mbar_wait(&buf_free[buf], (use - 1) & 1, 6);
          if (elect_one()) {
            int c = tc.n_idx * p.n_tile + s * p.slab_cols, w = tc.w0 + tc.cb * p.out_cb_w;
            if (p.res_fold_cout) {
              w = tc.cb * p.fold_wb + c / p.res_fold_cout;
              c = c % p.res_fold_cout;
            }
            mbar_arrive_expect_tx(&res_full[buf], p.res_bytes);
            tma_load_5d(smem_out + buf * kOutStageBytes, &p.res_map, &res_full[buf], c, w, tc.h0, tc.t0, tc.b0);
          }
          __syncwarp();
          if (++buf == R) {
            buf = 0;
            ++use;
          }
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps 0..15
    // dispatched ONCE on the layer's output format / columns per thread, so that the per-slab body is straight-line code
    // with compile-time shapes (the run-time `if (out_f32) .. else if (cpt == 16) .. if (f16)` ladder inside the loop
    // cost ~100 of the 173 instructions per warp and tile that bound the small-N layers)
    EpiCtx c;
    c.smem_out = smem_out, c.tmem_full = tmem_full, c.tmem_empty = tmem_empty, c.res_full = res_full;
    c.buf_free = buf_free, c.tmem_base = tmem_base, c.warp = warp, c.lane = lane;
    const int cpt = max(8, p.slab_cols >> 2);  // columns per thread per slab
    if (p.out_f32) epilogue_loop<8, false, true>(p, c);
    else if (cpt == 16) {
      if (p.f16) epilogue_loop<16, true, false>(p, c);
      else epilogue_loop<16, false, false>(p, c);
    } else {
      if (p.f16) epilogue_loop<8, true, false>(p, c);
      else epilogue_loop<8, false, false>(p, c);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------ host side
EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess || !p) return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

// Split shared memory between the operand pipeline and the output/residual staging ring.  Layers with a short K loop
// (1x1x1 expansions) are bound by the epilogue and the residual stream, so they get the deeper ring; layers with a
// long K loop need the stages.
static void plan_smem(IgemmParams& p, int* smem_bytes) {
  const int avail = kSmemLimit - 1024 - 512;
  const int stage_bytes = kAStageBytes + (int)p.b_stride;
  const int ksteps = p.num_taps * p.kchunks;
  const int want_stages = std::min(p.n_tile >= 256 ? 3 : 4, ksteps + 1);
  int R = p.has_res ? 6 : 3;
  while (R > 3 && (avail - R * kOutStageBytes) / stage_bytes < want_stages) --R;
  p.obufs = R;
  const int stages = (avail - R * kOutStageBytes) / stage_bytes;
  p.stages = std::max(2, std::min(stages, kMaxStages));
  *smem_bytes = 1024 + 512 + R * kOutStageBytes + p.stages * stage_bytes;
}

static CUtensorMapSwizzle swizzle_for_row_bytes(int row_bytes) {
  if (row_bytes == 128) return CU_TENSOR_MAP_SWIZZLE_128B;
  if (row_bytes == 64) return CU_TENSOR_MAP_SWIZZLE_64B;
  return CU_TENSOR_MAP_SWIZZLE_32B;
}

// 5-D map over a channels-last view: dims (C, W, H, T, B).
static int encode_act_map(CUtensorMap* m, CUtensorMapDataType dt, int esize, void* base, int64_t C, int64_t W,
                          int64_t H, int64_t T, int64_t B, int64_t sW, int64_t sH, int64_t sT, int64_t sB, int boxC,
                          int bw, int bh, int bt, int bb, CUtensorMapSwizzle swz_mode, const char* what) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return set_error(ESF_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)T, (cuuint64_t)B};
  cuuint64_t strides[4] = {(cuuint64_t)(sW * esize), (cuuint64_t)(sH * esize), (cuuint64_t)(sT * esize),
                           (cuuint64_t)(sB * esize)};
  cuuint32_t box[5] = {(cuuint32_t)boxC, (cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)bt, (cuuint32_t)bb};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0)
    return set_error(ESF_ERR_ARG, "%s: base address %p not 16-byte aligned", what, base);
  for (int i = 0; i < 4; ++i)
    if (strides[i] % 16 != 0)
      return set_error(ESF_ERR_ARG, "%s: stride %d = %llu bytes is not a multiple of 16", what, i,
                       (unsigned long long)strides[i]);
  CUresult r = enc(m, dt, 5, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz_mode,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return set_error(ESF_ERR_CUDA,
                     "cuTensorMapEncodeTiled(%s) failed with %d: dims (%lld,%lld,%lld,%lld,%lld) box (%d,%d,%d,%d,%d)",
                     what, (int)r, (long long)C, (long long)W, (long long)H, (long long)T, (long long)B, boxC, bw, bh,
                     bt, bb);
  return ESF_OK;
}

static int g_num_sms[kMaxDevices] = {0};
int num_sms() {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  if (dev >= 0 && dev < kMaxDevices && g_num_sms[dev] > 0) return g_num_sms[dev];
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
  if (dev >= 0 && dev < kMaxDevices) g_num_sms[dev] = n;
  return n;
}

struct IgemmOp : esf_op {
  IgemmParams params;
  int grid = 0;
  int smem_bytes = 0;
  int launch(cudaStream_t stream) override {
    igemm_kernel<<<grid, kThreads, smem_bytes, stream>>>(params);
    return check_launch("igemm_kernel");
  }
};

}  // namespace esf

using namespace esf;

static void magic_div(int d, uint32_t* mul, uint32_t* shr) {
  if (d <= 1) {
    *mul = 0, *shr = 0;     // fast_div: identity
    return;
  }
  int lg = 0;
  while ((1LL << lg) < d) ++lg;           // ceil(log2 d)
  const int pw = 31 + lg;
  *mul = (uint32_t)(((1ULL << pw) + (uint64_t)d - 1) / (uint64_t)d);
  *shr = (uint32_t)(pw - 32);
}

static int finish_op(IgemmOp* op) {
  {
    IgemmParams& p = op->params;
    const int dv[5] = {p.n_tiles, p.ncb, p.tw, p.th, p.tt};
    for (int i = 0; i < 5; ++i) magic_div(dv[i], &p.dv_mul[i], &p.dv_shr[i]);
  }
  const int sms = num_sms();
  if (sms <= 0) return set_error(ESF_ERR_CUDA, "no CUDA device");
  op->grid = std::min(op->params.num_tiles, sms);
  static unsigned char attr_done[kMaxDevices] = {0};
  unsigned char* slot = device_slot(attr_done);
  if (!slot || !*slot) {
    cudaError_t e = cudaFuncSetAttribute(igemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit);
    if (e != cudaSuccess) return set_error(ESF_ERR_CUDA, "cudaFuncSetAttribute(igemm) failed: %s", cudaGetErrorString(e));
    if (slot) *slot = 1;
  }
  return ESF_OK;
}

extern "C" int esf_igemm_geometry(int32_t cin, int32_t cout, int32_t* kc, int32_t* kchunks, int32_t* n_tile,
                                  int32_t* n_pad) {
  ESF_CHECK_ARG(cin > 0 && cout > 0, "esf_igemm_geometry: cin/cout must be positive");
  const int k = cin <= 16 ? 16 : (cin <= 32 ? 32 : 64);
  int nt = 16;
  while (nt < cout && nt < 256) nt *= 2;
  if (kc) *kc = k;
  if (kchunks) *kchunks = cdiv(cin, k);
  if (n_tile) *n_tile = nt;
  if (n_pad) *n_pad = cdiv(cout, nt) * nt;
  return ESF_OK;
}

// pick the output box (bw,bh,bt,bb), product <= 128, maximising the fraction of useful MMA rows
static void choose_box(int W, int H, int T, int B, int* obw, int* obh, int* obt, int* obb) {
  double best = -1.0;
  int best_sp = 0;
  int rb[4] = {1, 1, 1, 1};
  for (int bw = 1; bw <= std::min(W, 128); ++bw)
    for (int bh = 1; bh <= std::min(H, 128 / bw); ++bh)
      for (int bt = 1; bt <= std::min(T, 128 / (bw * bh)); ++bt) {
        const int bb = std::min(B, 128 / (bw * bh * bt));
        const double tiles = (double)cdiv(W, bw) * cdiv(H, bh) * cdiv(T, bt) * cdiv(B, bb);
        const double eff = ((double)W * H * T * B) / (tiles * 128.0);
        const int sp = bw * bh;
        if (eff > best + 1e-9 || (eff > best - 1e-9 && sp > best_sp)) {
          best = std::max(best, eff);
          best_sp = sp;
          rb[0] = bw, rb[1] = bh, rb[2] = bt, rb[3] = bb;
        }
      }
  *obw = rb[0], *obh = rb[1], *obt = rb[2], *obb = rb[3];
}



static inline int floordiv(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }

static int igemm_create_impl(const esf_conv_desc* d, int clip_weights, esf_op** out);

extern "C" int esf_conv_igemm_create(const esf_conv_desc* d, esf_op** out) { return igemm_create_impl(d, 0, out); }

extern "C" int esf_gemm_clip_weights_create(const esf_conv_desc* d, esf_op** out) {
  ESF_CHECK_ARG(d && d->kT == 1 && d->kH == 1 && d->kW == 1 && d->sT == 1 && d->sH == 1 && d->sW == 1 && d->pT == 0 &&
                    d->pH == 0 && d->pW == 0 && !d->res.ptr,
                "esf_gemm_clip_weights_create: 1x1x1, stride 1, no residual");
  return igemm_create_impl(d, 1, out);
}

static int igemm_create_impl(const esf_conv_desc* d, int clip_weights, esf_op** out) {
  ESF_CHECK_ARG(d && out, "esf_conv_igemm_create: null argument");
  ESF_CHECK_ARG(view_ok(&d->x) && view_ok(&d->y), "esf_conv_igemm_create: bad x/y view");
  ESF_CHECK_ARG(d->groups == 1, "esf_conv_igemm_create: groups must be 1 (use esf_conv_direct)");
  ESF_CHECK_ARG(d->w && d->bias, "esf_conv_igemm_create: null weights/bias");
  ESF_CHECK_ARG(d->kT >= 1 && d->kH >= 1 && d->kW >= 1 && d->sT >= 1 && d->sH >= 1 && d->sW >= 1 && d->dT >= 1 &&
                    d->dH >= 1 && d->dW >= 1 && d->pT >= 0 && d->pH >= 0 && d->pW >= 0,
                "esf_conv_igemm_create: bad kernel/stride/pad/dilation");
  const esf_view& x = d->x;
  const esf_view& y = d->y;
  const int To = (x.T + 2 * d->pT - d->dT * (d->kT - 1) - 1) / d->sT + 1;
  const int Ho = (x.H + 2 * d->pH - d->dH * (d->kH - 1) - 1) / d->sH + 1;
  const int Wo = (x.W + 2 * d->pW - d->dW * (d->kW - 1) - 1) / d->sW + 1;
  ESF_CHECK_ARG(y.B == x.B && y.T == To && y.H == Ho && y.W == Wo,
                "esf_conv_igemm_create: output view (%d,%d,%d,%d) does not match conv output (%d,%d,%d,%d)", y.B, y.T,
                y.H, y.W, x.B, To, Ho, Wo);
  const int num_taps = d->kT * d->kH * d->kW;
  ESF_CHECK_ARG(num_taps <= kMaxTaps, "esf_conv_igemm_create: %d taps > %d", num_taps, kMaxTaps);
  ESF_CHECK_ARG(is16(x.dtype), "esf_conv_igemm_create: input must be BF16 or F16");
  ESF_CHECK_ARG(d->out_dtype == ESF_F32 || d->out_dtype == x.dtype,
                "esf_conv_igemm_create: out_dtype must be F32 or the input's 16-bit format");
  ESF_CHECK_ARG(y.dtype == d->out_dtype, "esf_conv_igemm_create: y.dtype != out_dtype");
  ESF_CHECK_ARG(!(d->out_dtype == ESF_F32 && d->res.ptr), "esf_conv_igemm_create: residual needs a 16-bit output");
  if (d->res.ptr) ESF_CHECK_ARG(d->res.dtype == x.dtype, "esf_conv_igemm_create: residual format != input format");
  if (d->res.ptr)
    ESF_CHECK_ARG(d->res.B == y.B && d->res.T == y.T && d->res.H == y.H && d->res.W == y.W && d->res.C == y.C,
                  "esf_conv_igemm_create: residual view must match the output view");

  IgemmOp* op = new (std::nothrow) IgemmOp();
  if (!op) return set_error(ESF_ERR_ARG, "out of host memory");
  IgemmParams& p = op->params;
  memset(&p, 0, sizeof(p));
  int kc, kchunks, n_tile, n_pad;
  esf_igemm_geometry(x.C, y.C, &kc, &kchunks, &n_tile, &n_pad);
  p.kc = kc;
  p.kchunks = kchunks;
  p.n_tile = n_tile;
  p.n_tiles = n_pad / n_tile;
  p.num_taps = num_taps;
  choose_box(Wo, Ho, To, clip_weights ? 1 : y.B, &p.bw, &p.bh, &p.bt, &p.bb);
  p.b_clip_rows = clip_weights ? n_pad : 0;
  // A T-halo mode for k x 1 x 1 layers (one activation tile of bt + kT - 1 planes per chunk, shared by the kT taps)
  // was measured on the fast pathway's thirteen 3x1x1 layers of the headline workload and removed: correct, and the
  // L2 -> smem bytes drop from 3x to 1.2x, but 1.25 ms -> 1.88 ms in total (64->16 @56^2: 0.42 -> 0.58 ms): with
  // bw * bh = 8 only 112 of the 128 MMA rows are outputs and T = 32 splits into 14 + 14 + 4 planes, i.e. 1.5x the
  // tiles -- these layers are bound by the per-tile hand-over (accumulator, epilogue, store), not by the activation loads.
  p.tw = cdiv(Wo, p.bw);
  p.th = cdiv(Ho, p.bh);
  p.tt = cdiv(To, p.bt);
  p.tb = cdiv(y.B, p.bb);
  p.rows = p.bw * p.bh * p.bt * p.bb;
  const long long ntiles = (long long)p.tw * p.th * p.tt * p.tb * p.n_tiles;
  if (ntiles > 0x7fffffffLL) {
    delete op;
    return set_error(ESF_ERR_ARG, "too many tiles");
  }
  p.num_tiles = (int)ntiles;
  p.ncb = 1;
  p.a_cb_stride = p.out_cb_w = 0;
  const int row_bytes = kc * 2;
  p.a_bytes = p.rows * row_bytes;
  p.b_bytes = n_tile * row_bytes;
  p.b_stride = (p.b_bytes + 1023) & ~1023u;
  p.sbo = 8 * row_bytes;
  p.layout_type = row_bytes == 128 ? 2 : (row_bytes == 64 ? 4 : 6);
  p.bias = d->bias;
  p.act = d->act;
  p.has_res = d->res.ptr != nullptr;
  p.out_f32 = d->out_dtype == ESF_F32;
  p.f16 = x.dtype == ESF_F16;
  const CUtensorMapDataType dt16 = p.f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  const int oes = p.out_f32 ? 4 : 2;
  p.slab_cols = std::min(n_tile, 128 / oes);
  const int out_row_bytes = p.slab_cols * oes;
  p.out_swz = out_row_bytes == 128 ? 7 : (out_row_bytes == 64 ? 3 : 1);
  p.res_bytes = p.rows * p.slab_cols * 2;

  plan_smem(p, &op->smem_bytes);

  // ---- activation maps: one per distinct stride phase; taps carry the per-map coordinate offsets
  struct Phase {
    int pt, ph, pw;
  };
  std::vector<Phase> phases;
  int rc = ESF_OK;
  int tap_i = 0;
  for (int it = 0; it < d->kT && rc == ESF_OK; ++it)
    for (int ih = 0; ih < d->kH && rc == ESF_OK; ++ih)
      for (int iw = 0; iw < d->kW && rc == ESF_OK; ++iw, ++tap_i) {
        const int ot = it * d->dT - d->pT, oh = ih * d->dH - d->pH, ow = iw * d->dW - d->pW;
        const int qt = floordiv(ot, d->sT), qh = floordiv(oh, d->sH), qw = floordiv(ow, d->sW);
        const Phase ph = {ot - qt * d->sT, oh - qh * d->sH, ow - qw * d->sW};
        int idx = -1;
        for (size_t i = 0; i < phases.size(); ++i)
          if (phases[i].pt == ph.pt && phases[i].ph == ph.ph && phases[i].pw == ph.pw) idx = (int)i;
        if (idx < 0) {
          if ((int)phases.size() == kMaxAMaps) {
            rc = set_error(ESF_ERR_UNSUPPORTED, "conv needs more than %d stride phases", kMaxAMaps);
            break;
          }
          idx = (int)phases.size();
          phases.push_back(ph);
          // phase view: element (c, w', h', t', b) = x[b, sT*t'+pt, sH*h'+ph, sW*w'+pw, c]
          const int Tp = ph.pt < x.T ? cdiv(x.T - ph.pt, d->sT) : 0;
          const int Hp = ph.ph < x.H ? cdiv(x.H - ph.ph, d->sH) : 0;
          const int Wp = ph.pw < x.W ? cdiv(x.W - ph.pw, d->sW) : 0;
          if (Tp <= 0 || Hp <= 0 || Wp <= 0) {
            rc = set_error(ESF_ERR_UNSUPPORTED, "empty stride phase (input smaller than the stride)");
            break;
          }
          char* base = static_cast<char*>(x.ptr) + 2 * (ph.pt * x.sT + ph.ph * x.sH + ph.pw * x.sW);
          rc = encode_act_map(&p.a_maps[idx], dt16, 2, base, x.C, Wp, Hp, Tp, x.B,
                              x.sW * d->sW, x.sH * d->sH, x.sT * d->sT, x.sB, kc, p.bw, p.bh, p.bt, p.bb,
                              swizzle_for_row_bytes(row_bytes), "activation");
        }
        p.taps[tap_i] = make_int4(idx, qw, qh, qt);
      }
  // unused map slots alias map 0 so that the kernel parameter block is fully initialised
  if (rc == ESF_OK)
    for (int i = (int)phases.size(); i < kMaxAMaps; ++i) p.a_maps[i] = p.a_maps[0];

  // ---- packed weights: 2-D (K, n_pad), box (kc, n_tile)
  if (rc == ESF_OK) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) rc = set_error(ESF_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
    else {
      const cuuint64_t K = (cuuint64_t)num_taps * kchunks * kc;
      cuuint64_t dims[2] = {K, (cuuint64_t)n_pad * (clip_weights ? y.B : 1)};
      cuuint64_t strides[1] = {K * 2};
      cuuint32_t box[2] = {(cuuint32_t)kc, (cuuint32_t)n_tile};
      cuuint32_t estr[2] = {1, 1};
      CUresult r = enc(&p.b_map, dt16, 2, const_cast<void*>(d->w), dims, strides, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for_row_bytes(row_bytes),
                       CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) rc = set_error(ESF_ERR_CUDA, "cuTensorMapEncodeTiled(weights) failed with %d", (int)r);
    }
  }
  // ---- output (+ residual) maps: box (slab_cols, bw, bh, bt, bb)
  if (rc == ESF_OK)
    rc = encode_act_map(&p.out_map, p.out_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : dt16, oes,
                        y.ptr, y.C, y.W, y.H, y.T, y.B, y.sW, y.sH, y.sT, y.sB, p.slab_cols, p.bw, p.bh, p.bt, p.bb,
                        swizzle_for_row_bytes(out_row_bytes), "output");
  if (rc == ESF_OK) {
    if (p.has_res)
      rc = encode_act_map(&p.res_map, dt16, 2, d->res.ptr, d->res.C, d->res.W, d->res.H,
                          d->res.T, d->res.B, d->res.sW, d->res.sH, d->res.sT, d->res.sB, p.slab_cols, p.bw, p.bh, p.bt,
                          p.bb, swizzle_for_row_bytes(out_row_bytes), "residual");
    else
      p.res_map = p.out_map;
  }
  if (rc == ESF_OK) rc = finish_op(op);
  if (rc != ESF_OK) {
    delete op;
    return rc;
  }
  *out = op;
  return ESF_OK;
}

// ---- stem as a banded GEMM -------------------------------------------------------------------------------------
// A Cin = 3 stem conv has K = kT*kH*kW*3 with no 16-byte-aligned contiguous run to feed the tensor cores.  Instead,
// for a block of WB = 8 consecutive output columns the (kW, Cin) taps are folded into a banded weight matrix:
//   row   m = (b, t, ho)            one output row position, for a fixed block wb of 8 output columns
//   col   n = (i, co)               i = 0..7 output column inside the block, co output channel   (N = 8 * Cout)
//   k       = (kt, kh, j)           j = 0..63 indexes the contiguous run of ((8-1)*sW + kW) * Cin <= 64 input
//                                   elements of input row (t+kt-pT, sH*ho+kh-pH) that the block reads
//   Wb[n][k] = w[co][c][kt][kh][kw] with (w_in, c) = divmod(j, Cin), kw = w_in - sW*i   (zero outside the band)
// so every (kt,kh) tap is one 128 B-row TMA box of the packed channels-last clip (esf_stem_pack: BF16, left zero
// pad so that block starts are 16 B aligned) and the output tile (8*Cout contiguous BF16 per row) is one TMA store.
// ~1/3 of the MACs hit structural zeros of the band; that is the price of running a 3-channel conv at tensor speed.
constexpr int kStemWB = 8;

extern "C" int esf_stem_geometry(int32_t W, int32_t Cin, int32_t kW, int32_t sW, int32_t pW, int32_t* pitch,
                                 int32_t* lpad, int32_t* window) {
  ESF_CHECK_ARG(W > 0 && Cin > 0 && kW > 0 && sW > 0 && pW >= 0, "esf_stem_geometry: bad argument");
  const int win = ((kStemWB - 1) * sW + kW) * Cin;
  if (win > 64) return set_error(ESF_ERR_UNSUPPORTED, "stem window of %d elements exceeds one 64-element K chunk", win);
  if ((kStemWB * sW * Cin) % 8 != 0)
    return set_error(ESF_ERR_UNSUPPORTED, "stem block stride %d elements is not 16-byte aligned", kStemWB * sW * Cin);
  const int Wo = (W + 2 * pW - kW) / sW + 1;
  const int ncb = cdiv(Wo, kStemWB);
  const int lp = pW * Cin;
  int pt = std::max(lp + W * Cin, kStemWB * sW * Cin * (ncb - 1) + 64);
  pt = (pt + 7) & ~7;
  if (pitch) *pitch = pt;
  if (lpad) *lpad = lp;
  if (window) *window = win;
  return ESF_OK;
}

extern "C" int esf_stem_igemm_create(const void* xp, int32_t B, int32_t Cin, int32_t T, int32_t H, int32_t W,
                                     int32_t pitch, const void* w_band, const float* bias_tiled, int32_t Cout,
                                     int32_t kT, int32_t kH, int32_t kW, int32_t sH, int32_t sW, int32_t pT, int32_t pH,
                                     int32_t pW, int32_t act, const esf_view* y, esf_op** out) {
  ESF_CHECK_ARG(xp && w_band && bias_tiled && view_ok(y) && out, "esf_stem_igemm_create: null/bad argument");
  // an FP32 output view: raw accumulators of one of the three split products of the FP32-accurate plan; the operands
  // (packed rows, band weights) are then FP16
  ESF_CHECK_ARG(is16(y->dtype) || y->dtype == ESF_F32, "esf_stem_igemm_create: output must be BF16, F16 or F32");
  int pt_expected = 0, lpad = 0, win = 0;
  int rc = esf_stem_geometry(W, Cin, kW, sW, pW, &pt_expected, &lpad, &win);
  if (rc != ESF_OK) return rc;
  ESF_CHECK_ARG(pitch == pt_expected, "esf_stem_igemm_create: pitch %d != esf_stem_geometry pitch %d", pitch, pt_expected);
  const int To = T + 2 * pT - kT + 1;
  const int Ho = (H + 2 * pH - kH) / sH + 1;
  const int Wo = (W + 2 * pW - kW) / sW + 1;
  ESF_CHECK_ARG(y->B == B && y->T == To && y->H == Ho && y->W == Wo && y->C == Cout && y->sW == Cout,
                "esf_stem_igemm_create: output must be a dense (B,%d,%d,%d,%d) channels-last tensor", To, Ho, Wo, Cout);
  if (Wo % kStemWB != 0)
    return set_error(ESF_ERR_UNSUPPORTED, "banded stem needs an output width that is a multiple of %d (got %d)", kStemWB, Wo);
  const int num_taps = kT * kH;
  ESF_CHECK_ARG(num_taps <= kMaxTaps, "esf_stem_igemm_create: %d (kT*kH) taps > %d", num_taps, kMaxTaps);

  IgemmOp* op = new (std::nothrow) IgemmOp();
  if (!op) return set_error(ESF_ERR_ARG, "out of host memory");
  IgemmParams& p = op->params;
  memset(&p, 0, sizeof(p));
  const int N = kStemWB * Cout;
  int kc, kchunks, n_tile, n_pad;
  esf_igemm_geometry(64, N, &kc, &kchunks, &n_tile, &n_pad);
  p.kc = 64, p.kchunks = 1, p.n_tile = n_tile, p.n_tiles = n_pad / n_tile, p.num_taps = num_taps;
  choose_box(1, Ho, To, B, &p.bw, &p.bh, &p.bt, &p.bb);
  // A T-halo mode (the kT taps of one kh sharing ONE activation tile of (bt + kT - 1) planes x 8 rows -- 7 tile loads
  // per M tile instead of 35 for the 5x7x7 stem) was measured and removed: bit-correct, 4x fewer L2 -> smem bytes, but
  // 1.20 -> 1.36 ms: the stem is not bound by its 11.6 TB/s of smem fill either.  140 MMAs of 128 x 64 x 16 per tile
  // take ~100 cycles each instead of 32 -- the serial wait / issue / commit loop of the MMA warp per 4-MMA k-block is
  // the limit, and the halo adds a barrier to it.
  p.tw = 1, p.th = cdiv(Ho, p.bh), p.tt = cdiv(To, p.bt), p.tb = cdiv(B, p.bb);
  p.rows = p.bw * p.bh * p.bt * p.bb;
  p.ncb = cdiv(Wo, kStemWB);
  p.a_cb_stride = kStemWB * sW * Cin;
  p.out_cb_w = 1;
  const long long ntiles = (long long)p.ncb * p.th * p.tt * p.tb * p.n_tiles;
  if (ntiles > 0x7fffffffLL) {
    delete op;
    return set_error(ESF_ERR_ARG, "too many tiles");
  }
  p.num_tiles = (int)ntiles;
  p.a_bytes = p.rows * 128, p.b_bytes = n_tile * 128, p.b_stride = (p.b_bytes + 1023) & ~1023u;
  p.sbo = 1024, p.layout_type = 2;
  p.bias = bias_tiled, p.act = act, p.has_res = 0, p.out_f32 = y->dtype == ESF_F32;
  p.f16 = y->dtype == ESF_F16 || y->dtype == ESF_F32;
  const CUtensorMapDataType dt16 = p.f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  const int oes = p.out_f32 ? 4 : 2;
  p.slab_cols = std::min(n_tile, 128 / oes);
  const int out_row_bytes = p.slab_cols * oes;
  p.out_swz = out_row_bytes == 128 ? 7 : (out_row_bytes == 64 ? 3 : 1);
  p.res_bytes = 0;
  plan_smem(p, &op->smem_bytes);

  // one activation map per row phase of the H stride
  int phase_map[8];
  for (int i = 0; i < 8; ++i) phase_map[i] = -1;
  int nmaps = 0;
  for (int it = 0; it < kT && rc == ESF_OK; ++it)
    for (int ih = 0; ih < kH && rc == ESF_OK; ++ih) {
      const int tap_i = it * kH + ih;   // (kt, kh) as packed in the weights
      const int oh = ih - pH;
      const int qh = floordiv(oh, sH);
      const int ph = oh - qh * sH;
      if (ph >= 8 || sH > 8) {
        rc = set_error(ESF_ERR_UNSUPPORTED, "stem H stride > 8");
        break;
      }
      if (phase_map[ph] < 0) {
        const int Hp = ph < H ? cdiv(H - ph, sH) : 0;
        if (Hp <= 0) {
          rc = set_error(ESF_ERR_UNSUPPORTED, "empty stride phase");
          break;
        }
        char* base = static_cast<char*>(const_cast<void*>(xp)) + 2LL * ph * pitch;
        rc = encode_act_map(&p.a_maps[nmaps], dt16, 2, base, pitch, 1, Hp, T, B,
                            (int64_t)sH * pitch, (int64_t)sH * pitch, (int64_t)H * pitch, (int64_t)T * H * pitch, 64,
                            1, p.bh, p.bt, p.bb, CU_TENSOR_MAP_SWIZZLE_128B, "stem activation");
        phase_map[ph] = nmaps++;
      }
      p.taps[tap_i] = make_int4(phase_map[ph], 0, qh, it - pT);
    }
  if (rc == ESF_OK)
    for (int i = nmaps; i < kMaxAMaps; ++i) p.a_maps[i] = p.a_maps[0];
  if (rc == ESF_OK) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) rc = set_error(ESF_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
    else {
      const cuuint64_t K = (cuuint64_t)num_taps * 64;
      cuuint64_t dims[2] = {K, (cuuint64_t)n_pad};
      cuuint64_t strides[1] = {K * 2};
      cuuint32_t box[2] = {64, (cuuint32_t)n_tile};
      cuuint32_t estr[2] = {1, 1};
      CUresult r = enc(&p.b_map, dt16, 2, const_cast<void*>(w_band), dims, strides, box,
                       estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                       CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) rc = set_error(ESF_ERR_CUDA, "cuTensorMapEncodeTiled(stem weights) failed with %d", (int)r);
    }
  }
  if (rc == ESF_OK)
    // dims (8*Cout, Wo/8, Ho, To, B): the column block is the W coordinate, so a tile wider than 8*Cout is clipped
    rc = encode_act_map(&p.out_map, p.out_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : dt16, oes, y->ptr,
                        (int64_t)kStemWB * Cout, Wo / kStemWB, Ho, To, B, (int64_t)kStemWB * Cout, y->sH, y->sT, y->sB,
                        p.slab_cols, 1, p.bh, p.bt, p.bb, swizzle_for_row_bytes(out_row_bytes), "stem output");
  if (rc == ESF_OK) {
    p.res_map = p.out_map;
    rc = finish_op(op);
  }
  if (rc != ESF_OK) {
    delete op;
    return rc;
  }
  *out = op;
  return ESF_OK;
}

// ---- temporal-band stem: the kT x kH x kW stem with the TIME taps folded into N ------------------------------------
// Why: the banded stem above is bound by the shared-memory port, not by the tensor pipe (DESIGN.md 3.2).  Its N is one
// block of output columns (64), so every 16 KB activation tile is filled once and read once by MMAs that also re-read
// 8 KB of weights each: 1 680 KB per 128 x 8 outputs through a 128 B/clk port.  Here
//   * an M tile (128 rows = bh output rows x bb clips, one block of WB output columns) STAYS on its SM while the input
//     frames g = 0 .. T-1 stream through: the tile of input frame g and row tap kh is loaded once and multiplied by
//     the weights of ALL kT time taps at once -- N = (kT output frames) x (WB x Cout) -- so the A read of an MMA is
//     amortised over kT times more columns and the tile is fetched kT times less often;
//   * output frame t accumulates in its own TMEM slot (t mod nslots, NB = WB x Cout columns each; 512 columns = 16
//     slots of 32) from the kT input frames that touch it; a slot is published to the epilogue warps as soon as its last
//     input frame is done and is re-used nslots frames later -- the accumulators are a ring over time;
//   * the whole band matrix (kH tiles of [kT x NB rows][64]) is loaded ONCE per CTA and stays in shared memory.
// MMA of input frame g, tap kh, k-step ks:  D[slot(t_lo) ..][128 x cnt*NB] += A_g,kh[128 x 16] . Wb_kh[u_lo*NB ..]^T
// with t = g + pT - kT + 1 + u, weights of time tap kt = kT - 1 - u; split where the slot ring wraps and where a slot
// is written for the first time (accumulate flag off).
namespace esf {

constexpr int kTbThreads = 6 * 32;   // TMA producer, MMA issuer, 4 epilogue warps (one per TMEM lane quarter)
constexpr int kTbMaxKH = 8;
constexpr int kTbMaxStages = 8;
// Where the time of this kernel goes was measured with timing variants that switched parts of the work off (no MMAs, no
// tile loads, no epilogue, one k-step per tap, two alternating MMA issuers; profiles/r2_stem_tband.md).  They were
// compile-time instantiations because run-time switches in these loops are not free, and they were removed afterwards.

struct __align__(64) StemTbParams {
  CUtensorMap a_maps[kMaxAMaps];   // one per row phase of the H stride
  CUtensorMap b_map;
  int a_map_of_kh[kTbMaxKH], qh_of_kh[kTbMaxKH];
  int kT, kH, pT;
  int T, To, Ho, B;
  int bh, bb, th, tb, ncb, rows;
  int a_cb_stride;   // elements between the windows of consecutive column blocks
  int odd_shift;     // 1: the tile of an odd column block is loaded 16 B early (its rows then start on a 32 B sector) and
                     // its MMAs read from start address + 16 B
  int ksteps;        // 16-element K steps per tap
  int NB, nslots;    // columns per output-frame slot, slots in the ring (power of two)
  int stages;
  uint32_t a_bytes, b_tile_bytes;
  const float* bias;   // [NB] tiled (i, co)
  int act, f16;
  int out_f32;        // FP32 output (one of the three split products of the FP32-accurate plan): y counts floats
  __nv_bfloat16* y;
  long long ysB, ysT, ysH;
  int num_tiles;
};

// one k-step of a tap: the frames of segment 0 and, when the slot ring wraps inside the window, of segment 1
#define ESF_TB_KSTEP(ks)                                                                              \
  {                                                                                                   \
    umma_bf16_lohi(sd0, a_lo + 2 * (ks), desc_hi, b0 + 2 * (ks), desc_hi, si0, 1);                     \
    if (c1 > 0) umma_bf16_lohi(tmem_base, a_lo + 2 * (ks), desc_hi, b1 + 2 * (ks), desc_hi, si1, 1);   \
  }

template <int KSTEPS, bool F16>
__global__ void __launch_bounds__(kTbThreads, 1) stem_tband_kernel(const __grid_constant__ StemTbParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_b = smem;
  uint8_t* smem_a = smem_b + p.kH * p.b_tile_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_a + p.stages * kAStageBytes);
  uint64_t* a_full = bars;
  uint64_t* a_empty = a_full + kTbMaxStages;
  uint64_t* acc_full = a_empty + kTbMaxStages;   // [nslots <= 32]
  uint64_t* acc_free = acc_full + 32;
  uint64_t* b_full = acc_free + 32;
  uint64_t* tok = b_full + 1;          // [2] unused since the two-issuer timing variant was removed (layout kept)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tok + 2);
  float* bias_sh = reinterpret_cast<float*>(bars) + 256;   // [NB <= 64], 1 KB into the 2 KB barrier / bias area

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const int smask = p.nslots - 1;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&a_full[s], 1);
      mbar_init(&a_empty[s], 1);
    }
    for (int s = 0; s < p.nslots; ++s) {
      mbar_init(&acc_full[s], 1);
      mbar_init(&acc_free[s], 4);
    }
    mbar_init(b_full, 1);
    mbar_init(&tok[0], 1);
    mbar_init(&tok[1], 1);
    fence_barrier_init();
  }
  if (threadIdx.x >= 64 && threadIdx.x < 64 + p.NB) bias_sh[threadIdx.x - 64] = p.bias[threadIdx.x - 64];
  if (warp == 0 && lane == 0) {
    prefetch_tmap(&p.b_map);
    prefetch_tmap(&p.a_maps[0]);
    prefetch_tmap(&p.a_maps[1]);
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      mbar_arrive_expect_tx(b_full, p.kH * p.b_tile_bytes);
      for (int kh = 0; kh < p.kH; ++kh) tma_load_2d(smem_b + kh * p.b_tile_bytes, &p.b_map, b_full, kh * 64, 0);
    }
    __syncwarp();
    const int kH = p.kH, T = p.T, stages = p.stages;
    const uint32_t a_bytes = p.a_bytes;
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      const int cb = tile % p.ncb, m = tile / p.ncb;
      const int h0 = (m % p.th) * p.bh, b0 = (m / p.th) * p.bb, c0 = cb * p.a_cb_stride - ((cb & p.odd_shift) ? 8 : 0);
      for (int g = 0; g < T; ++g)
        for (int kh = 0; kh < kH; ++kh) {
          mbar_wait(&a_empty[stage], phase ^ 1, 51);
          if (elect_one()) {
            mbar_arrive_expect_tx(&a_full[stage], a_bytes);
            tma_load_5d(smem_a + stage * kAStageBytes, &p.a_maps[p.a_map_of_kh[kh]], &a_full[stage], c0, 0,
                        h0 + p.qh_of_kh[kh], g, b0);
          }
          __syncwarp();
          if (++stage == stages) {
            stage = 0;
            phase ^= 1;
          }
        }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    // The issuing thread is a serial instruction stream and a tap is only three or four MMAs: everything that depends
    // on the input frame alone -- D column, weight-row offset and instruction descriptor of each segment -- is computed
    // once per frame, the first tap of a frame (whose first k-step opens the new slot) is peeled off the tap loop, and
    // the k-step count is a template parameter.
    const uint32_t idesc0 = make_idesc_16(128, 0, F16);
    const uint32_t desc_hi = kmajor_desc_hi(1024, 2);
    const uint32_t a_lo0 = kmajor_desc_lo(smem_u32(smem_a)), b_lo0 = kmajor_desc_lo(smem_u32(smem_b));
    const uint32_t b_kh_step = p.b_tile_bytes >> 4, b_u_step = (uint32_t)(p.NB * 128) >> 4;
    const int kT = p.kT, kH = p.kH, pT = p.pT, T = p.T, To = p.To, NB = p.NB, nslots = p.nslots;
    const int stages = p.stages, num_tiles = p.num_tiles;
    const int back = kT - 1 - pT;   // output frame t is complete after input frame min(t + back, T - 1)
    mbar_wait(b_full, 0, 52);
    tc_fence_after();
    int stage = 0;
    uint32_t phase = 0, free_bits = 0;
    const int ncb = p.ncb, odd_shift = p.odd_shift;
    uint32_t a_rel = 0;    // stage * 1024: position of the current stage in the ring, in 16 B units
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const uint32_t a_base = a_lo0 + (((tile % ncb) & odd_shift) ? 1u : 0u);
      for (int g = 0; g < T; ++g) {
        const int t_base = g + pT - kT + 1;
        const int t_lo = max(t_base, 0), t_hi = min(g + pT, To - 1);
        const int new_lo = g == 0 ? 0 : g + pT;     // frames >= new_lo are written for the first time in this step
        for (int t = max(new_lo, t_lo); t <= t_hi; ++t) {   // their slots must have been drained by the epilogue
          const int s = t & smask;
          mbar_wait(&acc_free[s], ((free_bits >> s) & 1) ^ 1, 53);
          free_bits ^= 1u << s;
        }
        tc_fence_after();
        // segment = frames [a, a + n) in consecutive slots: (D address, weight-row offset in 16 B units, idesc)
        auto seg_d = [&](int a) { return tmem_base + (uint32_t)((a & smask) * NB); };
        auto seg_b = [&](int a) { return (uint32_t)(a - t_base) * b_u_step; };
        auto seg_i = [&](int n) { return idesc0 | ((uint32_t)((n * NB) >> 3) << 17); };
        // steady k-steps: [t_lo, t_hi], split where the slot ring wraps
        const int cnt = t_hi - t_lo + 1;
        const int c0 = min(cnt, nslots - (t_lo & smask)), c1 = cnt - c0;
        const uint32_t sd0 = seg_d(t_lo), sb0 = seg_b(t_lo), si0 = seg_i(c0);
        const uint32_t sb1 = seg_b(t_lo + c0), si1 = seg_i(c1);
        // first k-step of the frame: the frames below new_lo accumulate (same split), the new ones overwrite; the new
        // frames never straddle the wrap (frames 0 .. pT at g = 0, a single frame otherwise)
        const int old_cnt = max(min(new_lo - 1, t_hi) - t_lo + 1, 0);
        const int o0 = min(old_cnt, c0), o1 = old_cnt - o0;
        const int nw_lo = max(new_lo, t_lo), nw_cnt = t_hi - nw_lo + 1;
        const uint32_t oi0 = seg_i(o0), oi1 = seg_i(o1);
        const uint32_t nd = seg_d(nw_lo), nb = seg_b(nw_lo), ni = seg_i(nw_cnt);
        // frames completed by this input frame: t = g - back (and everything still open at the last input frame)
        const int done_lo = max(g == T - 1 ? t_lo : g - back, 0), done_hi = g == T - 1 ? t_hi : g - back;
        uint32_t b0 = b_lo0 + sb0, b1 = b_lo0 + sb1;
        // ---- tap kh = 0
        uint32_t a_lo = a_base + a_rel;
        mbar_wait(&a_full[stage], phase, 54);
        tc_fence_after();
        if (elect_one()) {
          if (o0 > 0) umma_bf16_lohi(sd0, a_lo, desc_hi, b0, desc_hi, oi0, 1);
          if (o1 > 0) umma_bf16_lohi(tmem_base, a_lo, desc_hi, b1, desc_hi, oi1, 1);
          if (nw_cnt > 0) umma_bf16_lohi(nd, a_lo, desc_hi, b_lo0 + nb, desc_hi, ni, 0);
          if (KSTEPS > 1) ESF_TB_KSTEP(1)
          if (KSTEPS > 2) ESF_TB_KSTEP(2)
          if (KSTEPS > 3) ESF_TB_KSTEP(3)
          umma_commit(&a_empty[stage]);
          if (kH == 1)
            for (int t = done_lo; t <= done_hi; ++t) umma_commit(&acc_full[t & smask]);
        }
        __syncwarp();
        a_rel += kAStageBytes >> 4;
        if (++stage == stages) stage = 0, phase ^= 1, a_rel = 0;
        // ---- taps kh = 1 .. kH - 1
        for (int kh = 1; kh < kH; ++kh) {
          b0 += b_kh_step, b1 += b_kh_step;
          a_lo = a_base + a_rel;
          mbar_wait(&a_full[stage], phase, 54);
          tc_fence_after();
          if (elect_one()) {
            ESF_TB_KSTEP(0)
            if (KSTEPS > 1) ESF_TB_KSTEP(1)
            if (KSTEPS > 2) ESF_TB_KSTEP(2)
            if (KSTEPS > 3) ESF_TB_KSTEP(3)
            umma_commit(&a_empty[stage]);
            if (kh == kH - 1)
              for (int t = done_lo; t <= done_hi; ++t) umma_commit(&acc_full[t & smask]);
          }
          __syncwarp();
          a_rel += kAStageBytes >> 4;
          if (++stage == stages) stage = 0, phase ^= 1, a_rel = 0;
        }
      }
    }
  } else if (warp >= 2 && warp <= 5) {
    // ------------------------------------------------------------------ epilogue: one warp per TMEM lane quarter
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
    const int NB = p.NB, To = p.To, act = p.act;
    const long long ysT = p.ysT;
    uint32_t full_bits = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      const int cb = tile % p.ncb, m = tile / p.ncb;
      const int ho = (m % p.th) * p.bh + r % p.bh, b = (m / p.th) * p.bb + r / p.bh;
      const bool valid = r < p.rows && ho < p.Ho && b < p.B;
      const long long yoff = b * p.ysB + ho * p.ysH + (long long)cb * NB;
      __nv_bfloat16* yrow = p.y + yoff;
      float* yrow32 = reinterpret_cast<float*>(p.y) + yoff;
      const bool out_f32 = p.out_f32 != 0;
      for (int t = 0; t < To; ++t, yrow += ysT, yrow32 += ysT) {
        const int s = t & smask;
        mbar_wait(&acc_full[s], (full_bits >> s) & 1, 55);
        full_bits ^= 1u << s;
        tc_fence_after();
        for (int c0 = 0; c0 < NB; c0 += 16) {
          float v[16];
          tmem_ld16(lane_addr + s * NB + c0, v);
          if (valid && out_f32) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float4 bv = *reinterpret_cast<const float4*>(bias_sh + c0 + 4 * i);
              *reinterpret_cast<float4*>(yrow32 + c0 + 4 * i) =
                  make_float4(apply_act(v[4 * i] + bv.x, act), apply_act(v[4 * i + 1] + bv.y, act),
                              apply_act(v[4 * i + 2] + bv.z, act), apply_act(v[4 * i + 3] + bv.w, act));
            }
          } else if (valid) {
            uint32_t pk[8];
#pragma unroll
            for (int i = 0; i < 4; ++i) {       // the bias vector comes from shared memory, four columns per load
              const float4 bv = *reinterpret_cast<const float4*>(bias_sh + c0 + 4 * i);
              pk[2 * i] = pack16x2(apply_act(v[4 * i] + bv.x, act), apply_act(v[4 * i + 1] + bv.y, act), F16);
              pk[2 * i + 1] = pack16x2(apply_act(v[4 * i + 2] + bv.z, act), apply_act(v[4 * i + 3] + bv.w, act), F16);
            }
            uint4* dst = reinterpret_cast<uint4*>(yrow + c0);
            dst[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            dst[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_free[s]);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

using StemTbKernel = void (*)(const StemTbParams);
static StemTbKernel stem_tband_fn(int ksteps, bool f16) {
  switch (ksteps * 2 + (f16 ? 1 : 0)) {
    case 2: return stem_tband_kernel<1, false>;
    case 3: return stem_tband_kernel<1, true>;
    case 4: return stem_tband_kernel<2, false>;
    case 5: return stem_tband_kernel<2, true>;
    case 6: return stem_tband_kernel<3, false>;
    case 7: return stem_tband_kernel<3, true>;
    case 8: return stem_tband_kernel<4, false>;
    default: return stem_tband_kernel<4, true>;
  }
}

}  // namespace esf

struct StemTbOp : esf_op {
  StemTbParams params;
  int grid = 0;
  int smem_bytes = 0;
  int launch(cudaStream_t stream) override {
    stem_tband_fn(params.ksteps, params.f16 != 0)<<<grid, kTbThreads, smem_bytes, stream>>>(params);
    return check_launch("stem_tband_kernel");
  }
};

// Width of the output-column block (WB) of the temporal-band stem for this geometry, 0 when it does not apply.
static int stem_tband_wb(int Cin, int Cout, int kT, int kH, int kW, int sW, int Wo) {
  if (kT < 2 || kT > 8 || kH > kTbMaxKH) return 0;
  const int cand[3] = {4, 8, 2};
  for (int i = 0; i < 3; ++i) {
    const int WB = cand[i];
    const int win = ((WB - 1) * sW + kW) * Cin, NB = WB * Cout;
    if (win > 64 || (WB * sW * Cin) % 8 != 0 || Wo % WB != 0) continue;
    if (NB != 16 && NB != 32 && NB != 64) continue;
    if (kT * NB > 256 || kTmemCols / NB < kT + 1) continue;
    const int b_bytes = kH * kT * NB * 128;
    if ((kSmemLimit - 1024 - 2048 - b_bytes) / kAStageBytes < 3) continue;
    return WB;
  }
  return 0;
}

extern "C" int esf_stem_tband_wb(int32_t W, int32_t Cin, int32_t Cout, int32_t kT, int32_t kH, int32_t kW, int32_t sW,
                                 int32_t pW) {
  if (W <= 0 || Cin <= 0 || Cout <= 0 || kW <= 0 || sW <= 0 || pW < 0) return 0;
  return stem_tband_wb(Cin, Cout, kT, kH, kW, sW, (W + 2 * pW - kW) / sW + 1);
}

extern "C" int esf_stem_tband_create(const void* xp, int32_t B, int32_t Cin, int32_t T, int32_t H, int32_t W,
                                     int32_t pitch, const void* w_band, const float* bias_tiled, int32_t Cout,
                                     int32_t kT, int32_t kH, int32_t kW, int32_t sH, int32_t sW, int32_t pT, int32_t pH,
                                     int32_t pW, int32_t act, const esf_view* y, esf_op** out) {
  ESF_CHECK_ARG(xp && w_band && bias_tiled && view_ok(y) && out, "esf_stem_tband_create: null/bad argument");
  ESF_CHECK_ARG(is16(y->dtype) || y->dtype == ESF_F32, "esf_stem_tband_create: output must be BF16, F16 or F32");
  ESF_CHECK_ARG(pT >= 0 && pT < kT && sH >= 1 && sH <= 8, "esf_stem_tband_create: bad temporal padding / H stride");
  int pt_expected = 0, lpad = 0, win8 = 0;
  int rc = esf_stem_geometry(W, Cin, kW, sW, pW, &pt_expected, &lpad, &win8);
  if (rc != ESF_OK) return rc;
  ESF_CHECK_ARG(pitch == pt_expected, "esf_stem_tband_create: pitch %d != esf_stem_geometry pitch %d", pitch, pt_expected);
  const int To = T + 2 * pT - kT + 1;
  const int Ho = (H + 2 * pH - kH) / sH + 1;
  const int Wo = (W + 2 * pW - kW) / sW + 1;
  ESF_CHECK_ARG(To >= 1 && y->B == B && y->T == To && y->H == Ho && y->W == Wo && y->C == Cout && y->sW == Cout,
                "esf_stem_tband_create: output must be a dense (B,%d,%d,%d,%d) channels-last tensor", To, Ho, Wo, Cout);
  const int WB = stem_tband_wb(Cin, Cout, kT, kH, kW, sW, Wo);
  if (WB == 0) return set_error(ESF_ERR_UNSUPPORTED, "temporal-band stem does not apply to this geometry");
  const int oes = y->dtype == ESF_F32 ? 4 : 2;
  ESF_CHECK_ARG((reinterpret_cast<uintptr_t>(y->ptr) & 15) == 0 && (y->sH * oes) % 16 == 0 && (y->sT * oes) % 16 == 0 &&
                    (y->sB * oes) % 16 == 0, "esf_stem_tband_create: output rows must be 16-byte aligned");

  StemTbOp* op = new (std::nothrow) StemTbOp();
  if (!op) return set_error(ESF_ERR_ARG, "out of host memory");
  StemTbParams& p = op->params;
  memset(&p, 0, sizeof(p));
  p.kT = kT, p.kH = kH, p.pT = pT, p.T = T, p.To = To, p.Ho = Ho, p.B = B;
  p.NB = WB * Cout, p.nslots = kTmemCols / p.NB;
  if (p.nslots > 32) p.nslots = 32;
  const int win = ((WB - 1) * sW + kW) * Cin;
  p.ksteps = cdiv(win, 16);
  p.ncb = Wo / WB, p.a_cb_stride = WB * sW * Cin;
  // TMA fetches rows that start in the middle of a 32 B sector at about 2/3 of the rate (measured: tile loads alone 0.59
  // -> 0.41 ms).  With Cin = 3 the blocks are 48 B apart, so every odd block is loaded 16 B early when the widened
  // window still fits the same number of k-steps
  p.odd_shift = ((p.a_cb_stride * 2) % 32 == 16 && win + 8 <= p.ksteps * 16) ? 1 : 0;
  int bw = 1, bt = 1;
  choose_box(1, Ho, 1, B, &bw, &p.bh, &bt, &p.bb);
  p.th = cdiv(Ho, p.bh), p.tb = cdiv(B, p.bb), p.rows = p.bh * p.bb;
  const long long ntiles = (long long)p.ncb * p.th * p.tb;
  if (ntiles > 0x7fffffffLL) {
    delete op;
    return set_error(ESF_ERR_ARG, "too many tiles");
  }
  p.num_tiles = (int)ntiles;
  p.a_bytes = p.rows * 128, p.b_tile_bytes = kT * p.NB * 128;
  // an FP32 output view: raw accumulators of one of the three split products of the FP32-accurate plan (FP16 operands)
  p.bias = bias_tiled, p.act = act, p.f16 = y->dtype == ESF_F16 || y->dtype == ESF_F32, p.out_f32 = y->dtype == ESF_F32;
  p.y = static_cast<__nv_bfloat16*>(y->ptr), p.ysB = y->sB, p.ysT = y->sT, p.ysH = y->sH;
  p.stages = std::min(kTbMaxStages, (kSmemLimit - 1024 - 2048 - (int)(kH * p.b_tile_bytes)) / kAStageBytes);
  op->smem_bytes = 1024 + 2048 + kH * p.b_tile_bytes + p.stages * kAStageBytes;   // alignment slack, barriers + bias
  const CUtensorMapDataType dt16 = p.f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;

  int phase_map[8];
  for (int i = 0; i < 8; ++i) phase_map[i] = -1;
  int nmaps = 0;
  for (int ih = 0; ih < kH && rc == ESF_OK; ++ih) {
    const int oh = ih - pH;
    const int qh = floordiv(oh, sH);
    const int ph = oh - qh * sH;
    if (phase_map[ph] < 0) {
      const int Hp = ph < H ? cdiv(H - ph, sH) : 0;
      if (Hp <= 0) {
        rc = set_error(ESF_ERR_UNSUPPORTED, "empty stride phase");
        break;
      }
      char* base = static_cast<char*>(const_cast<void*>(xp)) + 2LL * ph * pitch;
      rc = encode_act_map(&p.a_maps[nmaps], dt16, 2, base, pitch, 1, Hp, T, B, (int64_t)sH * pitch, (int64_t)sH * pitch,
                          (int64_t)H * pitch, (int64_t)T * H * pitch, 64, 1, p.bh, 1, p.bb, CU_TENSOR_MAP_SWIZZLE_128B,
                          "temporal-band stem activation");
      phase_map[ph] = nmaps++;
    }
    p.a_map_of_kh[ih] = phase_map[ph], p.qh_of_kh[ih] = qh;
  }
  if (rc == ESF_OK)
    for (int i = nmaps; i < kMaxAMaps; ++i) p.a_maps[i] = p.a_maps[0];
  if (rc == ESF_OK) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) rc = set_error(ESF_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
    else {
      const cuuint64_t K = (cuuint64_t)kH * 64;
      cuuint64_t dims[2] = {K, (cuuint64_t)(kT * p.NB)};
      cuuint64_t strides[1] = {K * 2};
      cuuint32_t box[2] = {64, (cuuint32_t)(kT * p.NB)};
      cuuint32_t estr[2] = {1, 1};
      CUresult r = enc(&p.b_map, dt16, 2, const_cast<void*>(w_band), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                       CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) rc = set_error(ESF_ERR_CUDA, "cuTensorMapEncodeTiled(temporal-band weights) failed with %d", (int)r);
    }
  }
  if (rc == ESF_OK) {
    const int sms = num_sms();
    if (sms <= 0) rc = set_error(ESF_ERR_CUDA, "no CUDA device");
    else {
      op->grid = std::min(p.num_tiles, sms);
      static unsigned char attr_done[kMaxDevices] = {0};
      unsigned char* slot = device_slot(attr_done);
      if (!slot || !*slot) {
        for (int ks = 1; ks <= 4 && rc == ESF_OK; ++ks)
          for (int f = 0; f < 2 && rc == ESF_OK; ++f) {
            cudaError_t e = cudaFuncSetAttribute(stem_tband_fn(ks, f != 0), cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit);
            if (e != cudaSuccess) rc = set_error(ESF_ERR_CUDA, "cudaFuncSetAttribute(stem_tband) failed: %s", cudaGetErrorString(e));
          }
        if (rc == ESF_OK && slot) *slot = 1;
      }
    }
  }
  if (rc != ESF_OK) {
    delete op;
    return rc;
  }
  *out = op;
  return ESF_OK;
}

// ---- W-folded dense conv for thin layers (C_in <= 32) ------------------------------------------------------------
// A (B,T,H,W,C) activation with C = 8..32 gives TMA rows of 16..64 bytes and MMA tiles of N = 8..32: both far below
// what the hardware wants.  Folding a block of WB output columns into the GEMM's N and the ((WB-1)*sW + kW) input
// columns it reads into the GEMM's K (the same banded / block-diagonal weight trick as the stem) turns every tap into
// 128-byte rows and N into WB * Cout (up to 256).  The extra MACs hit structural zeros; these layers are HBM bound.
extern "C" int esf_conv_wfold_create(const esf_conv_desc* d, int32_t WB, esf_op** out) {
  ESF_CHECK_ARG(d && out && WB >= 1, "esf_conv_wfold_create: null/bad argument");
  ESF_CHECK_ARG(view_ok(&d->x) && view_ok(&d->y) && d->w && d->bias, "esf_conv_wfold_create: bad views/weights");
  const esf_view& x = d->x;
  const esf_view& y = d->y;
  ESF_CHECK_ARG(d->groups == 1 && d->sT == 1 && d->dT == 1 && d->dH == 1 && d->dW == 1,
                "esf_conv_wfold_create: needs groups 1, temporal stride 1, no dilation");
  ESF_CHECK_ARG(is16(x.dtype) && y.dtype == x.dtype && d->out_dtype == x.dtype,
                "esf_conv_wfold_create: 16-bit input and output of the same format");
  ESF_CHECK_ARG(x.sW == x.C && x.C % 8 == 0, "esf_conv_wfold_create: input must be dense in (W,C) with C %% 8 == 0");
  const int To = x.T + 2 * d->pT - d->kT + 1;
  const int Ho = (x.H + 2 * d->pH - d->kH) / d->sH + 1;
  const int Wo = (x.W + 2 * d->pW - d->kW) / d->sW + 1;
  ESF_CHECK_ARG(y.B == x.B && y.T == To && y.H == Ho && y.W == Wo, "esf_conv_wfold_create: output shape mismatch");
  ESF_CHECK_ARG(Wo % WB == 0, "esf_conv_wfold_create: Wo %% WB != 0");
  const int C = x.C, Cout = y.C;
  const int win = ((WB - 1) * d->sW + d->kW) * C;
  ESF_CHECK_ARG(win <= 128, "esf_conv_wfold_create: window of %d elements > 128", win);
  const int kchunks = cdiv(win, 64);
  const int N = WB * Cout;
  ESF_CHECK_ARG(N <= 256, "esf_conv_wfold_create: WB * Cout = %d > 256", N);
  const int num_taps = d->kT * d->kH;
  ESF_CHECK_ARG(num_taps <= kMaxTaps, "esf_conv_wfold_create: too many taps");
  const bool y_dense = y.sW == y.C;
  const bool has_res = d->res.ptr != nullptr;
  const bool r_dense = has_res && d->res.sW == d->res.C;
  if (has_res)
    ESF_CHECK_ARG(d->res.dtype == x.dtype && d->res.B == y.B && d->res.T == y.T && d->res.H == y.H && d->res.W == y.W &&
                      d->res.C == y.C, "esf_conv_wfold_create: residual view must match the output view");

  IgemmOp* op = new (std::nothrow) IgemmOp();
  if (!op) return set_error(ESF_ERR_ARG, "out of host memory");
  IgemmParams& p = op->params;
  memset(&p, 0, sizeof(p));
  int kc, kch, n_tile, n_pad;
  esf_igemm_geometry(64, N, &kc, &kch, &n_tile, &n_pad);
  const bool need_pow2 = !y_dense || (has_res && !r_dense);
  if (need_pow2 && (n_pad != N || (Cout < 64 ? 64 % Cout : Cout % 64) != 0 || N % std::min(64, N) != 0)) {
    delete op;
    return set_error(ESF_ERR_UNSUPPORTED, "esf_conv_wfold_create: sliced output needs WB*Cout a power of two");
  }
  p.kc = 64, p.kchunks = kchunks, p.n_tile = n_tile, p.n_tiles = n_pad / n_tile, p.num_taps = num_taps;
  choose_box(1, Ho, To, y.B, &p.bw, &p.bh, &p.bt, &p.bb);
  p.tw = 1, p.th = cdiv(Ho, p.bh), p.tt = cdiv(To, p.bt), p.tb = cdiv(y.B, p.bb);
  p.rows = p.bw * p.bh * p.bt * p.bb;
  p.ncb = Wo / WB;
  p.a_cb_stride = WB * d->sW * C;
  p.a_c_base = -d->pW * C;
  p.fold_wb = WB;
  const long long ntiles = (long long)p.ncb * p.th * p.tt * p.tb * p.n_tiles;
  if (ntiles > 0x7fffffffLL) {
    delete op;
    return set_error(ESF_ERR_ARG, "too many tiles");
  }
  p.num_tiles = (int)ntiles;
  p.a_bytes = p.rows * 128, p.b_bytes = n_tile * 128, p.b_stride = (p.b_bytes + 1023) & ~1023u;
  p.sbo = 1024, p.layout_type = 2;
  p.bias = d->bias, p.act = d->act, p.has_res = has_res, p.out_f32 = 0;
  p.f16 = x.dtype == ESF_F16;
  const CUtensorMapDataType dt16 = p.f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  p.slab_cols = std::min(n_tile, 64);
  const int out_row_bytes = p.slab_cols * 2;
  // A sliced destination is written through a (c, w) box whose smem image is the plain row-major slab: no swizzle.
  // (Measured: declaring the 128 B swizzle on such a box does NOT reproduce the dense-row image -- the swizzle atom
  // follows the box's inner extent, not just the shared-memory address -- so the staging writes of this mode keep
  // their 8-way bank conflicts.)
  const bool slice_mode = need_pow2;
  const bool plain = slice_mode;
  p.out_swz = plain ? 0 : (out_row_bytes == 128 ? 7 : (out_row_bytes == 64 ? 3 : 1));
  const CUtensorMapSwizzle out_sw = plain ? CU_TENSOR_MAP_SWIZZLE_NONE : swizzle_for_row_bytes(out_row_bytes);
  p.res_bytes = p.rows * p.slab_cols * 2;
  plan_smem(p, &op->smem_bytes);

  int rc = ESF_OK;
  int phase_map[8];
  for (int i = 0; i < 8; ++i) phase_map[i] = -1;
  int nmaps = 0, tap_i = 0;
  for (int it = 0; it < d->kT && rc == ESF_OK; ++it)
    for (int ih = 0; ih < d->kH && rc == ESF_OK; ++ih, ++tap_i) {
      const int oh = ih - d->pH;
      const int qh = floordiv(oh, d->sH);
      const int ph = oh - qh * d->sH;
      if (ph >= 8) {
        rc = set_error(ESF_ERR_UNSUPPORTED, "H stride > 8");
        break;
      }
      if (phase_map[ph] < 0) {
        const int Hp = ph < x.H ? cdiv(x.H - ph, d->sH) : 0;
        if (Hp <= 0) {
          rc = set_error(ESF_ERR_UNSUPPORTED, "empty stride phase");
          break;
        }
        char* base = static_cast<char*>(x.ptr) + 2LL * ph * x.sH;
        rc = encode_act_map(&p.a_maps[nmaps], dt16, 2, base, (int64_t)x.W * C, 1, Hp, x.T, x.B, x.sH * d->sH,
                            x.sH * d->sH, x.sT, x.sB, 64, 1, p.bh, p.bt, p.bb, CU_TENSOR_MAP_SWIZZLE_128B,
                            "folded activation");
        phase_map[ph] = nmaps++;
      }
      p.taps[tap_i] = make_int4(phase_map[ph], 0, qh, it - d->pT);
    }
  if (rc == ESF_OK)
    for (int i = nmaps; i < kMaxAMaps; ++i) p.a_maps[i] = p.a_maps[0];
  if (rc == ESF_OK) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) rc = set_error(ESF_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
    else {
      const cuuint64_t K = (cuuint64_t)num_taps * kchunks * 64;
      cuuint64_t dims[2] = {K, (cuuint64_t)n_pad};
      cuuint64_t strides[1] = {K * 2};
      cuuint32_t box[2] = {64, (cuuint32_t)n_tile};
      cuuint32_t estr[2] = {1, 1};
      CUresult r = enc(&p.b_map, dt16, 2, const_cast<void*>(d->w), dims, strides, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) rc = set_error(ESF_ERR_CUDA, "cuTensorMapEncodeTiled(folded weights) failed with %d", (int)r);
    }
  }
  auto encode_io = [&](CUtensorMap* m, const esf_view& v, bool dense, int* fold_cout, const char* what) {
    if (dense && !slice_mode) {   // rows of WB*Cout contiguous elements: (WB*Cout, Wo/WB, Ho, To, B)
      *fold_cout = 0;
      return encode_act_map(m, dt16, 2, v.ptr, (int64_t)N, Wo / WB, Ho, To, v.B, (int64_t)N, v.sH, v.sT, v.sB,
                            p.slab_cols, 1, p.bh, p.bt, p.bb, out_sw, what);
    }
    *fold_cout = Cout;       // (Cout, Wo, Ho, To, B) with a (c, w) box per 64-column slab
    const int cbox = std::min(Cout, p.slab_cols), wbox = std::max(1, p.slab_cols / Cout);
    return encode_act_map(m, dt16, 2, v.ptr, Cout, Wo, Ho, To, v.B, v.sW, v.sH, v.sT, v.sB, cbox, wbox, p.bh, p.bt, p.bb,
                          out_sw, what);
  };
  if (rc == ESF_OK) rc = encode_io(&p.out_map, y, y_dense, &p.out_fold_cout, "folded output");
  if (rc == ESF_OK) {
    if (has_res) rc = encode_io(&p.res_map, d->res, r_dense, &p.res_fold_cout, "folded residual");
    else p.res_map = p.out_map;
  }
  p.out_cb_w = 1;
  if (rc == ESF_OK) rc = finish_op(op);
  if (rc != ESF_OK) {
    delete op;
    return rc;
  }
  *out = op;
  return ESF_OK;
}

extern "C" int esf_op_launch(esf_op* op, void* stream) {
  ESF_CHECK_ARG(op, "esf_op_launch: null op");
  return op->launch(static_cast<cudaStream_t>(stream));
}

extern "C" void esf_op_destroy(esf_op* op) { delete op; }
