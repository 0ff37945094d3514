// Tensor-core GEMM and implicit-GEMM 3x3 convolution for sm_100a.
//
//   out[M,N] = epilogue( A[M,K] * W[N,K]^T )          bf16 x bf16 -> fp32 (TMEM) -> bf16/fp32
//
// Replaces the nn.Linear / nn.Conv2d call sites of the reference UNet/ControlNet/TESTR
// (terediff/model/unet.py:152,170-197; attention.py:181-186,206,301-331;
//  controlnet.py:168-175,318-321; testr/adet/modeling/testr/models.py:76-88).
//
// Design (one persistent CTA per SM, 256 threads, warp-specialised):
//   warp 0      TMA producer : cp.async.bulk.tensor -> 128B-swizzled smem ring (STAGES deep)
//   warp 1      MMA issuer   : one thread issues tcgen05.mma (M=128, N=BN, K=16) x4 per k-block
//   warp 2      TMEM owner   : allocates 2 x BN fp32 accumulator columns (double buffered)
//   warps 4..7  epilogue     : tcgen05.ld 32x32b -> bias / timestep-row add / activation /
//                              residual -> 16-byte stores; overlaps the next tile's mainloop
// For the 3x3 convolution the A operand is never materialised: the producer walks the
// 9 filter taps x Cin/64 channel blocks and issues a 4-D TMA box load on the NHWC
// activation with shifted (w,h) start coordinates; TMA's out-of-bounds zero fill implements
// the padding and elementStrides implements stride 2.
#include <atomic>
#include <cstdlib>

#include "../../include/tair_b200.h"
#include <cstring>
#include <map>
#include <mutex>

#include "common.cuh"

namespace tair {

extern std::atomic<int64_t> g_launch_count;

namespace {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int GEMM_THREADS = 384;  // warp 0 TMA, 1 MMA, 2 TMEM alloc, 3 spare, 4..11 epilogue
constexpr uint32_t A_BYTES = BM * BK * 2;
// epilogue staging: each of the 8 epilogue warps owns one 32-row x 64-column bf16 sub-tile (4 KB) written in the
// 128B-swizzled layout of a TMA store box, so the global write is one cp.async.bulk.tensor per sub-tile
constexpr int EPI_WARPS = 8;
constexpr uint32_t STG_BYTES_PER_WARP = 32 * 128;
constexpr uint32_t STG_BYTES = EPI_WARPS * STG_BYTES_PER_WARP;

struct GemmParams {
  int M, N, K;
  int tiles_m, tiles_n, num_kb;
  int conv;        // 0 plain, 1 conv3x3
  int kb_per_tap;  // Cin / 64
  int Ho, Wo, stride, pad;
  int vec_out, vec_res, vec_rg, vec_bias;
  int tma_store;  // bf16 output eligible for the TMA-store epilogue
  int stages;     // depth of the operand ring and number of epilogue staging buffers per warp (1 or 2): chosen per launch
  int stg_bufs;   // (pick_staging) - a second staging buffer costs ring stages, which only short K loops can spare
  int epi_mode;   // TMA-store epilogue variant: 0 lean (bias / activation only), 1 lean + one prefetched bf16 row-add
                  // stream (residual, or bf16 row-group rows), 2 generic (fp32 row groups, folded LayerNorm, GEGLU, tails)
  int splits;      // split-K: each tile is computed by `splits` CTAs over kb_split k-blocks each; fp32 partials go to
  int kb_split;    // rows [split*M, split*M + M) of the (workspace) output, a second kernel reduces + applies the epilogue
  int dbg;  // bring-up probes (TAIR_GEMM_DEBUG): 1 skip global stores, 2 skip the epilogue body, 4 / 8 load B / A only for the first tile
  tair_epilogue epi;
};

template <int BN>
struct Cfg {
  static constexpr uint32_t B_BYTES = BN * BK * 2;
  static constexpr uint32_t STAGE_BYTES = A_BYTES + B_BYTES;
  // ring depth with `bufs` staging buffers per epilogue warp inside the 227 KB opt-in limit per CTA
  static constexpr int stages_for(int bufs) {
    const int fit = (int)((232448u - 1280u - (uint32_t)bufs * STG_BYTES) / STAGE_BYTES);
    return fit > 8 ? 8 : fit;
  }
  static constexpr uint32_t smem_for(int bufs) {
    return (uint32_t)stages_for(bufs) * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/ + (uint32_t)bufs * STG_BYTES;
  }
  static constexpr uint32_t TMEM_COLS = (2 * BN <= 128) ? 128 : ((2 * BN <= 256) ? 256 : 512);
  static constexpr uint32_t SMEM_MAX = smem_for(1) > smem_for(2) ? smem_for(1) : smem_for(2);
};

template <int ACT>
__device__ __forceinline__ float apply_act(float x) {
  if constexpr (ACT == TAIR_ACT_GELU) return gelu_f(x);
  else if constexpr (ACT == TAIR_ACT_SILU) return silu_f(x);
  else if constexpr (ACT == TAIR_ACT_RELU) return fmaxf(x, 0.f);
  else return x;
}

// one thread: NC consecutive output columns [n, n+NC) of row m, values in v[]
template <int NC>
__device__ __forceinline__ void epi_finish_store(const GemmParams& p, int m, int n, int ncols_total,
                                                 float (&v)[NC]) {
  const tair_epilogue& e = p.epi;
  const bool full = (n + NC <= ncols_total);
  if (e.residual != nullptr) {
    const __nv_bfloat16* rp = reinterpret_cast<const __nv_bfloat16*>(e.residual) + (int64_t)m * e.ldr + n;
    if (full && p.vec_res) {
#pragma unroll
      for (int j = 0; j < NC; j += 8) {
        uint4 q = __ldg(reinterpret_cast<const uint4*>(rp + j));
        float2 f0 = unpack_bf16(q.x), f1 = unpack_bf16(q.y), f2 = unpack_bf16(q.z), f3 = unpack_bf16(q.w);
        v[j + 0] += f0.x; v[j + 1] += f0.y; v[j + 2] += f1.x; v[j + 3] += f1.y;
        v[j + 4] += f2.x; v[j + 5] += f2.y; v[j + 6] += f3.x; v[j + 7] += f3.y;
      }
    } else {
#pragma unroll
      for (int j = 0; j < NC; ++j)
        if (n + j < ncols_total) v[j] += __bfloat162float(rp[j]);
    }
  }
  if (e.out_fp32) {
    float* op = reinterpret_cast<float*>(e.out) + (int64_t)m * e.ldc + n;
    if (full && p.vec_out) {
#pragma unroll
      for (int j = 0; j < NC; j += 4)
        *reinterpret_cast<float4*>(op + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
    } else {
#pragma unroll
      for (int j = 0; j < NC; ++j)
        if (n + j < ncols_total) op[j] = v[j];
    }
  } else {
    __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(e.out) + (int64_t)m * e.ldc + n;
    if (full && p.vec_out) {
#pragma unroll
      for (int j = 0; j < NC; j += 8) {
        uint4 q;
        q.x = pack_bf16(v[j + 0], v[j + 1]);
        q.y = pack_bf16(v[j + 2], v[j + 3]);
        q.z = pack_bf16(v[j + 4], v[j + 5]);
        q.w = pack_bf16(v[j + 6], v[j + 7]);
        *reinterpret_cast<uint4*>(op + j) = q;
      }
    } else {
#pragma unroll
      for (int j = 0; j < NC; ++j)
        if (n + j < ncols_total) op[j] = __float2bfloat16(v[j]);
    }
  }
}

// Drain one 128 x BN accumulator tile: this thread owns output row m (TMEM lane = row in tile).
// Templated on the activation so that each executed path is a compact straight-line loop
// (a runtime switch per element blew the instruction cache and throttled the epilogue ~10x).
template <int BN, int ACT>
__device__ __forceinline__ void epilogue_tile(const GemmParams& p, int m, int tn, bool row_ok, uint32_t taddr) {
  const tair_epilogue& e = p.epi;
      const float* rg = nullptr;
      if (e.rowgroup != nullptr && row_ok)
        rg = reinterpret_cast<const float*>(e.rowgroup) + (int64_t)(e.rows_per_group > 0 ? m / e.rows_per_group : m % (-e.rows_per_group)) * e.ldg;
      // folded LayerNorm: acc' = rstd * (acc - mean * colsum[n]) = acc * ln_r + ln_c * colsum[n]
      float ln_r = 1.f, ln_c = 0.f;
      const float* lcs = e.ln_row_stats != nullptr ? e.ln_col_sum : nullptr;
      if (lcs != nullptr && row_ok) {
        const float2 st = __ldg(reinterpret_cast<const float2*>(e.ln_row_stats) + m);
        ln_r = st.y;
        ln_c = -st.x * st.y;
      }

      if constexpr (ACT == TAIR_ACT_GEGLU) {
        constexpr int HALF = BN / 2;
        const int nout_total = p.N / 2;
#pragma unroll 1
        for (int c = 0; c < HALF; c += 16) {
          uint32_t rv[16], rgt[16];
          tmem_ld_32x16(taddr + c, rv);
          tmem_ld_32x16(taddr + HALF + c, rgt);
          tmem_ld_wait();
          if (row_ok) {
            float v[16];
            const int nv = tn * BN + c;          // row index (in the interleaved W) of the value part
            const int ng = tn * BN + HALF + c;   // ... and of the gate part
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              float a = __uint_as_float(rv[j]);
              float g = __uint_as_float(rgt[j]);
              if (lcs != nullptr) {
                a = fmaf(a, ln_r, ln_c * __ldg(lcs + nv + j));
                g = fmaf(g, ln_r, ln_c * __ldg(lcs + ng + j));
              }
              if (e.bias != nullptr) {
                a += __ldg(e.bias + nv + j);
                g += __ldg(e.bias + ng + j);
              }
              v[j] = a * gelu_tanh_f(g);
            }
            epi_finish_store<16>(p, m, tn * HALF + c, nout_total, v);
          }
        }
      } else {
#pragma unroll 1
        for (int c = 0; c < BN; c += 32) {
          uint32_t r[32];
          tmem_ld_32x32(taddr + c, r);
          tmem_ld_wait();
          const int n = tn * BN + c;
          if (row_ok && n < p.N) {
            float v[32];
            if (n + 32 <= p.N) {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                float a = __uint_as_float(r[j]);
                if (lcs != nullptr) a = fmaf(a, ln_r, ln_c * __ldg(lcs + n + j));
                if (e.bias != nullptr) a += __ldg(e.bias + n + j);
                if (rg != nullptr) a += __ldg(rg + n + j);
                v[j] = apply_act<ACT>(a);
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                float a = __uint_as_float(r[j]);
                if (n + j < p.N) {
                  if (lcs != nullptr) a = fmaf(a, ln_r, ln_c * __ldg(lcs + n + j));
                  if (e.bias != nullptr) a += __ldg(e.bias + n + j);
                  if (rg != nullptr) a += __ldg(rg + n + j);
                }
                v[j] = apply_act<ACT>(a);
              }
            }
            epi_finish_store<32>(p, m, n, p.N, v);
          }
        }
      }
}

// TMA-store epilogue (bf16 output).  Eight warps: warp e drains TMEM lane quadrant (e & 3) for the 64-column
// sub-tiles s with (s & 1) == (e >> 2).  Per sub-tile: tcgen05.ld (thread = output row) -> bias / row add /
// activation / residual -> bf16 -> swizzled smem -> one cp.async.bulk.tensor store (rows >= M and columns >= N are
// clipped by the hardware).  History: direct thread-per-row stores and a smem row-copy variant were both bound by
// the single epilogue warp per scheduler executing ~1000 dependent address/LSU instructions per tile (ncu source
// page, profiles/round1_summary.md); the bulk store removes that code entirely.
template <int BN, int ACT>
__device__ __forceinline__ void epilogue_tile_tma(const GemmParams& p, const CUtensorMap* tmC64,
                                                  const CUtensorMap* tmC32, int m0q, int tn, int half, int lane,
                                                  uint32_t taddr, uint8_t* stg0, uint32_t tempty_bar_addr,
                                                  bool remote_arrive, uint32_t tfull_bar_addr, uint32_t tfull_phase,
                                                  uint32_t& stg_sel) {
  const tair_epilogue& e = p.epi;
  constexpr bool GEGLU = (ACT == TAIR_ACT_GEGLU);
  constexpr int NT = GEGLU ? BN / 2 : BN;      // output columns produced by this tile
  constexpr int NSUB = (NT + 63) / 64;
  const int n_total = GEGLU ? p.N / 2 : p.N;
  const int n_out0 = tn * NT;
  const int m = m0q + lane;
  const bool row_ok = m < p.M;
  const float* rg = nullptr;
  if (!GEGLU && e.rowgroup != nullptr && row_ok)
    rg = reinterpret_cast<const float*>(e.rowgroup) + (int64_t)(e.rows_per_group > 0 ? m / e.rows_per_group : m % (-e.rows_per_group)) * e.ldg;
  const __nv_bfloat16* resp = (e.residual != nullptr && row_ok)
                                  ? reinterpret_cast<const __nv_bfloat16*>(e.residual) + (int64_t)m * e.ldr : nullptr;
  // folded LayerNorm (tair_epilogue.ln_row_stats): acc' = rstd * (acc - mean * colsum[n]) = acc * ln_r + ln_c * colsum[n]
  float ln_r = 1.f, ln_c = 0.f;
  const float* lcs = e.ln_row_stats != nullptr ? e.ln_col_sum : nullptr;
  if (lcs != nullptr && row_ok) {
    const float2 st = __ldg(reinterpret_cast<const float2*>(e.ln_row_stats) + m);
    ln_r = st.y;
    ln_c = -st.x * st.y;
  }
  const int sw7 = lane & 7, sw3 = (lane >> 1) & 3;

  auto release = [&]() {  // tempty lives in the leader CTA of a pair when remote_arrive is set
    if (remote_arrive) mbar_arrive_cluster(tempty_bar_addr);
    else mbar_arrive(tempty_bar_addr);
  };
  // Residual rows are prefetched one 32-column group ahead, the first group even before the accumulator is complete:
  // a thread-per-row read issued at its point of use exposes a full L2/HBM round trip per group (the K=320
  // projections with a residual ran 50 us against 23 us without one; 42 us with the prefetch).  A variant that also
  // made the loads row-contiguous through the staging buffer needed 8 more live 16-byte registers and spilled.
  uint4 rpre[4] = {};
  auto res_vec_ok = [&](int n) { return resp != nullptr && p.vec_res && n + 32 <= n_total; };
  auto prefetch = [&](int n) {
    if (res_vec_ok(n)) {
#pragma unroll
      for (int q = 0; q < 4; ++q) rpre[q] = __ldg(reinterpret_cast<const uint4*>(resp + n + q * 8));
    }
  };
  if (half < NSUB) prefetch(n_out0 + half * 64);
  mbar_wait(tfull_bar_addr, tfull_phase);
  tc_fence_after();
  if (half >= NSUB) {  // nothing to drain for this warp (narrow tiles): just release the accumulator
    tc_fence_before();
    __syncwarp();
    if (lane == 0) release();
    return;
  }
#pragma unroll 1
  for (int s = half; s < NSUB; s += 2) {
    const int c0 = s * 64;
    const int ncol = (NT - c0) < 64 ? (NT - c0) : 64;  // 64, or 32 for the tail of BN = 160
    uint8_t* stg = stg0 + stg_sel * STG_BYTES;         // this warp's staging buffer for this sub-tile (1 or 2 of them)
    const uint32_t stg_u32 = smem_u32(stg);
    if (elect_one()) {   // the store that last used this buffer has left it
      if (p.stg_bufs == 2) tma_store_wait_read<1>();
      else tma_store_wait_read<0>();
    }
    __syncwarp();
#pragma unroll 1
    for (int g = 0; g < ncol; g += 32) {
      float v[32];
      const int n = n_out0 + c0 + g;                   // first output column of this 32-wide group
      uint4 rcur[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) rcur[q] = rpre[q];
      {
        const int n_next = (g + 32 < ncol) ? n + 32 : n_out0 + (s + 2) * 64;   // next group of this warp, if any
        if ((g + 32 < ncol) || (s + 2 < NSUB)) prefetch(n_next);
      }
      if constexpr (GEGLU) {
#pragma unroll
        for (int h2 = 0; h2 < 2; ++h2) {               // 16 columns at a time keeps register pressure down
          uint32_t rv[16], rgt[16];
          tmem_ld_32x16(taddr + c0 + g + h2 * 16, rv);
          tmem_ld_32x16(taddr + NT + c0 + g + h2 * 16, rgt);
          tmem_ld_wait();
          const int nv = tn * BN + c0 + g + h2 * 16, ng = nv + NT;   // rows of the tile-interleaved weight
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            float a = __uint_as_float(rv[j]), gt = __uint_as_float(rgt[j]);
            if (lcs != nullptr) {   // warp-uniform; the column sums are broadcast loads like the bias
              a = fmaf(a, ln_r, ln_c * __ldg(lcs + nv + j));
              gt = fmaf(gt, ln_r, ln_c * __ldg(lcs + ng + j));
            }
            if (e.bias != nullptr) { a += __ldg(e.bias + nv + j); gt += __ldg(e.bias + ng + j); }
            v[h2 * 16 + j] = a * gelu_tanh_f(gt);
          }
        }
      } else {
        uint32_t r[32];
        tmem_ld_32x32(taddr + c0 + g, r);
        tmem_ld_wait();
        if (n + 32 <= p.N) {
          if (lcs != nullptr) {   // folded LayerNorm first: it rescales the raw accumulator
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const float4 t = __ldg(reinterpret_cast<const float4*>(lcs + n) + q);
              r[q * 4 + 0] = __float_as_uint(fmaf(__uint_as_float(r[q * 4 + 0]), ln_r, ln_c * t.x));
              r[q * 4 + 1] = __float_as_uint(fmaf(__uint_as_float(r[q * 4 + 1]), ln_r, ln_c * t.y));
              r[q * 4 + 2] = __float_as_uint(fmaf(__uint_as_float(r[q * 4 + 2]), ln_r, ln_c * t.z));
              r[q * 4 + 3] = __float_as_uint(fmaf(__uint_as_float(r[q * 4 + 3]), ln_r, ln_c * t.w));
            }
          }
          if (rg != nullptr && p.vec_rg) {
            // per-row add rows (positional projections): every lane reads its own row, so use 16-byte loads
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const float4 t = __ldg(reinterpret_cast<const float4*>(rg + n) + q);
              r[q * 4 + 0] = __float_as_uint(__uint_as_float(r[q * 4 + 0]) + t.x);
              r[q * 4 + 1] = __float_as_uint(__uint_as_float(r[q * 4 + 1]) + t.y);
              r[q * 4 + 2] = __float_as_uint(__uint_as_float(r[q * 4 + 2]) + t.z);
              r[q * 4 + 3] = __float_as_uint(__uint_as_float(r[q * 4 + 3]) + t.w);
            }
          }
          // null checks hoisted out of the element loop: a predicated-off load still costs its address arithmetic
          // and issue slots (ncu: ~33 issued instructions per output element before, most of them @!P LEA / LDG)
          if (rg != nullptr && !p.vec_rg) {
#pragma unroll
            for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) + __ldg(rg + n + j));
          }
          if (e.bias != nullptr) {
            if (p.vec_bias) {   // 16-byte loads, the same address in every lane (broadcast)
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                const float4 t = __ldg(reinterpret_cast<const float4*>(e.bias + n) + q);
                r[q * 4 + 0] = __float_as_uint(__uint_as_float(r[q * 4 + 0]) + t.x);
                r[q * 4 + 1] = __float_as_uint(__uint_as_float(r[q * 4 + 1]) + t.y);
                r[q * 4 + 2] = __float_as_uint(__uint_as_float(r[q * 4 + 2]) + t.z);
                r[q * 4 + 3] = __float_as_uint(__uint_as_float(r[q * 4 + 3]) + t.w);
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) + __ldg(e.bias + n + j));
            }
          }
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = apply_act<ACT>(__uint_as_float(r[j]));
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            float a = __uint_as_float(r[j]);
            if (n + j < p.N) {
              if (lcs != nullptr) a = fmaf(a, ln_r, ln_c * __ldg(lcs + n + j));
              if (e.bias != nullptr) a += __ldg(e.bias + n + j);
              if (rg != nullptr) a += __ldg(rg + n + j);
            }
            v[j] = apply_act<ACT>(a);
          }
        }
      }
      if (resp != nullptr) {
        if (res_vec_ok(n)) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const uint4 w = rcur[q];
            const float2 b0 = unpack_bf16(w.x), b1 = unpack_bf16(w.y), b2 = unpack_bf16(w.z), b3 = unpack_bf16(w.w);
            v[q * 8 + 0] += b0.x; v[q * 8 + 1] += b0.y; v[q * 8 + 2] += b1.x; v[q * 8 + 3] += b1.y;
            v[q * 8 + 4] += b2.x; v[q * 8 + 5] += b2.y; v[q * 8 + 6] += b3.x; v[q * 8 + 7] += b3.y;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (n + j < n_total) v[j] += __bfloat162float(resp[n + j]);
        }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint4 w;
        w.x = pack_bf16(v[q * 8 + 0], v[q * 8 + 1]);
        w.y = pack_bf16(v[q * 8 + 2], v[q * 8 + 3]);
        w.z = pack_bf16(v[q * 8 + 4], v[q * 8 + 5]);
        w.w = pack_bf16(v[q * 8 + 6], v[q * 8 + 7]);
        // swizzled position of 16-byte chunk (g/8 + q) of this row inside the TMA box
        uint8_t* dst = (ncol == 64) ? stg + lane * 128 + ((((g >> 3) + q) ^ sw7) << 4)
                                    : stg + lane * 64 + ((q ^ sw3) << 4);
        *reinterpret_cast<uint4*>(dst) = w;
      }
    }
    const bool last = (s + 2 >= NSUB);
    if (last) tc_fence_before();   // all TMEM reads of this tile by this warp are done
    fence_async_smem();            // staging writes -> visible to the TMA (async proxy)
    __syncwarp();
    if (elect_one()) {  // same elected lane every time: bulk-group commit / wait are per-thread state
      if (last) release();
      if (!(p.dbg & 1)) {
        tma_store_2d(ncol == 64 ? tmC64 : tmC32, stg_u32, n_out0 + c0, m0q);
      }
      tma_store_commit();   // (an empty group under dbg & 1 keeps the wait_group accounting of two buffers right)
    }
    stg_sel ^= (uint32_t)(p.stg_bufs - 1);
  }
}

// Lean variants of the TMA-store epilogue.  The generic function above executes ~110 instructions per 32-column group
// even when it has nothing to add (register copies of the residual prefetch, predicated-off loads, 64-bit generic store
// addressing, null checks: ncu source page of 151552x1024x256, profiles/round2_summary.md), and an epilogue warp is one
// serial instruction stream: at K = 256 the drain of a tile then takes longer than its main loop.  Here every group is
// tcgen05.ld -> bias -> activation -> (row add) -> pack -> 4 x st.shared.v4, and the row-add stream (the bf16 residual
// row, or the bf16 row-group row of this output row) is prefetched a whole 64-column sub-tile ahead into registers that
// are refilled in place (no copies).  Host guarantees (pick_epi_mode): N % 32 == 0, 16-byte aligned bias / add rows.
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};\n" ::"r"(addr), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}

template <int BN, int ACT, bool ROWADD>
__device__ __forceinline__ void epilogue_tile_tma_lean(const GemmParams& p, const CUtensorMap* tmC64,
                                                       const CUtensorMap* tmC32, int m0q, int tn, int half, int lane,
                                                       uint32_t taddr, uint8_t* stg0, uint32_t tempty_bar_addr,
                                                       bool remote_arrive, uint32_t tfull_bar_addr,
                                                       uint32_t tfull_phase, uint32_t& stg_sel) {
  const tair_epilogue& e = p.epi;
  constexpr int NSUB = (BN + 63) / 64;
  const int n_out0 = tn * BN;
  const int m = m0q + lane;
  const __nv_bfloat16* addp = nullptr;   // this row's bf16 add stream (ROWADD)
  if constexpr (ROWADD) {
    if (m < p.M) {
      if (e.residual != nullptr)
        addp = reinterpret_cast<const __nv_bfloat16*>(e.residual) + (int64_t)m * e.ldr;
      else
        addp = reinterpret_cast<const __nv_bfloat16*>(e.rowgroup) +
               (int64_t)(e.rows_per_group > 0 ? m / e.rows_per_group : m % (-e.rows_per_group)) * e.ldg;
    }
  }
  const float* bias = e.bias;
  const uint32_t sw7 = lane & 7, sw3 = (lane >> 1) & 3;
  auto release = [&]() {
    if (remote_arrive) mbar_arrive_cluster(tempty_bar_addr);
    else mbar_arrive(tempty_bar_addr);
  };
  // add rows of the sub-tile being drained: ra0 = its first 32 columns, ra1 = its second 32 columns.  Two named arrays
  // and two lambdas on purpose: indexing one array through a pointer argument put it in local memory.
  uint4 ra0[4] = {}, ra1[4] = {};
  auto prefetch0 = [&](int n) {   // columns [n, n + 32) of this row, if they exist
    if (addp != nullptr && n < p.N) {
#pragma unroll
      for (int q = 0; q < 4; ++q) ra0[q] = __ldg(reinterpret_cast<const uint4*>(addp + n) + q);
    }
  };
  auto prefetch1 = [&](int n) {
    if (addp != nullptr && n < p.N) {
#pragma unroll
      for (int q = 0; q < 4; ++q) ra1[q] = __ldg(reinterpret_cast<const uint4*>(addp + n) + q);
    }
  };
  if constexpr (ROWADD) {
    if (half < NSUB) {
      prefetch0(n_out0 + half * 64);
      if (BN - half * 64 > 32) prefetch1(n_out0 + half * 64 + 32);
    }
  }
  mbar_wait(tfull_bar_addr, tfull_phase);
  tc_fence_after();
  if (half >= NSUB) {
    tc_fence_before();
    __syncwarp();
    if (lane == 0) release();
    return;
  }
  // bias -> activation -> row add on one 32-column group held in r[] (in place)
  auto finish = [&](uint32_t (&r)[32], int n, const uint4 (&ra)[4]) {
    if (n >= p.N) return;                  // warp-uniform: whole 32-column groups are inside or outside N
    if (bias != nullptr) {                 // the same address in every lane: broadcast loads, L1-resident after tile 0
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(bias + n) + q);
        r[q * 4 + 0] = __float_as_uint(__uint_as_float(r[q * 4 + 0]) + t.x);
        r[q * 4 + 1] = __float_as_uint(__uint_as_float(r[q * 4 + 1]) + t.y);
        r[q * 4 + 2] = __float_as_uint(__uint_as_float(r[q * 4 + 2]) + t.z);
        r[q * 4 + 3] = __float_as_uint(__uint_as_float(r[q * 4 + 3]) + t.w);
      }
    }
    if constexpr (ACT != TAIR_ACT_NONE) {
#pragma unroll
      for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(apply_act<ACT>(__uint_as_float(r[j])));
    }
    if constexpr (ROWADD) {
      if (addp != nullptr) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const uint4 w = ra[q];
          const float2 b0 = unpack_bf16(w.x), b1 = unpack_bf16(w.y), b2 = unpack_bf16(w.z), b3 = unpack_bf16(w.w);
          r[q * 8 + 0] = __float_as_uint(__uint_as_float(r[q * 8 + 0]) + b0.x);
          r[q * 8 + 1] = __float_as_uint(__uint_as_float(r[q * 8 + 1]) + b0.y);
          r[q * 8 + 2] = __float_as_uint(__uint_as_float(r[q * 8 + 2]) + b1.x);
          r[q * 8 + 3] = __float_as_uint(__uint_as_float(r[q * 8 + 3]) + b1.y);
          r[q * 8 + 4] = __float_as_uint(__uint_as_float(r[q * 8 + 4]) + b2.x);
          r[q * 8 + 5] = __float_as_uint(__uint_as_float(r[q * 8 + 5]) + b2.y);
          r[q * 8 + 6] = __float_as_uint(__uint_as_float(r[q * 8 + 6]) + b3.x);
          r[q * 8 + 7] = __float_as_uint(__uint_as_float(r[q * 8 + 7]) + b3.y);
        }
      }
    }
  };
  auto stage = [&](const uint32_t (&r)[32], uint32_t stg_u32, int g, int ncol) {   // pack + swizzled 16-byte stores
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint32_t dst = (ncol == 64) ? stg_u32 + lane * 128 + (((uint32_t)((g >> 3) + q) ^ sw7) << 4)
                                        : stg_u32 + lane * 64 + (((uint32_t)q ^ sw3) << 4);
      sts128(dst, pack_bf16(__uint_as_float(r[q * 8 + 0]), __uint_as_float(r[q * 8 + 1])),
             pack_bf16(__uint_as_float(r[q * 8 + 2]), __uint_as_float(r[q * 8 + 3])),
             pack_bf16(__uint_as_float(r[q * 8 + 4]), __uint_as_float(r[q * 8 + 5])),
             pack_bf16(__uint_as_float(r[q * 8 + 6]), __uint_as_float(r[q * 8 + 7])));
    }
  };
  auto wait_buffer = [&]() {   // the store that last used the staging buffer about to be written has left it
    if (elect_one()) {
      if (p.stg_bufs == 2) tma_store_wait_read<1>();
      else tma_store_wait_read<0>();
    }
  };
  auto store = [&](uint32_t stg_u32, int n, bool wide, bool last) {
    if (last) tc_fence_before();   // all TMEM reads of this tile by this warp are done
    fence_async_smem();            // staging writes -> visible to the TMA (async proxy)
    __syncwarp();
    if (elect_one()) {
      if (last) release();
      if (!(p.dbg & 1)) tma_store_2d(wide ? tmC64 : tmC32, stg_u32, n, m0q);
      tma_store_commit();          // (an empty group under dbg & 1 keeps the two-buffer wait_group accounting right)
    }
    stg_sel ^= (uint32_t)(p.stg_bufs - 1);
  };
  constexpr int NFULL = BN / 64;             // full 64-column sub-tiles; BN = 96 / 160 / 224 end with a 32-column one
  constexpr bool TAIL = (BN % 64) != 0;
#pragma unroll 1
  for (int s = half; s < NFULL; s += 2) {
    const bool more = s + 2 < NSUB;
    const int n = n_out0 + s * 64;
    const uint32_t stg_u32 = smem_u32(stg0 + stg_sel * STG_BYTES);
    // both halves of the sub-tile leave tensor memory together: one load latency per 64 columns instead of two
    uint32_t r0[32], r1[32];
    tmem_ld_32x32(taddr + s * 64, r0);
    tmem_ld_32x32(taddr + s * 64 + 32, r1);
    wait_buffer();
    tmem_ld_wait();
    __syncwarp();
    finish(r0, n, ra0);
    if constexpr (ROWADD) {   // refill the registers just consumed with the same group of this warp's next sub-tile
      if (more) prefetch0(n + 128);
    }
    stage(r0, stg_u32, 0, 64);
    finish(r1, n + 32, ra1);
    if constexpr (ROWADD) {
      if (more && s * 64 + 128 + 32 < BN) prefetch1(n + 128 + 32);
    }
    stage(r1, stg_u32, 32, 64);
    store(stg_u32, n, true, !more);
  }
  if constexpr (TAIL) {
    if ((NFULL & 1) == half) {   // the 32-column tail belongs to the warp whose sub-tile parity it continues
      const int n = n_out0 + NFULL * 64;
      const uint32_t stg_u32 = smem_u32(stg0 + stg_sel * STG_BYTES);
      uint32_t r0[32];
      tmem_ld_32x32(taddr + NFULL * 64, r0);
      wait_buffer();
      tmem_ld_wait();
      __syncwarp();
      finish(r0, n, ra0);
      stage(r0, stg_u32, 0, 32);
      store(stg_u32, n, false, true);
    }
  }
}

// activation x variant dispatch of the TMA-store epilogue (warp-uniform switch, one call per tile)
template <int BN>
__device__ __forceinline__ void epilogue_dispatch_tma(const GemmParams& p, const CUtensorMap* tmC64,
                                                      const CUtensorMap* tmC32, int m0q, int tn, int half, int lane,
                                                      uint32_t taddr, uint8_t* stg, uint32_t tempty_bar_addr,
                                                      bool remote_arrive, uint32_t tfull_bar_addr,
                                                      uint32_t tfull_phase, uint32_t& stg_sel) {
#define TAIR_EPI_ARGS p, tmC64, tmC32, m0q, tn, half, lane, taddr, stg, tempty_bar_addr, remote_arrive, tfull_bar_addr, tfull_phase, stg_sel
  const int act = p.epi.act;
  if (p.epi_mode == 0) {
    switch (act) {
      case TAIR_ACT_GELU: epilogue_tile_tma_lean<BN, TAIR_ACT_GELU, false>(TAIR_EPI_ARGS); return;
      case TAIR_ACT_SILU: epilogue_tile_tma_lean<BN, TAIR_ACT_SILU, false>(TAIR_EPI_ARGS); return;
      case TAIR_ACT_RELU: epilogue_tile_tma_lean<BN, TAIR_ACT_RELU, false>(TAIR_EPI_ARGS); return;
      default: epilogue_tile_tma_lean<BN, TAIR_ACT_NONE, false>(TAIR_EPI_ARGS); return;
    }
  }
  if (p.epi_mode == 1) {   // activation NONE only (pick_epi_mode)
    epilogue_tile_tma_lean<BN, TAIR_ACT_NONE, true>(TAIR_EPI_ARGS);
    return;
  }
  switch (act) {
    case TAIR_ACT_GEGLU: epilogue_tile_tma<BN, TAIR_ACT_GEGLU>(TAIR_EPI_ARGS); break;
    case TAIR_ACT_GELU: epilogue_tile_tma<BN, TAIR_ACT_GELU>(TAIR_EPI_ARGS); break;
    case TAIR_ACT_SILU: epilogue_tile_tma<BN, TAIR_ACT_SILU>(TAIR_EPI_ARGS); break;
    case TAIR_ACT_RELU: epilogue_tile_tma<BN, TAIR_ACT_RELU>(TAIR_EPI_ARGS); break;
    default: epilogue_tile_tma<BN, TAIR_ACT_NONE>(TAIR_EPI_ARGS); break;
  }
#undef TAIR_EPI_ARGS
}

template <int BN>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmC64, const __grid_constant__ CUtensorMap tmC32,
               const GemmParams p) {
  using C = Cfg<BN>;
  const int STAGES = p.stages;   // runtime: see GemmParams.stages / stg_bufs
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* stg_base = smem + STAGES * C::STAGE_BYTES;  // 1024-byte aligned (stage sizes are multiples of 1 KB)
  uint64_t* bars = reinterpret_cast<uint64_t*>(stg_base + p.stg_bufs * STG_BYTES);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const uint32_t smem_base = smem_u32(smem);
  const uint32_t bar_base = smem_u32(bars);
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 2 + a); };

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), EPI_WARPS);
    }
    mbar_fence_init();
  }
  if (warp == 2) {
    tmem_alloc(smem_u32(tmem_slot), C::TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
  pdl_grid_sync();   // set-up above overlaps the previous kernel's tail; no global memory is touched before this point

  const int num_tiles = p.tiles_m * p.tiles_n * p.splits;   // work items: (tile, K split)
  const int mn_tiles = p.tiles_m * p.tiles_n;

  if (warp == 0) {
    // The whole warp runs the loop and ONE elected lane issues: with warp-uniform control flow ptxas keeps the TMA /
    // UMMA operands in uniform registers; a `lane == 0` branch instead makes every UTMALDG / UTCHMMA a
    // vote-elect-R2UR "waterfall" loop (measured: 93-118 cycles per MMA issue vs 41-60, tools/probes/mma_shape_probe.cu)
    if (elect_one()) {
      tma_prefetch_desc(&tmA);
      tma_prefetch_desc(&tmB);
    }
    int stage = 0;
    uint32_t phase = 0;
    for (int work = blockIdx.x; work < num_tiles && !(p.dbg & 32); work += gridDim.x) {
      const int split = work / mn_tiles, tile = work - split * mn_tiles;
      const int tm = tile / p.tiles_n, tn = tile - tm * p.tiles_n;
      const int m0 = tm * BM, n0 = tn * BN;
      int img = 0, ho0 = 0, wo0 = 0;
      if (p.conv) {
        const int hw = p.Ho * p.Wo;
        img = m0 / hw;
        const int rem = m0 - img * hw;
        ho0 = rem / p.Wo;
        wo0 = rem - ho0 * p.Wo;
      }
      const int kb0 = split * p.kb_split;
      const int kb1 = (kb0 + p.kb_split < p.num_kb) ? kb0 + p.kb_split : p.num_kb;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(empty_bar(stage), phase ^ 1);
        const bool skip_b = (p.dbg & 4) && work != (int)blockIdx.x;
        const bool skip_a = (p.dbg & 8) && work != (int)blockIdx.x;
        const uint32_t a_dst = smem_base + stage * C::STAGE_BYTES;
        const uint32_t b_dst = a_dst + A_BYTES;
        int c0 = kb * BK, c1 = m0, c2 = 0, c3 = 0;
        if (p.conv) {
          const int tap = kb / p.kb_per_tap, cb = kb - tap * p.kb_per_tap;
          const int dy = tap / 3, dx = tap - dy * 3;
          c0 = cb * BK;
          c1 = wo0 * p.stride + dx - p.pad;
          c2 = ho0 * p.stride + dy - p.pad;
          c3 = img;
        }
        if (elect_one()) {
          mbar_expect_tx(full_bar(stage), (skip_b ? 0u : C::B_BYTES) + (skip_a ? 0u : A_BYTES));
          if (skip_a) {
          } else if (!p.conv) {
            tma_load_2d(a_dst, &tmA, full_bar(stage), c0, c1);
          } else {
            tma_load_4d(a_dst, &tmA, full_bar(stage), c0, c1, c2, c3);
          }
          if (!skip_b) tma_load_2d(b_dst, &tmB, full_bar(stage), kb * BK, n0);
        }
        __syncwarp();
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = umma_idesc_bf16(BM, BN, 0, 0);
    constexpr uint32_t desc_hi = umma_desc_hi_sw128(1024);
    const uint32_t a_lo0 = umma_desc_lo(smem_base, 16);
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int work = blockIdx.x; work < num_tiles; work += gridDim.x) {
      mbar_wait(tempty_bar(acc), acc_phase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * BN;
      const int kb0 = (work / mn_tiles) * p.kb_split;
      const int kb1 = (kb0 + p.kb_split < p.num_kb) ? kb0 + p.kb_split : p.num_kb;
      for (int kb = kb0; kb < kb1; ++kb) {
        if (!(p.dbg & 32)) {  // dbg 32 (probe): back-to-back MMA issue without the smem pipeline handshake
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
        }
        const uint32_t a_lo = a_lo0 + stage * (C::STAGE_BYTES >> 4);
        const uint32_t b_lo = a_lo + (A_BYTES >> 4);
        if (elect_one()) {
          umma_ss_lohi(d_tmem, a_lo, b_lo, desc_hi, idesc, kb != kb0);
#pragma unroll
          for (int k = 1; k < BK / 16; ++k)  // +32 bytes along K inside the 128-byte swizzle atom = +2 in the address field
            umma_ss_lohi(d_tmem, a_lo + 2 * k, b_lo + 2 * k, desc_hi, idesc, 1);
          if (!(p.dbg & 32)) umma_commit(empty_bar(stage));
        }
        __syncwarp();
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
      if (elect_one()) umma_commit(tfull_bar(acc));
      __syncwarp();
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  } else if (warp >= 4) {
    const int ew = warp - 4;
    const int quad = ew & 3;   // TMEM lane quadrant (== warp % 4, the only lanes this warp may read)
    const int half = ew >> 2;  // which alternate 64-column sub-tiles this warp drains
    const tair_epilogue& e = p.epi;
    uint8_t* stg = stg_base + ew * STG_BYTES_PER_WARP;   // buffer b of this warp: + b * STG_BYTES
    uint32_t stg_sel = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int work = blockIdx.x; work < num_tiles; work += gridDim.x) {
      const int split = work / mn_tiles, tile = work - split * mn_tiles;
      const int tm = tile / p.tiles_n, tn = tile - tm * p.tiles_n;
      const int m0q = tm * BM + quad * 32;
      if (!p.tma_store || (p.dbg & 2)) {   // the TMA-store epilogue waits itself, after its first residual prefetch
        mbar_wait(tfull_bar(acc), acc_phase);
        tc_fence_after();
      }
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + acc * BN;
      if ((p.dbg & 2) || (!p.tma_store && half == 1)) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(acc));
      } else if (p.tma_store) {
        epilogue_dispatch_tma<BN>(p, &tmC64, &tmC32, m0q, tn, half, lane, taddr, stg, tempty_bar(acc), false, tfull_bar(acc), acc_phase, stg_sel);
      } else {
        // fp32 / unaligned outputs (small heads): direct thread-per-row stores by the first four epilogue warps
        const bool row_ok = m0q + lane < p.M;
        const int m = m0q + lane + split * p.M;   // split-K partials: split s owns rows [s*M, s*M + M) of the workspace
        switch (e.act) {
          case TAIR_ACT_GEGLU: epilogue_tile<BN, TAIR_ACT_GEGLU>(p, m, tn, row_ok, taddr); break;
          case TAIR_ACT_GELU: epilogue_tile<BN, TAIR_ACT_GELU>(p, m, tn, row_ok, taddr); break;
          case TAIR_ACT_SILU: epilogue_tile<BN, TAIR_ACT_SILU>(p, m, tn, row_ok, taddr); break;
          case TAIR_ACT_RELU: epilogue_tile<BN, TAIR_ACT_RELU>(p, m, tn, row_ok, taddr); break;
          default: epilogue_tile<BN, TAIR_ACT_NONE>(p, m, tn, row_ok, taddr); break;
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(acc));
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (elect_one()) tma_store_wait_all<0>();  // bulk stores must have completed before the CTA releases its smem
    __syncwarp();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------------------
// 2-CTA variant: a CTA pair (one cluster, two SMs of a TPC) computes 256 x BN tiles with tcgen05.mma.cta_group::2.
// CTA r of the pair loads rows [128r, 128r+128) of A and rows [r*BN/2, (r+1)*BN/2) of the weight tile; the leader
// (rank 0) issues the MMAs for both, each SM accumulating its own 128 rows in its own TMEM.  Per-SM shared-memory
// operand traffic per K=16 step drops from 4 KB + BN*32 B to 4 KB + BN*16 B for twice the math, which takes the
// BN=160 convolution tiles off the smem-bandwidth limit (115 -> 82 B/clk).
template <int BN>
struct Cfg2 {
  static constexpr uint32_t B_BYTES = (BN / 2) * BK * 2;
  static constexpr uint32_t STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int stages_for(int bufs) {
    const int fit = (int)((232448u - 1280u - (uint32_t)bufs * STG_BYTES) / STAGE_BYTES);
    return fit > 8 ? 8 : fit;
  }
  static constexpr uint32_t smem_for(int bufs) {
    return (uint32_t)stages_for(bufs) * STAGE_BYTES + 1024 + 256 + (uint32_t)bufs * STG_BYTES;
  }
  static constexpr uint32_t TMEM_COLS = (2 * BN <= 128) ? 128 : ((2 * BN <= 256) ? 256 : 512);
  static constexpr uint32_t SMEM_MAX = smem_for(1) > smem_for(2) ? smem_for(1) : smem_for(2);
};

template <int BN>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                const __grid_constant__ CUtensorMap tmC64, const __grid_constant__ CUtensorMap tmC32,
                const GemmParams p) {
  using C = Cfg2<BN>;
  const int STAGES = p.stages;   // runtime: see GemmParams.stages / stg_bufs
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* stg_base = smem + STAGES * C::STAGE_BYTES;  // 1024-byte aligned (stage sizes are multiples of 1 KB)
  uint64_t* bars = reinterpret_cast<uint64_t*>(stg_base + p.stg_bufs * STG_BYTES);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const uint32_t smem_base = smem_u32(smem);
  const uint32_t bar_base = smem_u32(bars);
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 2 + a); };

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);   // leader only is waited on; one arrive.expect_tx covering both CTAs' bytes
      mbar_init(empty_bar(s), 1);  // MMA commit is multicast to both CTAs
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 2 * EPI_WARPS);  // leader's copy collects the epilogue warps of both CTAs
    }
    mbar_fence_init();
  }
  if (warp == 2) {
    tmem_alloc_2cta(smem_u32(tmem_slot), C::TMEM_COLS);
    tmem_relinquish_2cta();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
  pdl_grid_sync();

  const int tiles_m2 = (p.tiles_m + 1) >> 1;  // 256-row tiles
  const int num_tiles = tiles_m2 * p.tiles_n;

  if (warp == 0) {
    if (elect_one()) {
      tma_prefetch_desc(&tmA);
      tma_prefetch_desc(&tmB);
    }
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = pair; tile < num_tiles; tile += num_pairs) {
      const int tm2 = tile / p.tiles_n, tn = tile - tm2 * p.tiles_n;
      const int m0 = (tm2 * 2 + (int)rank) * BM, n0 = tn * BN + (int)rank * (BN / 2);
      int img = 0, ho0 = 0, wo0 = 0;
      if (p.conv) {
        const int hw = p.Ho * p.Wo;
        img = m0 / hw;
        const int rem = m0 - img * hw;
        ho0 = rem / p.Wo;
        wo0 = rem - ho0 * p.Wo;
      }
      for (int kb = 0; kb < p.num_kb; ++kb) {
        mbar_wait(empty_bar(stage), phase ^ 1);
        const uint32_t full_leader = mapa_shared(full_bar(stage), 0);
        const bool skip_b = (p.dbg & 4) && tile != pair;
        const bool skip_a = (p.dbg & 8) && tile != pair;
        const uint32_t a_dst = smem_base + stage * C::STAGE_BYTES;
        const uint32_t b_dst = a_dst + A_BYTES;
        int c0 = kb * BK, c1 = m0, c2 = 0, c3 = 0;
        if (p.conv) {
          const int tap = kb / p.kb_per_tap, cb = kb - tap * p.kb_per_tap;
          const int dy = tap / 3, dx = tap - dy * 3;
          c0 = cb * BK;
          c1 = wo0 * p.stride + dx - p.pad;
          c2 = ho0 * p.stride + dy - p.pad;
          c3 = img;
        }
        if (elect_one()) {
          if (leader) mbar_expect_tx(full_bar(stage), 2 * ((skip_b ? 0u : C::B_BYTES) + (skip_a ? 0u : A_BYTES)));
          if (skip_a) {
          } else if (!p.conv) {
            tma_load_2d_2cta(a_dst, &tmA, full_leader, c0, c1);
          } else {
            tma_load_4d_2cta(a_dst, &tmA, full_leader, c0, c1, c2, c3);
          }
          if (!skip_b) tma_load_2d_2cta(b_dst, &tmB, full_leader, kb * BK, n0);
        }
        __syncwarp();
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    if (leader) {
      constexpr uint32_t idesc = umma_idesc_bf16(2 * BM, BN, 0, 0);
      constexpr uint32_t desc_hi = umma_desc_hi_sw128(1024);
      const uint32_t a_lo0 = umma_desc_lo(smem_base, 16);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = pair; tile < num_tiles; tile += num_pairs) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint32_t a_lo = a_lo0 + stage * (C::STAGE_BYTES >> 4);
          const uint32_t b_lo = a_lo + (A_BYTES >> 4);
          if (elect_one()) {
            umma_ss_2cta_lohi(d_tmem, a_lo, b_lo, desc_hi, idesc, kb != 0);
#pragma unroll
            for (int k = 1; k < BK / 16; ++k)
              umma_ss_2cta_lohi(d_tmem, a_lo + 2 * k, b_lo + 2 * k, desc_hi, idesc, 1);
            umma_commit_2cta(empty_bar(stage), 3);
          }
          __syncwarp();
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (elect_one()) umma_commit_2cta(tfull_bar(acc), 3);
        __syncwarp();
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else if (warp >= 4) {
    const int ew = warp - 4;
    const int quad = ew & 3;
    const int half = ew >> 2;
    const tair_epilogue& e = p.epi;
    uint8_t* stg = stg_base + ew * STG_BYTES_PER_WARP;   // buffer b of this warp: + b * STG_BYTES
    uint32_t stg_sel = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = pair; tile < num_tiles; tile += num_pairs) {
      const int tm2 = tile / p.tiles_n, tn = tile - tm2 * p.tiles_n;
      const int m0q = (tm2 * 2 + (int)rank) * BM + quad * 32;
      if (p.dbg & 2) {   // otherwise the epilogue waits itself, after its first residual prefetch
        mbar_wait(tfull_bar(acc), acc_phase);
        tc_fence_after();
      }
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + acc * BN;
      const uint32_t tempty_leader = leader ? tempty_bar(acc) : mapa_shared(tempty_bar(acc), 0);
      if (p.dbg & 2) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) { if (leader) mbar_arrive(tempty_leader); else mbar_arrive_cluster(tempty_leader); }
      } else
        epilogue_dispatch_tma<BN>(p, &tmC64, &tmC32, m0q, tn, half, lane, taddr, stg, tempty_leader, !leader, tfull_bar(acc), acc_phase, stg_sel);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (elect_one()) tma_store_wait_all<0>();
    __syncwarp();
  }

  tc_fence_before();
  cluster_sync_all();  // the peer's smem / barriers must stay alive until every remote arrive and TMA signal landed
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_2cta(tmem_base, C::TMEM_COLS);
  }
}

// One or two epilogue staging buffers per warp.  With one, a warp cannot write sub-tile i+1 before the bulk store of
// sub-tile i has read the buffer (ncu source page of 151552x1024x256: the largest single stall of the epilogue warps).
// Measured, though, the second buffer (which costs 32 KB = one stage of the operand ring) changes nothing: K = 256 GEMMs
// 39.4 / 36.6 / 28.1 / 91.0 us with two buffers vs 39.3 / 35.9 / 26.7 / 89.5 with one, B=16 step 22.75 ms both ways
// (profiles/round2_summary.md) - these GEMMs are bound by HBM reads competing with their own output writes, not by
// the drain.  Default is therefore one buffer; TAIR_EPI_STG=2 selects two for K <= 512 GEMMs (probe).
int pick_staging(const GemmParams& p) {
  static int forced = -1;
  if (forced < 0) {
    const char* v = getenv("TAIR_EPI_STG");
    forced = v ? atoi(v) : 1;
  }
  if (forced == 2) return (p.tma_store && !p.conv && p.num_kb <= 8) ? 2 : 1;
  return 1;
}

template <int BN>
int launch_bn2(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC64, const CUtensorMap& tmC32,
               const GemmParams& p, cudaStream_t st) {
  TAIR_SMEM_OPTIN(gemm_tc2_kernel<BN>, Cfg2<BN>::SMEM_MAX);
  GemmParams q = p;
  q.stg_bufs = pick_staging(p);
  q.stages = Cfg2<BN>::stages_for(q.stg_bufs);
  const int tiles2 = ((p.tiles_m + 1) / 2) * p.tiles_n;
  int pairs = num_sms() / 2;
  if (tiles2 < pairs) pairs = tiles2;
  TAIR_LAUNCH((gemm_tc2_kernel<BN>), 2 * pairs, GEMM_THREADS, Cfg2<BN>::smem_for(q.stg_bufs), st, tmA, tmB, tmC64, tmC32, q);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return check_launch("gemm_tc2_kernel");
}

template <int BN>
int launch_bn(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC64, const CUtensorMap& tmC32,
              const GemmParams& p, cudaStream_t st) {
  TAIR_SMEM_OPTIN(gemm_tc_kernel<BN>, Cfg<BN>::SMEM_MAX);
  GemmParams q = p;
  q.stg_bufs = pick_staging(p);
  q.stages = Cfg<BN>::stages_for(q.stg_bufs);
  const int tiles = p.tiles_m * p.tiles_n * p.splits;
  const int grid = tiles < num_sms() ? tiles : num_sms();
  TAIR_LAUNCH((gemm_tc_kernel<BN>), grid, GEMM_THREADS, Cfg<BN>::smem_for(q.stg_bufs), st, tmA, tmB, tmC64, tmC32, q);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return check_launch("gemm_tc_kernel");
}

// Fallback tile choice (used while a stream is being captured, or when autotuning is off / not applicable).
// Per K=16 step a 128xBN tile costs max(MMA pipe, operand ingest): the tensor pipe needs ~N/2 + 43 cycles for an SS-mode
// MMA (tools/probes/mma_shape_probe.cu) and each SM ingests TMA operand rows (128 B each) at ~64 B/clk:
// (4 KB of A + BN*32 B of B) per step.
int tile_cost(int bn) {
  const int mma = bn / 2 + 43, ingest = 64 + bn / 2;
  return mma > ingest ? mma : ingest;
}

// Pick the N tile that minimises  waves x (mainloop cycles + fixed per-tile overhead).
int pick_bn(int M, int N, int num_kb, int act) {
  if (act == TAIR_ACT_GEGLU) return (N % 256 == 0) ? 256 : ((N % 128 == 0) ? 128 : 0);
  const int cands[4] = {256, 160, 128, 64};
  const int tiles_m = (M + BM - 1) / BM;
  const int sms = num_sms();
  long best = -1;
  int best_bn = 128;
  for (int i = 0; i < 4; ++i) {
    const int bn = cands[i];
    const long tiles = (long)tiles_m * ((N + bn - 1) / bn);
    const long waves = (tiles + sms - 1) / sms;
    const long cost = waves * ((long)num_kb * (BK / 16) * tile_cost(bn) + 700);
    if (best < 0 || cost < best) {
      best = cost;
      best_bn = bn;
    }
  }
  return best_bn;
}

// 2-CTA tiles need the TMA-store epilogue
bool legal_2cta(const GemmParams& p, int bn) {
  return (bn == 256 || bn == 160 || bn == 128) && !p.epi.out_fp32 && p.vec_out;
}

// heuristic: pays off only for wide, MMA-bound tiles with at least one full 256-row tile per SM pair
bool use_2cta(const GemmParams& p, int bn) {
  static int mode = -1;  // TAIR_GEMM_2CTA: 0 never, 1 heuristic (default), 2 always when legal
  if (mode < 0) {
    const char* e = getenv("TAIR_GEMM_2CTA");
    mode = e ? atoi(e) : 1;
  }
  if (mode == 0 || !legal_2cta(p, bn)) return false;
  if (mode == 2) return true;
  const long tiles2 = (long)((p.tiles_m + 1) / 2) * ((p.N + bn - 1) / bn);
  return bn == 256 && p.num_kb >= 16 && tiles2 >= 2 * (num_sms() / 2);
}

// Which TMA-store epilogue drains the tiles (GemmParams.epi_mode).  TAIR_EPI_LEAN=0 forces the generic one (A/B probe).
int pick_epi_mode(const GemmParams& p) {
  static int lean = -1;
  if (lean < 0) {
    const char* v = getenv("TAIR_EPI_LEAN");
    lean = v ? atoi(v) : 1;
  }
  const tair_epilogue& e = p.epi;
  const bool rg16 = e.rowgroup != nullptr && e.rowgroup_bf16;
  if (!p.tma_store || e.act == TAIR_ACT_GEGLU || e.ln_row_stats != nullptr || p.N % 32 != 0 || p.splits != 1 ||
      (e.bias != nullptr && !p.vec_bias) || (e.rowgroup != nullptr && !rg16) || (!lean && !rg16))
    return 2;
  if (e.residual == nullptr && !rg16) return 0;
  if (e.act != TAIR_ACT_NONE || (e.residual != nullptr && rg16)) return 2;
  if (rg16) return ((reinterpret_cast<uintptr_t>(e.rowgroup) % 16) == 0 && e.ldg % 8 == 0) ? 1 : 2;
  return p.vec_res ? 1 : 2;
}

int dispatch(const CUtensorMap& tmA, const void* W, int64_t ldw, GemmParams& p, int bn, bool two,
             cudaStream_t st) {
  CUtensorMap tmB;
  p.tiles_m = (p.M + BM - 1) / BM;
  const uint64_t dimsB[2] = {(uint64_t)p.K, (uint64_t)p.N};
  const uint64_t strB[1] = {(uint64_t)ldw * 2};
  const uint32_t boxB[2] = {BK, (uint32_t)(two ? bn / 2 : bn)};
  int rc = make_tmap_bf16(&tmB, W, 2, dimsB, strB, boxB, nullptr, true);
  if (rc) return rc;
  p.tiles_m = (p.M + BM - 1) / BM;
  p.tiles_n = (p.N + bn - 1) / bn;
  // output maps for the TMA-store epilogue: 32-row x 64-column (128B swizzle) and 32 x 32 (64B swizzle) boxes
  CUtensorMap tmC64 = tmB, tmC32 = tmB;
  p.tma_store = (!p.epi.out_fp32 && p.vec_out) ? 1 : 0;
  if (p.tma_store) {
    const int n_out = (p.epi.act == TAIR_ACT_GEGLU) ? p.N / 2 : p.N;
    const uint64_t dimsC[2] = {(uint64_t)n_out, (uint64_t)p.M};
    const uint64_t strC[1] = {(uint64_t)p.epi.ldc * 2};
    const uint32_t box64[2] = {64, 32}, box32[2] = {32, 32};
    if ((rc = make_tmap_bf16(&tmC64, p.epi.out, 2, dimsC, strC, box64, nullptr, 3))) return rc;
    if ((rc = make_tmap_bf16(&tmC32, p.epi.out, 2, dimsC, strC, box32, nullptr, 2))) return rc;
  }
  p.epi_mode = pick_epi_mode(p);
  TAIR_REQUIRE(!p.epi.rowgroup_bf16 || p.epi_mode == 1,
               "bf16 row groups need the row-add epilogue: GEMM / conv with a 16-byte aligned bf16 output, N %% 32 == 0, "
               "no activation, no residual, no folded LayerNorm, rows 16-byte aligned (ldg %% 8 == 0)");
  if (two) {
    switch (bn) {
      case 256: return launch_bn2<256>(tmA, tmB, tmC64, tmC32, p, st);
      case 160: return launch_bn2<160>(tmA, tmB, tmC64, tmC32, p, st);
      case 128: return launch_bn2<128>(tmA, tmB, tmC64, tmC32, p, st);
    }
  }
  switch (bn) {
    case 256: return launch_bn<256>(tmA, tmB, tmC64, tmC32, p, st);
    case 160: return launch_bn<160>(tmA, tmB, tmC64, tmC32, p, st);
    case 128: return launch_bn<128>(tmA, tmB, tmC64, tmC32, p, st);
    case 64: return launch_bn<64>(tmA, tmB, tmC64, tmC32, p, st);
    case 96: return launch_bn<96>(tmA, tmB, tmC64, tmC32, p, st);
    case 192: return launch_bn<192>(tmA, tmB, tmC64, tmC32, p, st);
    case 224: return launch_bn<224>(tmA, tmB, tmC64, tmC32, p, st);
  }
  set_error("gemm: unsupported BN %d", bn);
  return TAIR_ERR_UNSUPPORTED;
}

int check_epilogue(const tair_epilogue* e, GemmParams& p, int n_out) {
  TAIR_REQUIRE(e != nullptr && e->out != nullptr, "epilogue/out pointer is NULL");
  TAIR_REQUIRE(e->ldc >= n_out, "ldc (%lld) < output columns (%d)", (long long)e->ldc, n_out);
  TAIR_REQUIRE(e->act >= 0 && e->act <= TAIR_ACT_RELU, "unknown activation %d", e->act);
  if (e->rowgroup) TAIR_REQUIRE(e->rows_per_group != 0, "rows_per_group must be non-zero");
  if (e->act == TAIR_ACT_GEGLU)
    TAIR_REQUIRE(e->rowgroup == nullptr, "GEGLU epilogue does not take a row-group add");
  TAIR_REQUIRE((e->ln_row_stats == nullptr) == (e->ln_col_sum == nullptr), "ln_row_stats and ln_col_sum go together");
  if (e->ln_row_stats)
    TAIR_REQUIRE(p.conv == 0 && (reinterpret_cast<uintptr_t>(e->ln_row_stats) % 8) == 0 &&
                     (reinterpret_cast<uintptr_t>(e->ln_col_sum) % 16) == 0 && p.N % 4 == 0,
                 "folded LayerNorm: GEMM only, row stats 8-byte / column sums 16-byte aligned, N %% 4 == 0");
  p.epi = *e;
  {
    const char* d = getenv("TAIR_GEMM_DEBUG");
    p.dbg = d ? atoi(d) : 0;
  }
  const int esz = e->out_fp32 ? 4 : 2;
  p.vec_out = ((reinterpret_cast<uintptr_t>(e->out) % 16) == 0) && ((e->ldc * esz) % 16 == 0);
  p.vec_bias = e->bias && ((reinterpret_cast<uintptr_t>(e->bias) % 16) == 0);
  p.vec_rg = e->rowgroup && !e->rowgroup_bf16 && ((reinterpret_cast<uintptr_t>(e->rowgroup) % 16) == 0) && (e->ldg % 4 == 0);
  p.vec_res = e->residual && ((reinterpret_cast<uintptr_t>(e->residual) % 16) == 0) &&
              ((e->ldr * 2) % 16 == 0);
  return TAIR_OK;
}


// ---------------------------------------------------------------------------------------------------------------------
// Split-K for small-M / deep-K problems (the 8x8 levels: M = 64 * batch pixels, K = 9 * 1280 ... 9 * 2560).  With
// 128-row tiles such a problem has only 64-80 tiles, every active SM is pinned at its ~55 B/clk operand ingest (ncu:
// 622 cycles per k-block on 80 SMs, tensor pipe 44 %) and half the chip idles.  `splits` CTAs share a tile's K range,
// write fp32 partial tiles to a workspace, and a second small kernel sums them in a FIXED order (deterministic) and
// applies the epilogue.
__global__ void __launch_bounds__(256)
splitk_reduce_kernel(const float* __restrict__ ws, int splits, int M, int N, const tair_epilogue e) {
  pdl_grid_sync();
  const int64_t idx4 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // one thread = 4 consecutive columns
  const int n4 = N >> 2;
  if (idx4 >= (int64_t)M * n4) return;
  const int m = (int)(idx4 / n4), n = (int)(idx4 - (int64_t)m * n4) * 4;
  float4 acc = *reinterpret_cast<const float4*>(ws + (int64_t)m * N + n);
  for (int s = 1; s < splits; ++s) {
    const float4 t = *reinterpret_cast<const float4*>(ws + ((int64_t)s * M + m) * N + n);
    acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w;
  }
  float v[4] = {acc.x, acc.y, acc.z, acc.w};
  const float* rg = e.rowgroup == nullptr ? nullptr
                    : reinterpret_cast<const float*>(e.rowgroup) + (int64_t)(e.rows_per_group > 0 ? m / e.rows_per_group : m % (-e.rows_per_group)) * e.ldg;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (e.bias != nullptr) v[j] += __ldg(e.bias + n + j);
    if (rg != nullptr) v[j] += __ldg(rg + n + j);
    switch (e.act) {
      case TAIR_ACT_GELU: v[j] = gelu_f(v[j]); break;
      case TAIR_ACT_SILU: v[j] = silu_f(v[j]); break;
      case TAIR_ACT_RELU: v[j] = fmaxf(v[j], 0.f); break;
      default: break;
    }
    if (e.residual != nullptr)
      v[j] += __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(e.residual)[(int64_t)m * e.ldr + n + j]);
  }
  if (e.out_fp32) {
    float* o = reinterpret_cast<float*>(e.out) + (int64_t)m * e.ldc + n;
    for (int j = 0; j < 4; ++j) o[j] = v[j];
  } else {
    __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(e.out) + (int64_t)m * e.ldc + n;
    for (int j = 0; j < 4; ++j) o[j] = __float2bfloat16(v[j]);
  }
}

bool legal_splitk(const GemmParams& p, int act, int bn, int splits) {
  if (act == TAIR_ACT_GEGLU || p.N % 4 != 0 || splits < 2) return false;
  const long tiles = (long)((p.M + BM - 1) / BM) * ((p.N + bn - 1) / bn);
  return tiles * splits <= num_sms() && p.num_kb / splits >= 8;
}

int dispatch(const CUtensorMap& tmA, const void* W, int64_t ldw, GemmParams& p, int bn, bool two, cudaStream_t st);

// `ws` holds splits * M * N floats
int dispatch_splitk(const CUtensorMap& tmA, const void* W, int64_t ldw, GemmParams& p, int bn, int splits,
                    cudaStream_t st, void* ws) {
  TAIR_REQUIRE(!p.epi.rowgroup_bf16, "bf16 row groups are not supported by the split-K path");
  GemmParams q = p;
  q.splits = splits;
  q.kb_split = (p.num_kb + splits - 1) / splits;
  q.epi = tair_epilogue{};
  q.epi.out = ws; q.epi.ldc = p.N; q.epi.out_fp32 = 1;
  q.vec_out = 1; q.vec_res = 0; q.vec_rg = 0;
  int rc = dispatch(tmA, W, ldw, q, bn, false, st);
  if (rc) return rc;
  const int64_t n4 = (int64_t)p.M * (p.N / 4);
  TAIR_LAUNCH((splitk_reduce_kernel), (unsigned)((n4 + 255) / 256), 256, 0, st, reinterpret_cast<const float*>(ws), splits, p.M, p.N, p.epi);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return check_launch("splitk_reduce_kernel");
}

// ---------------------------------------------------------------------------------------------------------------------
// Tile autotuner.  Which (BN, 1-CTA / 2-CTA pair) is fastest depends on wave quantisation, on the K depth and on how
// many SMs share the L2 -> SM operand path; no closed-form rule got within 25 % on every shape of the UNet
// (tools/bn_sweep.py), so the first call for a problem shape times every legal candidate on the caller's stream
// (1 warm-up + 5 timed launches each) and caches the winner per device.  All candidates compute bit-identical
// results (same K order per output element), so tuning never changes the numbers.  Tuning is skipped — and the
// closed-form pick used, uncached — while the stream is being captured, when the output aliases an input, or when
// TAIR_AUTOTUNE=0.  It synchronises the stream once per new shape.
struct TuneKey {
  int dev, conv, M, N, K, Wo, stride, act, flags;
  bool operator<(const TuneKey& o) const {
    return std::memcmp(this, &o, sizeof(TuneKey)) < 0;
  }
};
struct TuneChoice { int bn; bool two; int splits; };

std::mutex g_tune_mu;
std::map<TuneKey, TuneChoice> g_tuned;

bool autotune_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("TAIR_AUTOTUNE");
    on = (e && atoi(e) == 0) ? 0 : 1;
  }
  return on == 1;
}

bool overlaps(const void* a, size_t na, const void* b, size_t nb) {
  const uintptr_t x = reinterpret_cast<uintptr_t>(a), y = reinterpret_cast<uintptr_t>(b);
  return a && b && x < y + nb && y < x + na;
}

// Decide the tile for this problem and launch it.  `in_bytes` is the extent of the A operand (aliasing check).
int tuned_dispatch(const CUtensorMap& tmA, const void* A, size_t in_bytes, const void* W, int64_t ldw, GemmParams& p,
                   int act, cudaStream_t st) {
  p.tiles_m = (p.M + BM - 1) / BM;
  if (const char* f = getenv("TAIR_GEMM_BN")) {  // bring-up probe only
    const int bn = atoi(f);
    // a GEGLU weight is interleaved for one tile width (interleave_geglu): any other BN would pair value rows with value rows
    const int geglu_bn = act == TAIR_ACT_GEGLU ? pick_bn(p.M, p.N, p.num_kb, act) : bn;
    TAIR_REQUIRE(bn == geglu_bn, "gemm: TAIR_GEMM_BN=%d does not match the GEGLU weight interleave (BN=%d for N=%d)", bn,
                 geglu_bn, p.N);
    if (const char* sp = getenv("TAIR_GEMM_SPLITS")) {   // probe: needs a caller workspace
      const int splits = atoi(sp);
      if (legal_splitk(p, act, bn, splits) && p.epi.workspace != nullptr &&
          (size_t)p.epi.workspace_bytes >= (size_t)splits * p.M * p.N * sizeof(float))
        return dispatch_splitk(tmA, W, ldw, p, bn, splits, st, p.epi.workspace);
    }
    return dispatch(tmA, W, ldw, p, bn, use_2cta(p, bn), st);
  }
  const int heur = pick_bn(p.M, p.N, p.num_kb, act);
  TAIR_REQUIRE(heur != 0, "gemm: GEGLU epilogue needs N %% 128 == 0 (N=%d)", p.N);
  const size_t esz = p.epi.out_fp32 ? 4 : 2;
  const int n_out = act == TAIR_ACT_GEGLU ? p.N / 2 : p.N;
  const size_t out_bytes = ((size_t)(p.M - 1) * p.epi.ldc + n_out) * esz;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) { cudaGetLastError(); cap = cudaStreamCaptureStatusActive; }
  const bool tunable = autotune_enabled() && act != TAIR_ACT_GEGLU && p.dbg == 0 && cap == cudaStreamCaptureStatusNone &&
                       !overlaps(p.epi.out, out_bytes, A, in_bytes) &&
                       !overlaps(p.epi.out, out_bytes, p.epi.residual, p.epi.residual ? ((size_t)(p.M - 1) * p.epi.ldr + n_out) * 2 : 0);
  TuneKey key;
  std::memset(&key, 0, sizeof(key));
  cudaGetDevice(&key.dev);
  key.conv = p.conv; key.M = p.M; key.N = p.N; key.K = p.K; key.Wo = p.Wo; key.stride = p.stride; key.act = act;
  key.flags = (p.epi.out_fp32 ? 1 : 0) | (p.vec_out ? 2 : 0) | (p.epi.residual ? 4 : 0) | (p.epi.rowgroup ? 8 : 0) |
              (p.epi.ln_row_stats ? 16 : 0) | (p.epi.rowgroup_bf16 ? 32 : 0);
  {
    std::lock_guard<std::mutex> lk(g_tune_mu);
    auto it = g_tuned.find(key);
    if (it != g_tuned.end()) return dispatch(tmA, W, ldw, p, it->second.bn, it->second.two, st);
  }
  if (!tunable) return dispatch(tmA, W, ldw, p, heur, use_2cta(p, heur), st);

  const int cands[7] = {256, 224, 192, 160, 128, 96, 64};
  cudaEvent_t e0, e1;
  TAIR_CUDA(cudaEventCreate(&e0));
  TAIR_CUDA(cudaEventCreate(&e1));
  const int64_t launches_before = g_launch_count.load();
  TuneChoice best{heur, use_2cta(p, heur), 1};
  float best_ms = -1.f;
  int rc = TAIR_OK;
  for (int i = 0; i < 7 && rc == TAIR_OK; ++i) {
    for (int two = 0; two < 2 && rc == TAIR_OK; ++two) {
      const int bn = cands[i];
      if (two && !legal_2cta(p, bn)) continue;
      if ((long)p.tiles_m * ((p.N + bn - 1) / bn) > 8L * num_sms() && bn < 128) continue;  // hopeless: skip
      if ((rc = dispatch(tmA, W, ldw, p, bn, two != 0, st))) break;  // warm-up (also sets the smem attribute)
      cudaEventRecord(e0, st);
      for (int r = 0; r < 5 && rc == TAIR_OK; ++r) rc = dispatch(tmA, W, ldw, p, bn, two != 0, st);
      cudaEventRecord(e1, st);
      if (cudaEventSynchronize(e1) != cudaSuccess) { rc = check_launch("gemm autotune"); if (rc == TAIR_OK) rc = TAIR_ERR_CUDA; break; }
      float ms = 0.f;
      cudaEventElapsedTime(&ms, e0, e1);
      if (best_ms < 0.f || ms < best_ms) { best_ms = ms; best = TuneChoice{bn, two != 0, 1}; }
    }
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  g_launch_count.store(launches_before);  // tuning launches are not part of the caller's work
  if (rc) return rc;
  {
    std::lock_guard<std::mutex> lk(g_tune_mu);
    g_tuned[key] = best;
  }
  if (getenv("TAIR_AUTOTUNE_VERBOSE"))
    fprintf(stderr, "[tair autotune] %s M=%d N=%d K=%d act=%d -> BN=%d%s (%.1f us; closed-form pick BN=%d)\n",
            p.conv ? "conv" : "gemm", p.M, p.N, p.K, act, best.bn, best.two ? " 2-CTA" : "", best_ms / 5 * 1e3, heur);
  return dispatch(tmA, W, ldw, p, best.bn, best.two, st);
}

}  // namespace
}  // namespace tair

using namespace tair;

extern "C" int tair_gemm_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, int32_t M,
                              int32_t N, int32_t K, const tair_epilogue* epi, void* stream) {
  TAIR_REQUIRE(A && W, "gemm: NULL operand");
  TAIR_REQUIRE(M > 0 && N > 0 && K > 0, "gemm: bad shape M=%d N=%d K=%d", M, N, K);
  TAIR_REQUIRE(lda % 8 == 0 && ldw % 8 == 0 && lda >= K && ldw >= K,
               "gemm: lda/ldw must be >= K and multiples of 8 (lda=%lld ldw=%lld K=%d)",
               (long long)lda, (long long)ldw, K);
  TAIR_REQUIRE((reinterpret_cast<uintptr_t>(A) % 16) == 0 && (reinterpret_cast<uintptr_t>(W) % 16) == 0,
               "gemm: operands must be 16-byte aligned");
  GemmParams p{};
  p.M = M; p.N = N; p.K = K;
  p.num_kb = (K + BK - 1) / BK;
  p.splits = 1; p.kb_split = p.num_kb;
  p.conv = 0;
  const int act = epi ? epi->act : 0;
  const int n_out = (act == TAIR_ACT_GEGLU) ? N / 2 : N;
  int rc = check_epilogue(epi, p, n_out);
  if (rc) return rc;
  CUtensorMap tmA;
  const uint64_t dimsA[2] = {(uint64_t)K, (uint64_t)M};
  const uint64_t strA[1] = {(uint64_t)lda * 2};
  const uint32_t boxA[2] = {BK, BM};
  rc = make_tmap_bf16(&tmA, A, 2, dimsA, strA, boxA, nullptr, true);
  if (rc) return rc;
  return tuned_dispatch(tmA, A, ((size_t)(M - 1) * lda + K) * 2, W, ldw, p, act, static_cast<cudaStream_t>(stream));
}

extern "C" int tair_conv3x3_bf16(const void* x, const void* w, int32_t B, int32_t H, int32_t W,
                                 int32_t Cin, int32_t Cout, int32_t stride, int32_t pad, const tair_epilogue* epi,
                                 void* stream) {
  TAIR_REQUIRE(x && w, "conv3x3: NULL operand");
  TAIR_REQUIRE(B > 0 && H > 0 && W > 0 && Cin > 0 && Cout > 0, "conv3x3: bad shape");
  TAIR_REQUIRE(stride == 1 || stride == 2, "conv3x3: stride must be 1 or 2 (got %d)", stride);
  TAIR_REQUIRE(Cin % 64 == 0, "conv3x3: Cin must be a multiple of 64 (got %d)", Cin);
  TAIR_REQUIRE((reinterpret_cast<uintptr_t>(x) % 16) == 0 && (reinterpret_cast<uintptr_t>(w) % 16) == 0,
               "conv3x3: operands must be 16-byte aligned");
  TAIR_REQUIRE(pad == 0 || pad == 1, "conv3x3: pad (top/left) must be 0 or 1 (got %d)", pad);
  // k=3; `pad` zeros on the top/left, one zero row/column on the bottom/right: pad=1 is PyTorch padding=1, pad=0 is the
  // asymmetric F.pad(x,(0,1,0,1)) + padding=0 of the VAE downsampler (terediff/model/vae.py:51-55)
  const int Ho = (H + pad + 1 - 3) / stride + 1, Wo = (W + pad + 1 - 3) / stride + 1;
  // An M tile is 128 consecutive output pixels = bn images x bh rows x bw columns.
  const int bw = Wo < BM ? Wo : BM;
  TAIR_REQUIRE(BM % bw == 0 && Wo % bw == 0, "conv3x3: output width %d does not tile 128", Wo);
  int bh = BM / bw;
  if (bh > Ho) bh = Ho;
  TAIR_REQUIRE(Ho % bh == 0 && BM % (bw * bh) == 0, "conv3x3: output height %d does not tile 128", Ho);
  const int bimg = BM / (bw * bh);
  TAIR_REQUIRE(bimg == 1 || bh == Ho, "conv3x3: internal tiling error");
  TAIR_REQUIRE(bw * stride <= 256 && bh * stride <= 256, "conv3x3: TMA box too large");

  GemmParams p{};
  p.M = B * Ho * Wo; p.N = Cout; p.K = 9 * Cin;
  p.num_kb = 9 * (Cin / BK);
  p.splits = 1; p.kb_split = p.num_kb;
  p.conv = 1; p.kb_per_tap = Cin / BK;
  p.Ho = Ho; p.Wo = Wo; p.stride = stride; p.pad = pad;
  const int act = epi ? epi->act : 0;
  TAIR_REQUIRE(act != TAIR_ACT_GEGLU, "conv3x3: GEGLU epilogue not supported");
  int rc = check_epilogue(epi, p, Cout);
  if (rc) return rc;
  CUtensorMap tmA;
  const uint64_t dimsA[4] = {(uint64_t)Cin, (uint64_t)W, (uint64_t)H, (uint64_t)B};
  const uint64_t strA[3] = {(uint64_t)Cin * 2, (uint64_t)W * Cin * 2, (uint64_t)H * W * Cin * 2};
  const uint32_t boxA[4] = {BK, (uint32_t)(bw * stride), (uint32_t)(bh * stride), (uint32_t)bimg};
  const uint32_t es[4] = {1, (uint32_t)stride, (uint32_t)stride, 1};
  rc = make_tmap_bf16(&tmA, x, 4, dimsA, strA, boxA, es, true);
  if (rc) return rc;
  // Deep-K layers on the 8x8 level (<= 64 output pixels per image): 3-way split-K when the caller lends a workspace.
  // The rule looks at the layer geometry only, so a tile's numbers do not depend on the batch it is processed in.
  constexpr int SPLITS = 3;
  if (Ho * Wo <= 64 && p.num_kb >= 64 && Cout % 4 == 0 && p.dbg == 0 && !getenv("TAIR_GEMM_BN") && p.epi.workspace != nullptr &&
      (reinterpret_cast<uintptr_t>(p.epi.workspace) % 16) == 0 &&
      (size_t)p.epi.workspace_bytes >= (size_t)SPLITS * p.M * p.N * sizeof(float)) {
    const int bn = Cout % 256 == 0 ? 256 : (Cout % 160 == 0 ? 160 : 128);
    return dispatch_splitk(tmA, w, (int64_t)9 * Cin, p, bn, SPLITS, static_cast<cudaStream_t>(stream), p.epi.workspace);
  }
  return tuned_dispatch(tmA, x, (size_t)B * H * W * Cin * 2, w, (int64_t)9 * Cin, p, act, static_cast<cudaStream_t>(stream));
}
