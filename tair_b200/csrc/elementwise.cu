// Memory-bound elementwise / layout kernels of the denoising step.
//
//   tair_sampler_update   : v -> x0 -> posterior mean/variance -> x_{t-1}, optional CFG combine
//                           (terediff/sampler/spaced_sampler.py:141-147,123-131,149-164,167-189)
//   tair_sampler_multistep_update: v -> x0 -> DDIM / DPM-Solver++(2M) step with an in-place x0 history
//   tair_timestep_embedding: cos||sin sinusoidal embedding (terediff/model/util.py:128-148)
//   tair_nchw_to_nhwc_bf16 / tair_nhwc_to_nchw_f32 : reference (B,C,H,W) fp32 <-> internal [B*H*W, C] bf16
//   tair_concat_add       : out = [a | b (+ c)] along channels  (decoder skip: controlnet.py:46-50)
//   tair_add_bf16         : out = a + b                          (mid-block control add: controlnet.py:41-42)
//   tair_upsample2x_nhwc  : nearest x2 (unet.py:73-75)
#include <atomic>

#include "../../include/tair_b200.h"
#include "common.cuh"

namespace tair {
extern std::atomic<int64_t> g_launch_count;
namespace {

__global__ void sampler_update_kernel(const float* __restrict__ x, const float* __restrict__ v_cond,
                                      const float* __restrict__ v_uncond, const float* __restrict__ noise,
                                      float* __restrict__ x_prev, float* __restrict__ x0_out,
                                      const int64_t* __restrict__ t, const float* __restrict__ sqrt_ac,
                                      const float* __restrict__ sqrt_1mac, const float* __restrict__ coef1,
                                      const float* __restrict__ coef2, const float* __restrict__ post_var,
                                      float cfg_scale, const float* __restrict__ cfg_scale_dev, int per_sample,
                                      int total) {
  pdl_grid_sync();
  // 4 elements per thread; per_sample % 4 == 0 so a float4 never straddles two samples
  const int i4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i4 >= total) return;
  const int b = i4 / per_sample;
  const int64_t ti = t[b];
  const float sa = sqrt_ac[ti], sm = sqrt_1mac[ti], c1 = coef1[ti], c2 = coef2[ti];
  const float sigma = (ti != 0) ? sqrtf(post_var[ti]) : 0.f;
  const float4 xv = *reinterpret_cast<const float4*>(x + i4);
  float4 vv = *reinterpret_cast<const float4*>(v_cond + i4);
  if (v_uncond != nullptr) {
    if (cfg_scale_dev != nullptr) cfg_scale = *cfg_scale_dev;  // device scalar: one captured graph, any scale
    const float4 vu = *reinterpret_cast<const float4*>(v_uncond + i4);
    vv.x = __fadd_rn(vu.x, __fmul_rn(cfg_scale, __fsub_rn(vv.x, vu.x)));
    vv.y = __fadd_rn(vu.y, __fmul_rn(cfg_scale, __fsub_rn(vv.y, vu.y)));
    vv.z = __fadd_rn(vu.z, __fmul_rn(cfg_scale, __fsub_rn(vv.z, vu.z)));
    vv.w = __fadd_rn(vu.w, __fmul_rn(cfg_scale, __fsub_rn(vv.w, vu.w)));
  }
  const float4 nz = *reinterpret_cast<const float4*>(noise + i4);
  float4 x0, out;
  // same operation order as the reference, no fused multiply-add, so fp32 results are bit-identical
  x0.x = __fsub_rn(__fmul_rn(sa, xv.x), __fmul_rn(sm, vv.x));
  x0.y = __fsub_rn(__fmul_rn(sa, xv.y), __fmul_rn(sm, vv.y));
  x0.z = __fsub_rn(__fmul_rn(sa, xv.z), __fmul_rn(sm, vv.z));
  x0.w = __fsub_rn(__fmul_rn(sa, xv.w), __fmul_rn(sm, vv.w));
  out.x = __fadd_rn(__fadd_rn(__fmul_rn(c1, x0.x), __fmul_rn(c2, xv.x)), __fmul_rn(sigma, nz.x));
  out.y = __fadd_rn(__fadd_rn(__fmul_rn(c1, x0.y), __fmul_rn(c2, xv.y)), __fmul_rn(sigma, nz.y));
  out.z = __fadd_rn(__fadd_rn(__fmul_rn(c1, x0.z), __fmul_rn(c2, xv.z)), __fmul_rn(sigma, nz.z));
  out.w = __fadd_rn(__fadd_rn(__fmul_rn(c1, x0.w), __fmul_rn(c2, xv.w)), __fmul_rn(sigma, nz.w));
  *reinterpret_cast<float4*>(x_prev + i4) = out;
  if (x0_out != nullptr) *reinterpret_cast<float4*>(x0_out + i4) = x0;
}

// DDIM / DPM-Solver++(2M) step: x_next = ((b*x0 + a*x) + c*x0_hist) + d*noise, x0_hist <- x0.  The CFG combine and the
// x0 line are those of sampler_update_kernel, in the same order.  Each thread reads and then overwrites its own float4 of
// x0_hist, so the in-place history update has no race.
__global__ void sampler_multistep_kernel(const float* __restrict__ x, const float* __restrict__ v_cond,
                                         const float* __restrict__ v_uncond, const float* __restrict__ noise,
                                         float* __restrict__ x_next, float* __restrict__ x0_hist,
                                         const int64_t* __restrict__ t, const float* __restrict__ P,
                                         const float* __restrict__ Q, const float* __restrict__ A,
                                         const float* __restrict__ Bc, const float* __restrict__ Cc,
                                         const float* __restrict__ D, float cfg_scale,
                                         const float* __restrict__ cfg_scale_dev, int per_sample, int total) {
  pdl_grid_sync();
  const int i4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i4 >= total) return;
  const int b = i4 / per_sample;
  const int64_t ti = t[b];
  const float p = P[ti], q = Q[ti], ca = A[ti], cb = Bc[ti], cc = Cc[ti], cd = D[ti];
  const float4 xv = *reinterpret_cast<const float4*>(x + i4);
  float4 vv = *reinterpret_cast<const float4*>(v_cond + i4);
  if (v_uncond != nullptr) {
    if (cfg_scale_dev != nullptr) cfg_scale = *cfg_scale_dev;
    const float4 vu = *reinterpret_cast<const float4*>(v_uncond + i4);
    vv.x = __fadd_rn(vu.x, __fmul_rn(cfg_scale, __fsub_rn(vv.x, vu.x)));
    vv.y = __fadd_rn(vu.y, __fmul_rn(cfg_scale, __fsub_rn(vv.y, vu.y)));
    vv.z = __fadd_rn(vu.z, __fmul_rn(cfg_scale, __fsub_rn(vv.z, vu.z)));
    vv.w = __fadd_rn(vu.w, __fmul_rn(cfg_scale, __fsub_rn(vv.w, vu.w)));
  }
  const float4 nz = *reinterpret_cast<const float4*>(noise + i4);
  // c == 0 is uniform per sample: the history is not read, so a first step never sees stale (or NaN) history
  float4 h = make_float4(0.f, 0.f, 0.f, 0.f);
  if (cc != 0.f && x0_hist != nullptr) h = *reinterpret_cast<const float4*>(x0_hist + i4);
  float4 x0, out;
  x0.x = __fsub_rn(__fmul_rn(p, xv.x), __fmul_rn(q, vv.x));
  x0.y = __fsub_rn(__fmul_rn(p, xv.y), __fmul_rn(q, vv.y));
  x0.z = __fsub_rn(__fmul_rn(p, xv.z), __fmul_rn(q, vv.z));
  x0.w = __fsub_rn(__fmul_rn(p, xv.w), __fmul_rn(q, vv.w));
  out.x = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(cb, x0.x), __fmul_rn(ca, xv.x)), __fmul_rn(cc, h.x)), __fmul_rn(cd, nz.x));
  out.y = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(cb, x0.y), __fmul_rn(ca, xv.y)), __fmul_rn(cc, h.y)), __fmul_rn(cd, nz.y));
  out.z = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(cb, x0.z), __fmul_rn(ca, xv.z)), __fmul_rn(cc, h.z)), __fmul_rn(cd, nz.z));
  out.w = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(cb, x0.w), __fmul_rn(ca, xv.w)), __fmul_rn(cc, h.w)), __fmul_rn(cd, nz.w));
  *reinterpret_cast<float4*>(x_next + i4) = out;
  if (x0_hist != nullptr) *reinterpret_cast<float4*>(x0_hist + i4) = x0;
}

__global__ void timestep_embedding_kernel(const int64_t* __restrict__ t, __nv_bfloat16* __restrict__ out, int B,
                                          int dim, float max_period) {
  pdl_grid_sync();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int half = dim / 2;
  if (i >= B * dim) return;
  const int b = i / dim, j = i - b * dim;
  float val = 0.f;
  if (j < 2 * half) {
    const int k = j < half ? j : j - half;
    const float freq = expf(-logf(max_period) * (float)k / (float)half);
    const float ang = (float)t[b] * freq;
    val = j < half ? cosf(ang) : sinf(ang);
  }
  out[i] = __float2bfloat16(val);
}

// (B, C, HW) fp32 -> [B, HW, Cpad] bf16 (channels >= C zero-filled); 32x32 smem transpose
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, int C, int HW,
                                    int Cpad) {
  pdl_grid_sync();
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x, ty = threadIdx.y;  // 32 x 8
  for (int k = ty; k < 32; k += 8) {
    const int c = c0 + k, px = p0 + tx;
    tile[k][tx] = (c < C && px < HW) ? in[((int64_t)b * C + c) * HW + px] : 0.f;
  }
  __syncthreads();
  for (int k = ty; k < 32; k += 8) {
    const int px = p0 + k, c = c0 + tx;
    if (px < HW && c < Cpad) out[((int64_t)b * HW + px) * Cpad + c] = __float2bfloat16(tile[tx][k]);
  }
}

// [B, HW, ld] bf16 (first C channels) -> (B, C, HW) fp32
__global__ void nhwc_to_nchw_kernel(const __nv_bfloat16* __restrict__ in, float* __restrict__ out, int C, int HW,
                                    int64_t ld) {
  pdl_grid_sync();
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x, ty = threadIdx.y;
  for (int k = ty; k < 32; k += 8) {
    const int px = p0 + k, c = c0 + tx;
    tile[k][tx] = (px < HW && c < C) ? __bfloat162float(in[((int64_t)b * HW + px) * ld + c]) : 0.f;
  }
  __syncthreads();
  for (int k = ty; k < 32; k += 8) {
    const int c = c0 + k, px = p0 + tx;
    if (c < C && px < HW) out[((int64_t)b * C + c) * HW + px] = tile[tx][k];
  }
}

__device__ __forceinline__ uint4 add_bf16x8(uint4 a, uint4 b) {
  uint4 r;
  float2 x, y;
  x = unpack_bf16(a.x); y = unpack_bf16(b.x); r.x = pack_bf16(x.x + y.x, x.y + y.y);
  x = unpack_bf16(a.y); y = unpack_bf16(b.y); r.y = pack_bf16(x.x + y.x, x.y + y.y);
  x = unpack_bf16(a.z); y = unpack_bf16(b.z); r.z = pack_bf16(x.x + y.x, x.y + y.y);
  x = unpack_bf16(a.w); y = unpack_bf16(b.w); r.w = pack_bf16(x.x + y.x, x.y + y.y);
  return r;
}

// out[M, C1+C2] = [a[M,C1] | b[M,C2] (+ c[M,C2])]; one 16-byte vector per thread
__global__ void concat_add_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b,
                                  const uint4* __restrict__ c, uint4* __restrict__ out, int64_t M, int v1, int v2) {
  pdl_grid_sync();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int vt = v1 + v2;
  if (i >= M * vt) return;
  const int64_t row = i / vt;
  const int col = (int)(i - row * vt);
  uint4 r;
  if (col < v1) {
    r = __ldg(a + row * v1 + col);
  } else {
    const int64_t j = row * v2 + (col - v1);
    r = __ldg(b + j);
    if (c != nullptr) r = add_bf16x8(r, __ldg(c + j));
  }
  out[i] = r;
}

__global__ void add_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b, uint4* __restrict__ out,
                           int64_t n) {
  pdl_grid_sync();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = add_bf16x8(__ldg(a + i), __ldg(b + i));
}

// [B, H, W, C] -> [B, 2H, 2W, C] nearest; one 16-byte vector of the OUTPUT per thread
__global__ void upsample2x_kernel(const uint4* __restrict__ in, uint4* __restrict__ out, int B, int H, int W, int vc) {
  pdl_grid_sync();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = (int64_t)B * 4 * H * W * vc;
  if (i >= total) return;
  const int v = (int)(i % vc);
  int64_t r = i / vc;
  const int xo = (int)(r % (2 * W)); r /= 2 * W;
  const int yo = (int)(r % (2 * H));
  const int b = (int)(r / (2 * H));
  out[i] = __ldg(in + (((int64_t)b * H + (yo >> 1)) * W + (xo >> 1)) * vc + v);
}


// row softmax of a bf16 matrix: y[r, :] = softmax(scale * x[r, :]); one warp per row, values cached in registers
// (cols <= 8192).  Used by the single-head, 512-wide VAE attention (terediff/model/vae.py:253-281).
template <int MAXV>
__global__ void softmax_rows_kernel(const __nv_bfloat16* __restrict__ x, int64_t ldx, __nv_bfloat16* __restrict__ y,
                                    int64_t ldy, int rows, int cols, float scale_log2) {
  pdl_grid_sync();
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int nvec = cols >> 3;
  float v[MAXV][8];
  float mx = -3.0e38f;
#pragma unroll
  for (int k = 0; k < MAXV; ++k) {
    const int vi = lane + k * 32;
    if (vi < nvec) {
      const uint4 q = __ldg(reinterpret_cast<const uint4*>(x + (int64_t)row * ldx + vi * 8));
      const float2 a = unpack_bf16(q.x), b = unpack_bf16(q.y), c = unpack_bf16(q.z), d = unpack_bf16(q.w);
      v[k][0] = a.x; v[k][1] = a.y; v[k][2] = b.x; v[k][3] = b.y; v[k][4] = c.x; v[k][5] = c.y; v[k][6] = d.x; v[k][7] = d.y;
#pragma unroll
      for (int i = 0; i < 8; ++i) mx = fmaxf(mx, v[k][i]);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float sum = 0.f;
#pragma unroll
  for (int k = 0; k < MAXV; ++k) {
    const int vi = lane + k * 32;
    if (vi < nvec) {
#pragma unroll
      for (int i = 0; i < 8; ++i) { v[k][i] = ex2_approx((v[k][i] - mx) * scale_log2); sum += v[k][i]; }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float inv = 1.f / sum;
#pragma unroll
  for (int k = 0; k < MAXV; ++k) {
    const int vi = lane + k * 32;
    if (vi < nvec) {
      uint4 q;
      q.x = pack_bf16(v[k][0] * inv, v[k][1] * inv); q.y = pack_bf16(v[k][2] * inv, v[k][3] * inv);
      q.z = pack_bf16(v[k][4] * inv, v[k][5] * inv); q.w = pack_bf16(v[k][6] * inv, v[k][7] * inv);
      *reinterpret_cast<uint4*>(y + (int64_t)row * ldy + vi * 8) = q;
    }
  }
}

// bf16 [R, C] (row stride ldi) -> [C, R] (row stride ldo), batched over blockIdx.z; 32x32 smem tiles
__global__ void transpose_bf16_kernel(const __nv_bfloat16* __restrict__ in, int64_t ldi, int64_t in_batch,
                                      __nv_bfloat16* __restrict__ out, int64_t ldo, int64_t out_batch, int R, int C) {
  pdl_grid_sync();
  __shared__ __nv_bfloat16 tile[32][34];
  in += (int64_t)blockIdx.z * in_batch;
  out += (int64_t)blockIdx.z * out_batch;
  const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
  const int tx = threadIdx.x, ty = threadIdx.y;
  for (int k = ty; k < 32; k += 8) {
    const int r = r0 + k, c = c0 + tx;
    tile[k][tx] = (r < R && c < C) ? in[(int64_t)r * ldi + c] : __float2bfloat16(0.f);
  }
  __syncthreads();
  for (int k = ty; k < 32; k += 8) {
    const int c = c0 + k, r = r0 + tx;
    if (c < C && r < R) out[(int64_t)c * ldo + r] = tile[tx][k];
  }
}

}  // namespace
}  // namespace tair

using namespace tair;

static inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) % 16) == 0; }

extern "C" int tair_sampler_update(const float* x, const float* v_cond, const float* v_uncond, float cfg_scale,
                                   const float* cfg_scale_dev, const float* noise, float* x_prev, float* pred_x0,
                                   const int64_t* t,
                                   const float* sqrt_alphas_cumprod, const float* sqrt_one_minus_alphas_cumprod,
                                   const float* posterior_mean_coef1, const float* posterior_mean_coef2,
                                   const float* posterior_variance, int32_t B, int32_t per_sample, void* stream) {
  TAIR_REQUIRE(x && v_cond && noise && x_prev && t, "sampler_update: NULL pointer");
  TAIR_REQUIRE(sqrt_alphas_cumprod && sqrt_one_minus_alphas_cumprod && posterior_mean_coef1 &&
                   posterior_mean_coef2 && posterior_variance, "sampler_update: NULL schedule table");
  TAIR_REQUIRE(B > 0 && per_sample > 0 && per_sample % 4 == 0, "sampler_update: per_sample must be a multiple of 4");
  TAIR_REQUIRE(al16(x) && al16(v_cond) && al16(noise) && al16(x_prev) && (!v_uncond || al16(v_uncond)) &&
                   (!pred_x0 || al16(pred_x0)), "sampler_update: tensors must be 16-byte aligned");
  const int total = B * per_sample;
  const int threads = 256, grid = (total / 4 + threads - 1) / threads;
  TAIR_LAUNCH((sampler_update_kernel), grid, threads, 0, static_cast<cudaStream_t>(stream), 
      x, v_cond, v_uncond, noise, x_prev, pred_x0, t, sqrt_alphas_cumprod, sqrt_one_minus_alphas_cumprod,
      posterior_mean_coef1, posterior_mean_coef2, posterior_variance, cfg_scale, cfg_scale_dev, per_sample, total);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return check_launch("sampler_update_kernel");
}

extern "C" int tair_sampler_multistep_update(const float* x, const float* v_cond, const float* v_uncond,
                                             float cfg_scale, const float* cfg_scale_dev, const float* noise,
                                             float* x_next, float* x0_hist, const int64_t* t, const float* P,
                                             const float* Q, const float* a, const float* b, const float* c,
                                             const float* d, int32_t B, int32_t per_sample, void* stream) {
  TAIR_REQUIRE(x && v_cond && noise && x_next && t, "sampler_multistep_update: NULL pointer");
  TAIR_REQUIRE(P && Q && a && b && c && d, "sampler_multistep_update: NULL schedule table");
  TAIR_REQUIRE(B > 0 && per_sample > 0 && per_sample % 4 == 0,
               "sampler_multistep_update: per_sample must be a multiple of 4");
  TAIR_REQUIRE(al16(x) && al16(v_cond) && al16(noise) && al16(x_next) && (!v_uncond || al16(v_uncond)) &&
                   (!x0_hist || al16(x0_hist)), "sampler_multistep_update: tensors must be 16-byte aligned");
  TAIR_REQUIRE(x_next != x && x_next != v_cond && x_next != v_uncond && x_next != x0_hist,
               "sampler_multistep_update: x_next must not alias an input");
  const int total = B * per_sample;
  const int threads = 256, grid = (total / 4 + threads - 1) / threads;
  TAIR_LAUNCH((sampler_multistep_kernel), grid, threads, 0, static_cast<cudaStream_t>(stream),
      x, v_cond, v_uncond, noise, x_next, x0_hist, t, P, Q, a, b, c, d, cfg_scale, cfg_scale_dev, per_sample, total);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return check_launch("sampler_multistep_kernel");
}

extern "C" int tair_timestep_embedding(const int64_t* t, void* out, int32_t B, int32_t dim, float max_period,
                                       void* stream) {
  TAIR_REQUIRE(t && out && B > 0 && dim > 0, "timestep_embedding: bad arguments");
  const int n = B * dim;
  TAIR_LAUNCH((timestep_embedding_kernel), (n + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream), 
      t, reinterpret_cast<__nv_bfloat16*>(out), B, dim, max_period);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return check_launch("timestep_embedding_kernel");
}

extern "C" int tair_nchw_to_nhwc_bf16(const float* in, void* out, int32_t B, int32_t C, int32_t HW, int32_t Cpad,
                                      void* stream) {
  TAIR_REQUIRE(in && out && B > 0 && C > 0 && HW > 0 && Cpad >= C, "nchw_to_nhwc: bad arguments");
  dim3 grid((HW + 31) / 32, (Cpad + 31) / 32, B), block(32, 8);
  TAIR_LAUNCH((nchw_to_nhwc_kernel), grid, block, 0, static_cast<cudaStream_t>(stream), 
      in, reinterpret_cast<__nv_bfloat16*>(out), C, HW, Cpad);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return check_launch("nchw_to_nhwc_kernel");
}

extern "C" int tair_nhwc_to_nchw_f32(const void* in, int64_t ld, float* out, int32_t B, int32_t C, int32_t HW,
                                     void* stream) {
  TAIR_REQUIRE(in && out && B > 0 && C > 0 && HW > 0 && ld >= C, "nhwc_to_nchw: bad arguments");
  dim3 grid((HW + 31) / 32, (C + 31) / 32, B), block(32, 8);
  TAIR_LAUNCH((nhwc_to_nchw_kernel), grid, block, 0, static_cast<cudaStream_t>(stream), 
      reinterpret_cast<const __nv_bfloat16*>(in), out, C, HW, ld);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return check_launch("nhwc_to_nchw_kernel");
}

extern "C" int tair_concat_add(const void* a, const void* b, const void* c, void* out, int64_t M, int32_t C1,
                               int32_t C2, void* stream) {
  TAIR_REQUIRE(a && b && out && M > 0 && C1 > 0 && C2 > 0, "concat_add: bad arguments");
  TAIR_REQUIRE(C1 % 8 == 0 && C2 % 8 == 0, "concat_add: channel counts must be multiples of 8");
  TAIR_REQUIRE(al16(a) && al16(b) && al16(out) && (!c || al16(c)), "concat_add: tensors must be 16-byte aligned");
  const int64_t n = M * ((C1 + C2) / 8);
  TAIR_LAUNCH((concat_add_kernel), (unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream), 
      reinterpret_cast<const uint4*>(a), reinterpret_cast<const uint4*>(b), reinterpret_cast<const uint4*>(c),
      reinterpret_cast<uint4*>(out), M, C1 / 8, C2 / 8);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return check_launch("concat_add_kernel");
}

extern "C" int tair_add_bf16(const void* a, const void* b, void* out, int64_t n, void* stream) {
  TAIR_REQUIRE(a && b && out && n > 0 && n % 8 == 0, "add: n must be a positive multiple of 8");
  TAIR_REQUIRE(al16(a) && al16(b) && al16(out), "add: tensors must be 16-byte aligned");
  const int64_t nv = n / 8;
  TAIR_LAUNCH((add_kernel), (unsigned)((nv + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream), 
      reinterpret_cast<const uint4*>(a), reinterpret_cast<const uint4*>(b), reinterpret_cast<uint4*>(out), nv);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return check_launch("add_kernel");
}

extern "C" int tair_upsample2x_nhwc(const void* in, void* out, int32_t B, int32_t H, int32_t W, int32_t C,
                                    void* stream) {
  TAIR_REQUIRE(in && out && B > 0 && H > 0 && W > 0 && C > 0 && C % 8 == 0, "upsample2x: bad arguments");
  TAIR_REQUIRE(al16(in) && al16(out), "upsample2x: tensors must be 16-byte aligned");
  const int64_t n = (int64_t)B * 4 * H * W * (C / 8);
  TAIR_LAUNCH((upsample2x_kernel), (unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream), 
      reinterpret_cast<const uint4*>(in), reinterpret_cast<uint4*>(out), B, H, W, C / 8);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return check_launch("upsample2x_kernel");
}

extern "C" int tair_softmax_rows_bf16(const void* x, int64_t ldx, void* y, int64_t ldy, int32_t rows, int32_t cols,
                                      float scale, void* stream) {
  TAIR_REQUIRE(x && y && rows > 0 && cols > 0, "softmax_rows: bad arguments");
  TAIR_REQUIRE(cols % 8 == 0 && cols <= 8192, "softmax_rows: cols must be a multiple of 8 and <= 8192 (got %d)", cols);
  TAIR_REQUIRE(ldx % 8 == 0 && ldy % 8 == 0 && ldx >= cols && ldy >= cols && al16(x) && al16(y),
               "softmax_rows: misaligned rows");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const __nv_bfloat16* xp = reinterpret_cast<const __nv_bfloat16*>(x);
  __nv_bfloat16* yp = reinterpret_cast<__nv_bfloat16*>(y);
  const float sl2 = scale * 1.4426950408889634f;
  const int warps = 4, grid = (rows + warps - 1) / warps;
  const int nvec = cols / 8;
  if (nvec <= 32) TAIR_LAUNCH((softmax_rows_kernel<1>), grid, warps * 32, 0, st, xp, ldx, yp, ldy, rows, cols, sl2);
  else if (nvec <= 128) TAIR_LAUNCH((softmax_rows_kernel<4>), grid, warps * 32, 0, st, xp, ldx, yp, ldy, rows, cols, sl2);
  else if (nvec <= 512) TAIR_LAUNCH((softmax_rows_kernel<16>), grid, warps * 32, 0, st, xp, ldx, yp, ldy, rows, cols, sl2);
  else TAIR_LAUNCH((softmax_rows_kernel<32>), grid, warps * 32, 0, st, xp, ldx, yp, ldy, rows, cols, sl2);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return check_launch("softmax_rows_kernel");
}

extern "C" int tair_transpose_bf16(const void* in, int64_t ldi, int64_t in_batch_stride, void* out, int64_t ldo,
                                   int64_t out_batch_stride, int32_t batch, int32_t R, int32_t C, void* stream) {
  TAIR_REQUIRE(in && out && batch > 0 && R > 0 && C > 0 && ldi >= C && ldo >= R, "transpose: bad arguments");
  dim3 grid((C + 31) / 32, (R + 31) / 32, batch), block(32, 8);
  TAIR_LAUNCH((transpose_bf16_kernel), grid, block, 0, static_cast<cudaStream_t>(stream), 
      reinterpret_cast<const __nv_bfloat16*>(in), ldi, in_batch_stride, reinterpret_cast<__nv_bfloat16*>(out), ldo,
      out_batch_stride, R, C);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return check_launch("transpose_bf16_kernel");
}

// ---- row gather (window partition / cyclic shift of the SwinIR blocks as one index map, swinir.py:37-66,262-281) and
// LeakyReLU (swinir.py:777-801) ----
namespace tair {
namespace {
__global__ void gather_rows_kernel(const uint4* __restrict__ x, int64_t ldx16, const int32_t* __restrict__ idx,
                                   uint4* __restrict__ y, int64_t ldy16, int64_t rows, int vec_per_row) {
  pdl_grid_sync();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= rows * vec_per_row) return;
  const int64_t r = t / vec_per_row;
  const int v = (int)(t - r * vec_per_row);
  y[r * ldy16 + v] = __ldg(x + (int64_t)__ldg(idx + r) * ldx16 + v);
}

__global__ void leaky_relu_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, int64_t n16, float slope) {
  pdl_grid_sync();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n16) return;
  const uint4 q = __ldg(x + t);
  const uint32_t in[4] = {q.x, q.y, q.z, q.w};
  uint32_t out[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 f = unpack_bf16(in[i]);
    f.x = f.x >= 0.f ? f.x : f.x * slope;
    f.y = f.y >= 0.f ? f.y : f.y * slope;
    out[i] = pack_bf16(f.x, f.y);
  }
  y[t] = make_uint4(out[0], out[1], out[2], out[3]);
}
}  // namespace
}  // namespace tair

extern "C" int tair_gather_rows_bf16(const void* x, int64_t ldx, const int32_t* idx, void* y, int64_t ldy, int64_t rows,
                                     int32_t cols, void* stream) {
  TAIR_REQUIRE(x && idx && y, "gather_rows: NULL pointer");
  TAIR_REQUIRE(rows > 0 && cols > 0 && cols % 8 == 0 && ldx % 8 == 0 && ldy % 8 == 0 && ldx >= cols && ldy >= cols,
               "gather_rows: cols and row strides must be multiples of 8");
  TAIR_REQUIRE((reinterpret_cast<uintptr_t>(x) % 16) == 0 && (reinterpret_cast<uintptr_t>(y) % 16) == 0,
               "gather_rows: tensors must be 16-byte aligned");
  const int vpr = cols / 8;
  const int64_t total = rows * vpr;
  TAIR_LAUNCH((tair::gather_rows_kernel), (unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream), 
      reinterpret_cast<const uint4*>(x), ldx / 8, idx, reinterpret_cast<uint4*>(y), ldy / 8, rows, vpr);
  tair::g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return tair::check_launch("gather_rows_kernel");
}

extern "C" int tair_leaky_relu_bf16(const void* x, void* y, int64_t n, float slope, void* stream) {
  TAIR_REQUIRE(x && y && n > 0 && n % 8 == 0, "leaky_relu: n must be a positive multiple of 8");
  TAIR_REQUIRE((reinterpret_cast<uintptr_t>(x) % 16) == 0 && (reinterpret_cast<uintptr_t>(y) % 16) == 0,
               "leaky_relu: tensors must be 16-byte aligned");
  const int64_t n16 = n / 8;
  TAIR_LAUNCH((tair::leaky_relu_kernel), (unsigned)((n16 + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream), 
      reinterpret_cast<const uint4*>(x), reinterpret_cast<uint4*>(y), n16, slope);
  tair::g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return tair::check_launch("leaky_relu_kernel");
}
