// vitk_norm.cu — LayerNorm forward / backward for the fp32 residual stream (HBM-bound kernels).
//
// Replaces aten::native_layer_norm(+_backward) at the reference's norm1/norm2/norm/fc_norm call
// sites (/root/reference/models/vision_transformer.py:148,163,603,616; timm LayerNorm, eps 1e-6).
// One warp owns one row: the row lives in registers (<= 1024 columns), statistics are two-pass in
// fp32, all global accesses are 16-byte (fp32) / 8-byte (bf16) vectors and fully coalesced.  The kernels are
// instantiated per row width (VPL float4 vectors per lane) with the column guards compiled out when D == 128*VPL.
// Large backward calls stream their rows through a per-warp shared-memory ring instead (second half of the file).
//
// Algorithmic bytes per row (D columns): fwd 4D (x) + 2D (y) + 8 (stats);
// bwd 2D (dy) + 4D (x) + 4D (g_in) + 4D (g_out) + 2D (gb) + 8.
#include "vitk_common.cuh"
#include "vitk_internal.h"

namespace {
using namespace vitk;

constexpr int MAXV = 8;  // float4 vectors per lane -> up to 1024 columns
constexpr int LN_WARPS = 8;

template <int VPL, bool EXACT>
__global__ void __launch_bounds__(LN_WARPS * 32)
ln_fwd_kernel(const float* __restrict__ x, long long ld_x, const float* __restrict__ gamma,
              const float* __restrict__ beta, __nv_bfloat16* __restrict__ y, long long ld_y,
              float* __restrict__ mean, float* __restrict__ rstd, long long rows, int dim, float eps) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * LN_WARPS + warp;
  if (row >= rows) return;
  const int nvec = dim >> 2;
  const float4* xr = reinterpret_cast<const float4*>(x + row * ld_x);
  float4 v[VPL];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int c = lane + i * 32;
    if (EXACT || c < nvec) {
      v[i] = xr[c];
      s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
  }
  const float mu = warp_sum(s) / (float)dim;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int c = lane + i * 32;
    if (EXACT || c < nvec) {
      const float a = v[i].x - mu, b = v[i].y - mu, cc = v[i].z - mu, d = v[i].w - mu;
      q += (a * a + b * b) + (cc * cc + d * d);
    }
  }
  const float rs = rsqrtf(warp_sum(q) / (float)dim + eps);
  if (lane == 0) {
    if (mean) mean[row] = mu;
    if (rstd) rstd[row] = rs;
  }
  uint2* yr = reinterpret_cast<uint2*>(y + row * ld_y);
  const float4* g4 = reinterpret_cast<const float4*>(gamma);
  const float4* b4 = reinterpret_cast<const float4*>(beta);
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int c = lane + i * 32;
    if (EXACT || c < nvec) {
      const float4 g = __ldg(g4 + c);
      const float4 b = __ldg(b4 + c);
      uint2 o;
      o.x = pack_bf16x2(fmaf((v[i].x - mu) * rs, g.x, b.x), fmaf((v[i].y - mu) * rs, g.y, b.y));
      o.y = pack_bf16x2(fmaf((v[i].z - mu) * rs, g.z, b.z), fmaf((v[i].w - mu) * rs, g.w, b.w));
      yr[c] = o;
    }
  }
}

// Backward.  VPL = float4 vectors per lane (dim <= 128 * VPL).  Register budget per lane: xhat (4*VPL),
// packed dy (2*VPL), prefetched g_in (4*VPL), dgamma/dbeta partials (8*VPL) -> 2 CTAs of 8 warps per SM at VPL = 6.
template <int VPL, bool EXACT>
__global__ void __launch_bounds__(LN_WARPS * 32, (VPL <= 6) ? 2 : 1)
ln_bwd_kernel(const __nv_bfloat16* __restrict__ dy, long long ld_dy, const float* __restrict__ x,
              long long ld_x, const float* __restrict__ mean, const float* __restrict__ rstd,
              const float* __restrict__ gamma, const float* __restrict__ g_in,
              float* __restrict__ g_out, long long ld_g, __nv_bfloat16* __restrict__ gb_out,
              const float* __restrict__ rowscale, int rows_per_group, float* __restrict__ dgamma,
              float* __restrict__ dbeta, long long rows, int dim) {
  extern __shared__ float red[];  // [2][dim]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nvec = dim >> 2;
  for (int i = threadIdx.x; i < 2 * dim; i += blockDim.x) red[i] = 0.f;
  __syncthreads();

  float4 ag[VPL], ab[VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    ag[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    ab[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const float4* gm4 = reinterpret_cast<const float4*>(gamma);
  const float inv_dim = 1.0f / (float)dim;

  for (long long row = (long long)blockIdx.x * LN_WARPS + warp; row < rows;
       row += (long long)gridDim.x * LN_WARPS) {
    const uint2* dyr = reinterpret_cast<const uint2*>(dy + row * ld_dy);
    const float4* xr = reinterpret_cast<const float4*>(x + row * ld_x);
    const float4* gir = g_in ? reinterpret_cast<const float4*>(g_in + row * ld_g) : nullptr;
    // issue every load of the row up front (dy, x, g_in): 3 * VPL independent 8/16-byte requests per lane
    uint2 dyp[VPL];
    float4 xh[VPL], gi[VPL];
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      const int c = lane + i * 32;
      if (EXACT || c < nvec) {
        dyp[i] = dyr[c];
        xh[i] = xr[c];
        gi[i] = gir ? gir[c] : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    const float mu = mean[row], rs = rstd[row];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      const int c = lane + i * 32;
      if (EXACT || c < nvec) {
        const float2 d0 = unpack_bf16x2(dyp[i].x), d1 = unpack_bf16x2(dyp[i].y);
        const float4 g = __ldg(gm4 + c);
        xh[i] = make_float4((xh[i].x - mu) * rs, (xh[i].y - mu) * rs, (xh[i].z - mu) * rs, (xh[i].w - mu) * rs);
        ab[i].x += d0.x; ab[i].y += d0.y; ab[i].z += d1.x; ab[i].w += d1.y;
        ag[i].x = fmaf(d0.x, xh[i].x, ag[i].x); ag[i].y = fmaf(d0.y, xh[i].y, ag[i].y);
        ag[i].z = fmaf(d1.x, xh[i].z, ag[i].z); ag[i].w = fmaf(d1.y, xh[i].w, ag[i].w);
        const float a0 = d0.x * g.x, a1 = d0.y * g.y, a2 = d1.x * g.z, a3 = d1.y * g.w;
        s1 += (a0 + a1) + (a2 + a3);
        s2 += (a0 * xh[i].x + a1 * xh[i].y) + (a2 * xh[i].z + a3 * xh[i].w);
      }
    }
    const float c1 = warp_sum(s1) * inv_dim;
    const float c2 = warp_sum(s2) * inv_dim;
    const float scale = (rowscale != nullptr) ? __ldg(rowscale + (unsigned)row / (unsigned)rows_per_group) : 1.0f;
    float4* gor = reinterpret_cast<float4*>(g_out + row * ld_g);
    uint2* gbr = gb_out ? reinterpret_cast<uint2*>(gb_out + row * (long long)dim) : nullptr;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      const int c = lane + i * 32;
      if (EXACT || c < nvec) {
        const float2 d0 = unpack_bf16x2(dyp[i].x), d1 = unpack_bf16x2(dyp[i].y);
        const float4 g = __ldg(gm4 + c);
        float4 r;
        r.x = fmaf(rs, d0.x * g.x - c1 - xh[i].x * c2, gi[i].x);
        r.y = fmaf(rs, d0.y * g.y - c1 - xh[i].y * c2, gi[i].y);
        r.z = fmaf(rs, d1.x * g.z - c1 - xh[i].z * c2, gi[i].z);
        r.w = fmaf(rs, d1.y * g.w - c1 - xh[i].w * c2, gi[i].w);
        gor[c] = r;
        if (gbr) {
          uint2 o;
          o.x = pack_bf16x2(r.x * scale, r.y * scale);
          o.y = pack_bf16x2(r.z * scale, r.w * scale);
          gbr[c] = o;
        }
      }
    }
  }

  // CTA-level reduction of the per-lane column partials, then one atomic per column per CTA.
  if (dgamma != nullptr || dbeta != nullptr) {
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      const int c = lane + i * 32;
      if (EXACT || c < nvec) {
        float* rg = red + c * 4;
        float* rb = red + dim + c * 4;
        atomicAdd(rg + 0, ag[i].x); atomicAdd(rg + 1, ag[i].y);
        atomicAdd(rg + 2, ag[i].z); atomicAdd(rg + 3, ag[i].w);
        atomicAdd(rb + 0, ab[i].x); atomicAdd(rb + 1, ab[i].y);
        atomicAdd(rb + 2, ab[i].z); atomicAdd(rb + 3, ab[i].w);
      }
    }
    __syncthreads();
    // one 16-byte reduction per 4 columns (every CTA of the grid hits the same 2*dim addresses at the end of the kernel)
    for (int i = threadIdx.x; i < (dim >> 2); i += blockDim.x) {
      const float4 a = *reinterpret_cast<const float4*>(red + i * 4);
      const float4 b = *reinterpret_cast<const float4*>(red + dim + i * 4);
      if (dgamma)
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dgamma + i * 4), "f"(a.x), "f"(a.y), "f"(a.z), "f"(a.w) : "memory");
      if (dbeta)
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dbeta + i * 4), "f"(b.x), "f"(b.y), "f"(b.z), "f"(b.w) : "memory");
    }
  }
}

template <int VPL, bool EXACT>
int launch_ln_bwd(const void* dy_bf16, int64_t ld_dy, const float* x, int64_t ld_x, const float* mean,
                  const float* rstd, const float* gamma, const float* g_in, float* g_out, int64_t ld_g,
                  void* gb_out_bf16, const float* rowscale, int32_t rows_per_group, float* dgamma, float* dbeta,
                  int64_t rows, int32_t dim, void* stream) {
  const long long want = (rows + LN_WARPS - 1) / LN_WARPS;
  const long long cap = (long long)vitk_num_sms() * ((VPL <= 6) ? 2 : 1);  // exactly one resident wave
  const unsigned grid = (unsigned)(want < cap ? want : cap);
  ln_bwd_kernel<VPL, EXACT><<<grid, LN_WARPS * 32, 2 * dim * sizeof(float), (cudaStream_t)stream>>>(
      (const __nv_bfloat16*)dy_bf16, ld_dy, x, ld_x, mean, rstd, gamma, g_in, g_out, ld_g,
      (__nv_bfloat16*)gb_out_bf16, rowscale, rows_per_group > 0 ? rows_per_group : 1, dgamma, dbeta, rows, dim);
  return vitk_check_launch("layernorm_bwd");
}

// ---- Backward, staged through shared memory by bulk async copies (TMA, 1-D) ------------------------------------------
// The register-resident kernel above keeps one row per warp in flight, computes between its loads and its stores, and
// is capped at 128 registers by its two CTAs per SM; ncu shows 59 % of its stall samples on the loads (long scoreboard) and
// its rate follows the SM clock: 119 us at 1.9 GHz, 150 us at the ~1.45 GHz a power-capped training step runs at
// (tools/ln_ctx_bench.py; a library copy of the same bytes does not move).  Here every warp owns a private ring in shared
// memory: one elected lane issues the three row copies (x, g_in, dy: 10*D bytes) of row k+stages with cp.async.bulk as soon
// as row k has been consumed, so the loads of the next row are in flight whatever the warp is computing and need no
// registers; 12 warps at up to 168 registers and, when D is exactly 128*VPL, no column guards (EXACT).  Measured at
// 50432 x 768: 110 us at either clock (5.6 TB/s of algorithmic bytes).  Sweep (warps, stages) at the capped clock:
// (6,2) 126 us, (8,2) 124, (9..12,2) 110-112, (9,3) 122 -- profiles/r01_ln_ring_sweep.txt.
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

constexpr int RING_MAX_STAGES = 4;   // the barrier slots reserved per warp; the host launches RING_STAGES of them
constexpr int RING_STAGES = 2;
constexpr int RING_MAX_WARPS = 16;

__host__ __device__ inline uint32_t ring_header_bytes(int dim, int warps) {
  return (uint32_t)((8 * dim + warps * RING_MAX_STAGES * 8 + 127) / 128 * 128);
}

template <int VPL, bool EXACT>
__global__ void __launch_bounds__((VPL <= 4 ? RING_MAX_WARPS : VPL <= 6 ? 12 : 8) * 32, 1)
ln_bwd_ring_kernel(const __nv_bfloat16* __restrict__ dy, long long ld_dy, const float* __restrict__ x,
                   long long ld_x, const float* __restrict__ mean, const float* __restrict__ rstd,
                   const float* __restrict__ gamma, const float* __restrict__ g_in,
                   float* __restrict__ g_out, long long ld_g, __nv_bfloat16* __restrict__ gb_out,
                   const float* __restrict__ rowscale, int rows_per_group, float* __restrict__ dgamma,
                   float* __restrict__ dbeta, long long rows, int dim, int stages) {
  extern __shared__ __align__(128) unsigned char ring_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nw = blockDim.x >> 5;
  const int nvec = dim >> 2;
  float* red = reinterpret_cast<float*>(ring_smem);  // [2][dim]
  uint64_t* bars = reinterpret_cast<uint64_t*>(ring_smem + 8 * dim) + warp * RING_MAX_STAGES;
  const uint32_t stage_bytes = 10u * (uint32_t)dim;  // x (4D) | g_in (4D) | dy (2D)
  unsigned char* ring = ring_smem + ring_header_bytes(dim, nw) + (size_t)warp * stages * stage_bytes;

  for (int i = threadIdx.x; i < 2 * dim; i += blockDim.x) red[i] = 0.f;
  if (lane == 0) {
    for (int s = 0; s < stages; ++s) mbar_init(bars + s, 1);
    fence_mbar_init();
  }
  __syncthreads();

  const long long first = (long long)blockIdx.x * nw + warp;
  const long long stride = (long long)gridDim.x * nw;
  const uint32_t tx_bytes = (g_in != nullptr ? 10u : 6u) * (uint32_t)dim;
  auto issue = [&](long long row, int s) {
    if (elect_one()) {
      unsigned char* st = ring + (size_t)s * stage_bytes;
      mbar_arrive_expect_tx(bars + s, tx_bytes);
      bulk_load_1d(st, x + row * ld_x, 4u * dim, bars + s);
      if (g_in != nullptr) bulk_load_1d(st + 4 * dim, g_in + row * ld_g, 4u * dim, bars + s);
      bulk_load_1d(st + 8 * dim, dy + row * ld_dy, 2u * dim, bars + s);
    }
    __syncwarp();
  };
  for (int s = 0; s < stages; ++s)
    if (first + s * stride < rows) issue(first + s * stride, s);

  float4 ag[VPL], ab[VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    ag[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    ab[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const float4* gm4 = reinterpret_cast<const float4*>(gamma);
  const float inv_dim = 1.0f / (float)dim;

  int s = 0;
  uint32_t parity = 0;
  for (long long row = first; row < rows; row += stride) {
    const float mu = __ldg(mean + row), rs = __ldg(rstd + row);
    const float scale = (rowscale != nullptr) ? __ldg(rowscale + (unsigned)row / (unsigned)rows_per_group) : 1.0f;
    mbar_wait(bars + s, parity);
    const unsigned char* st = ring + (size_t)s * stage_bytes;
    const float4* xs = reinterpret_cast<const float4*>(st);
    const float4* gs = reinterpret_cast<const float4*>(st + 4 * dim);
    const uint2* ds = reinterpret_cast<const uint2*>(st + 8 * dim);
    uint2 dyp[VPL];
    float4 xh[VPL];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      const int c = lane + i * 32;
      if (EXACT || c < nvec) {
        dyp[i] = ds[c];
        const float4 xv = xs[c];
        const float2 d0 = unpack_bf16x2(dyp[i].x), d1 = unpack_bf16x2(dyp[i].y);
        const float4 g = __ldg(gm4 + c);
        xh[i] = make_float4((xv.x - mu) * rs, (xv.y - mu) * rs, (xv.z - mu) * rs, (xv.w - mu) * rs);
        ab[i].x += d0.x; ab[i].y += d0.y; ab[i].z += d1.x; ab[i].w += d1.y;
        ag[i].x = fmaf(d0.x, xh[i].x, ag[i].x); ag[i].y = fmaf(d0.y, xh[i].y, ag[i].y);
        ag[i].z = fmaf(d1.x, xh[i].z, ag[i].z); ag[i].w = fmaf(d1.y, xh[i].w, ag[i].w);
        const float a0 = d0.x * g.x, a1 = d0.y * g.y, a2 = d1.x * g.z, a3 = d1.y * g.w;
        s1 += (a0 + a1) + (a2 + a3);
        s2 += (a0 * xh[i].x + a1 * xh[i].y) + (a2 * xh[i].z + a3 * xh[i].w);
      }
    }
    const float c1 = warp_sum(s1) * inv_dim;
    const float c2 = warp_sum(s2) * inv_dim;
    float4* gor = reinterpret_cast<float4*>(g_out + row * ld_g);
    uint2* gbr = gb_out ? reinterpret_cast<uint2*>(gb_out + row * (long long)dim) : nullptr;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      const int c = lane + i * 32;
      if (EXACT || c < nvec) {
        const float2 d0 = unpack_bf16x2(dyp[i].x), d1 = unpack_bf16x2(dyp[i].y);
        const float4 g = __ldg(gm4 + c);
        const float4 gi = (g_in != nullptr) ? gs[c] : make_float4(0.f, 0.f, 0.f, 0.f);
        float4 r;
        r.x = fmaf(rs, d0.x * g.x - c1 - xh[i].x * c2, gi.x);
        r.y = fmaf(rs, d0.y * g.y - c1 - xh[i].y * c2, gi.y);
        r.z = fmaf(rs, d1.x * g.z - c1 - xh[i].z * c2, gi.z);
        r.w = fmaf(rs, d1.y * g.w - c1 - xh[i].w * c2, gi.w);
        gor[c] = r;
        if (gbr) {
          uint2 o;
          o.x = pack_bf16x2(r.x * scale, r.y * scale);
          o.y = pack_bf16x2(r.z * scale, r.w * scale);
          gbr[c] = o;
        }
      }
    }
    // every lane has consumed the stage (its values are in registers): hand it back to the async proxy
    __syncwarp();
    const long long next = row + stages * stride;
    if (next < rows) {
      fence_proxy_async_smem();
      issue(next, s);
    }
    if (++s == stages) {
      s = 0;
      parity ^= 1u;
    }
  }

  if (dgamma != nullptr || dbeta != nullptr) {
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      const int c = lane + i * 32;
      if (EXACT || c < nvec) {
        float* rg = red + c * 4;
        float* rb = red + dim + c * 4;
        atomicAdd(rg + 0, ag[i].x); atomicAdd(rg + 1, ag[i].y);
        atomicAdd(rg + 2, ag[i].z); atomicAdd(rg + 3, ag[i].w);
        atomicAdd(rb + 0, ab[i].x); atomicAdd(rb + 1, ab[i].y);
        atomicAdd(rb + 2, ab[i].z); atomicAdd(rb + 3, ab[i].w);
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < (dim >> 2); i += blockDim.x) {
      const float4 a = *reinterpret_cast<const float4*>(red + i * 4);
      const float4 b = *reinterpret_cast<const float4*>(red + dim + i * 4);
      if (dgamma)
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dgamma + i * 4), "f"(a.x), "f"(a.y), "f"(a.z), "f"(a.w) : "memory");
      if (dbeta)
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dbeta + i * 4), "f"(b.x), "f"(b.y), "f"(b.z), "f"(b.w) : "memory");
    }
  }
}

// Largest warp count whose rings fit the 227 KB of one SM (0: does not fit, use the register-resident kernel).
inline int ring_warps(int dim) {
  const long long budget = 227 * 1024 - 1024;
  const int wmax = (dim <= 512 ? RING_MAX_WARPS : dim <= 768 ? 12 : 8);  // the launch bounds of VPL = 6 / 8
  for (int w = wmax; w >= 1; --w)
    if ((long long)ring_header_bytes(dim, w) + (long long)w * RING_STAGES * 10 * dim <= budget) return w;
  return 0;
}

template <int VPL, bool EXACT>
int launch_ln_bwd_ring(const void* dy_bf16, int64_t ld_dy, const float* x, int64_t ld_x, const float* mean,
                       const float* rstd, const float* gamma, const float* g_in, float* g_out, int64_t ld_g,
                       void* gb_out_bf16, const float* rowscale, int32_t rows_per_group, float* dgamma, float* dbeta,
                       int64_t rows, int32_t dim, int warps, void* stream) {
  const size_t smem = ring_header_bytes(dim, warps) + (size_t)warps * RING_STAGES * 10 * dim;
  static bool configured = false;  // per instantiation
  if (!configured) {
    if (cudaFuncSetAttribute(ln_bwd_ring_kernel<VPL, EXACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess)
      return vitk_check_launch("layernorm_bwd (shared memory opt-in)");
    configured = true;
  }
  const long long want = (rows + warps - 1) / warps;
  const long long cap = vitk_num_sms();
  const unsigned grid = (unsigned)(want < cap ? want : cap);
  ln_bwd_ring_kernel<VPL, EXACT><<<grid, warps * 32, smem, (cudaStream_t)stream>>>(
      (const __nv_bfloat16*)dy_bf16, ld_dy, x, ld_x, mean, rstd, gamma, g_in, g_out, ld_g,
      (__nv_bfloat16*)gb_out_bf16, rowscale, rows_per_group > 0 ? rows_per_group : 1, dgamma, dbeta, rows, dim, RING_STAGES);
  return vitk_check_launch("layernorm_bwd");
}

}  // namespace

extern "C" int vitk_layernorm_fwd(const float* x, int64_t ld_x, const float* gamma, const float* beta,
                                  void* y_bf16, int64_t ld_y, float* mean, float* rstd, int64_t rows,
                                  int32_t dim, float eps, void* stream) {
  VITK_REQUIRE(rows >= 0 && dim > 0, VITK_ERR_SHAPE, "layernorm_fwd: bad shape rows=%lld dim=%d", (long long)rows, dim);
  VITK_REQUIRE(dim % 4 == 0 && dim <= MAXV * 128, VITK_ERR_SHAPE, "layernorm_fwd: dim=%d must be a multiple of 4 and <= %d", dim, MAXV * 128);
  VITK_REQUIRE(ld_x % 4 == 0 && ld_y % 4 == 0, VITK_ERR_ALIGN, "layernorm_fwd: row pitches must be multiples of 4 elements");
  VITK_REQUIRE(((uintptr_t)x & 15) == 0 && ((uintptr_t)y_bf16 & 7) == 0 && ((uintptr_t)gamma & 15) == 0 && ((uintptr_t)beta & 15) == 0,
               VITK_ERR_ALIGN, "layernorm_fwd: pointers must be 16-byte aligned");
  if (rows == 0) return VITK_OK;
  const int vpl = (dim + 127) / 128;
#define VITK_LN_FWD_CASES(CALL) \
  if (vpl <= 2) { CALL(2); }    \
  else if (vpl <= 3) { CALL(3); } \
  else if (vpl <= 4) { CALL(4); } \
  else if (vpl <= 6) { CALL(6); } \
  else { CALL(8); }
  const unsigned grid = (unsigned)((rows + LN_WARPS - 1) / LN_WARPS);
#define VITK_LN_FWD_CALL(V)                                                                                   \
  do {                                                                                                        \
    auto kern = (dim == (V) * 128) ? ln_fwd_kernel<V, true> : ln_fwd_kernel<V, false>;                        \
    kern<<<grid, LN_WARPS * 32, 0, (cudaStream_t)stream>>>(x, ld_x, gamma, beta, (__nv_bfloat16*)y_bf16, ld_y, \
                                                           mean, rstd, rows, dim, eps);                       \
  } while (0)
  VITK_LN_FWD_CASES(VITK_LN_FWD_CALL)
#undef VITK_LN_FWD_CALL
#undef VITK_LN_FWD_CASES
  return vitk_check_launch("layernorm_fwd");
}

extern "C" int vitk_layernorm_bwd(const void* dy_bf16, int64_t ld_dy, const float* x, int64_t ld_x,
                                  const float* mean, const float* rstd, const float* gamma,
                                  const float* g_in, float* g_out, int64_t ld_g, void* gb_out_bf16,
                                  const float* rowscale, int32_t rows_per_group, float* dgamma,
                                  float* dbeta, int64_t rows, int32_t dim, void* stream) {
  // both kernels read x, g_in, gamma and write g_out as float4, read dy and write gb_out as 8-byte vectors
  VITK_REQUIRE_ALIGNED("layernorm_bwd", "x", x, 16);
  VITK_REQUIRE_ALIGNED("layernorm_bwd", "g_in", g_in, 16);
  VITK_REQUIRE_ALIGNED("layernorm_bwd", "g_out", g_out, 16);
  VITK_REQUIRE_ALIGNED("layernorm_bwd", "gamma", gamma, 16);
  VITK_REQUIRE_ALIGNED("layernorm_bwd", "dy", dy_bf16, 8);
  VITK_REQUIRE_ALIGNED("layernorm_bwd", "gb_out", gb_out_bf16, 8);
  VITK_REQUIRE_ALIGNED("layernorm_bwd", "dgamma", dgamma, 16);   // 16-byte vector reductions
  VITK_REQUIRE_ALIGNED("layernorm_bwd", "dbeta", dbeta, 16);
  VITK_REQUIRE(rows >= 0 && rows < (1LL << 31) && dim > 0, VITK_ERR_SHAPE, "layernorm_bwd: bad shape");
  VITK_REQUIRE(dim % 4 == 0 && dim <= MAXV * 128, VITK_ERR_SHAPE, "layernorm_bwd: dim=%d must be a multiple of 4 and <= %d", dim, MAXV * 128);
  VITK_REQUIRE(ld_x % 4 == 0 && ld_dy % 4 == 0 && ld_g % 4 == 0, VITK_ERR_ALIGN, "layernorm_bwd: row pitches must be multiples of 4 elements");
  VITK_REQUIRE(mean && rstd && g_out, VITK_ERR_SHAPE, "layernorm_bwd: mean/rstd/g_out required");
  if (rows == 0) return VITK_OK;
  const int vpl = (dim + 127) / 128;
  // bulk-copy path: 16-byte aligned rows of every stream (x and g_in are by the checks above)
  const int rw = ring_warps(dim);
  const bool ring_ok = rw > 0 && rows >= 4096 && dim % 8 == 0 && ld_dy % 8 == 0 && ((uintptr_t)dy_bf16 & 15) == 0;
  if (ring_ok) {
#define LN_RING_CASE(V)                                                                                              \
  return (dim == (V) * 128 ? launch_ln_bwd_ring<V, true> : launch_ln_bwd_ring<V, false>)(dy_bf16, ld_dy, x, ld_x, mean, rstd, gamma, g_in, g_out, ld_g, gb_out_bf16, rowscale, \
                               rows_per_group, dgamma, dbeta, rows, dim, rw, stream)
    if (vpl <= 2) LN_RING_CASE(2);
    if (vpl <= 3) LN_RING_CASE(3);
    if (vpl <= 4) LN_RING_CASE(4);
    if (vpl <= 6) LN_RING_CASE(6);
    LN_RING_CASE(8);
#undef LN_RING_CASE
  }
#define LN_BWD_CASE(V)                                                                                          \
  return launch_ln_bwd<V, false>(dy_bf16, ld_dy, x, ld_x, mean, rstd, gamma, g_in, g_out, ld_g, gb_out_bf16, rowscale, \
                          rows_per_group, dgamma, dbeta, rows, dim, stream)
  if (vpl <= 2) LN_BWD_CASE(2);
  if (vpl <= 3) LN_BWD_CASE(3);
  if (vpl <= 4) LN_BWD_CASE(4);
  if (vpl <= 6) LN_BWD_CASE(6);
  LN_BWD_CASE(8);
#undef LN_BWD_CASE
}
