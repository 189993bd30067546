// vitk_elementwise.cu — bandwidth-bound helpers of the ViT training step:
// patchify (im2col + cast), prefix-token rows, embedding backward, pooling, bias-gradient column
// sums, fused cross-entropy (soft-target / label-smoothing / KD) forward+backward, flat AdamW.
//
// Reference call sites: PatchEmbed + _pos_embed (/root/reference/models/vision_transformer.py:552-560,
// 743-780), global_pool_nlc (:419-441), losses (/root/reference/main.py:926-968, timm.loss),
// torch.optim.AdamW (/root/reference/optim_factory.py:248-249).
#include "vitk_common.cuh"
#include "vitk_internal.h"

namespace {
using namespace vitk;

// ------------------------------------------------------------------------------------------------
// patchify: fp32 NCHW -> bf16 [B*P, C*ps*ps], column order (c, ph, pw)
// ------------------------------------------------------------------------------------------------
// IDX: unsigned when the flat index fits 32 bits (the usual case) - the 64-bit divisions of the long long version are
// several hundred instructions per 32-byte load
template <typename IDX>
__global__ void patchify_kernel(const float* __restrict__ img, __nv_bfloat16* __restrict__ out,
                                int B, int C, int H, int W, int ps) {
  const long long total = (long long)B * C * H * (W / 8);
  const long long idx64 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx64 >= total) return;
  const IDX idx = (IDX)idx64;
  const IDX wv = (IDX)(W / 8);
  const int xv = (int)(idx % wv);
  IDX t = idx / wv;
  const int y = (int)(t % (IDX)H);
  t /= (IDX)H;
  const int c = (int)(t % (IDX)C);
  const int b = (int)(t / (IDX)C);
  const float4* src = reinterpret_cast<const float4*>(img + (((long long)b * C + c) * H + y) * W + xv * 8);
  const float4 a0 = __ldg(src), a1 = __ldg(src + 1);
  const int gw = W / ps, gh = H / ps;
  const int py = y / ps, ph = y - py * ps;
  const int x0 = xv * 8;
  const int px = x0 / ps, pw = x0 - px * ps;
  const long long row = (long long)b * gh * gw + (long long)py * gw + px;
  const int col = (c * ps + ph) * ps + pw;
  uint4 u;
  u.x = pack_bf16x2(a0.x, a0.y);
  u.y = pack_bf16x2(a0.z, a0.w);
  u.z = pack_bf16x2(a1.x, a1.y);
  u.w = pack_bf16x2(a1.z, a1.w);
  *reinterpret_cast<uint4*>(out + row * ((long long)C * ps * ps) + col) = u;
}

__global__ void prefix_rows_kernel(float* __restrict__ x, const float* __restrict__ tok,
                                   const float* __restrict__ pos, int B, int N, int D, int prefix) {
  const long long total = (long long)B * prefix * D;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int d = (int)(idx % D);
  const int j = (int)((idx / D) % prefix);
  const int b = (int)(idx / ((long long)D * prefix));
  x[((long long)b * N + j) * D + d] = tok[j * D + d] + pos[j * D + d];
}

// grid: (ceil(N*D/4 / 256), bchunks).  Thread owns one float4 column group of one token.
// gw > 0: gp is written in the padded row order of an image operand, row (b, gy, gx') = (b * gh + gy) * gwp + gx'.
__global__ void embed_bwd_kernel(const float* __restrict__ g, __nv_bfloat16* __restrict__ gp,
                                 float* __restrict__ dpos, float* __restrict__ dprefix0, float* __restrict__ dprefix1,
                                 int B, int N, int D, int prefix, int gw, int gwp) {
  const int dv = D / 4;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)N * dv) return;
  const int n = (int)(idx / dv);
  const int c = (int)(idx % dv);
  const int bper = (B + gridDim.y - 1) / gridDim.y;
  const int b0 = blockIdx.y * bper;
  const int b1 = min(B, b0 + bper);
  const int P = N - prefix;
  long long prow = n - prefix, rows_per_img = P;   // patch row inside the image, rows of gp per image
  if (gw > 0 && n >= prefix) {
    const int t = n - prefix, gy = t / gw;
    prow = (long long)gy * gwp + (t - gy * gw);
    rows_per_img = (long long)(P / gw) * gwp;
  }
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
  for (int b = b0; b < b1; ++b) {
    const float4 v = *reinterpret_cast<const float4*>(g + ((long long)b * N + n) * D + c * 4);
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    if (gp != nullptr && n >= prefix) {
      uint2 o;
      o.x = pack_bf16x2(v.x, v.y);
      o.y = pack_bf16x2(v.z, v.w);
      *reinterpret_cast<uint2*>(gp + ((long long)b * rows_per_img + prow) * D + c * 4) = o;
    }
  }
  if (b1 > b0) {
    if (dpos) {
      float* o = dpos + (long long)n * D + c * 4;
      atomicAdd(o + 0, acc.x); atomicAdd(o + 1, acc.y); atomicAdd(o + 2, acc.z); atomicAdd(o + 3, acc.w);
    }
    float* dpre = n == 0 ? dprefix0 : dprefix1;   // cls_token / dist_token gradient rows (may be NULL: frozen)
    if (n < prefix && dpre != nullptr) {
      float* o = dpre + c * 4;
      atomicAdd(o + 0, acc.x); atomicAdd(o + 1, acc.y); atomicAdd(o + 2, acc.z); atomicAdd(o + 3, acc.w);
    }
  }
}

// zero rows gx' in [gw, gwp) of every (b, gy) group of the padded gp: they multiply zero-filled image rows in the weight
// gradient, and 0 * garbage must not be NaN.  One thread per 8 bytes.
__global__ void embed_bwd_pad_kernel(__nv_bfloat16* __restrict__ gp, long long groups, int D, int gw, int gwp) {
  const int dv = D / 4, pad = gwp - gw;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= groups * pad * dv) return;
  const int c = (int)(idx % dv);
  const long long r = idx / dv;
  const long long grp = r / pad;
  const int k = (int)(r - grp * pad);
  *reinterpret_cast<uint2*>(gp + (grp * gwp + gw + k) * D + c * 4) = make_uint2(0u, 0u);
}

// pooled[b, d] = mean_{t >= prefix} x[b, t, d]   (mode 0)  or  x[b, 0, d]  (mode 1)
// grid: (ceil(D/4/64), B), block (64, 4): 4 token lanes reduced through smem.
__global__ void pool_fwd_kernel(const float* __restrict__ x, float* __restrict__ pooled, int N, int D,
                                int prefix, int mode) {
  __shared__ float4 part[4][64];
  const int c = blockIdx.x * 64 + threadIdx.x;
  const int b = blockIdx.y;
  const int dv = D / 4;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (c < dv) {
    if (mode == 1) {
      if (threadIdx.y == 0) acc = *reinterpret_cast<const float4*>(x + ((long long)b * N) * D + c * 4);
    } else {
      for (int t = prefix + threadIdx.y; t < N; t += 4) {
        const float4 v = *reinterpret_cast<const float4*>(x + ((long long)b * N + t) * D + c * 4);
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
      }
    }
  }
  part[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && c < dv) {
    float4 r = part[0][threadIdx.x];
    for (int k = 1; k < 4; ++k) {
      const float4 v = part[k][threadIdx.x];
      r.x += v.x; r.y += v.y; r.z += v.z; r.w += v.w;
    }
    if (mode == 0) {
      const float inv = 1.0f / (float)(N - prefix);
      r.x *= inv; r.y *= inv; r.z *= inv; r.w *= inv;
    }
    *reinterpret_cast<float4*>(pooled + (long long)b * D + c * 4) = r;
  }
}

// one block per token row (no per-thread 64-bit index arithmetic: the flat-index version spent ~300 instructions
// per 16-byte store on three 64-bit divisions)
__global__ void pool_bwd_kernel(const float* __restrict__ dpooled, float* __restrict__ g, int B, int N,
                                int D, int prefix, int mode) {
  const unsigned row = blockIdx.x;
  const unsigned b = row / (unsigned)N, t = row - b * (unsigned)N;
  const bool live = (mode == 1) ? (t == 0) : ((int)t >= prefix);
  const float inv = (mode == 0) ? 1.0f / (float)(N - prefix) : 1.0f;
  const float4* src = reinterpret_cast<const float4*>(dpooled + (long long)b * D);
  float4* dst = reinterpret_cast<float4*>(g + (long long)row * D);
  for (int c = threadIdx.x; c < D / 4; c += blockDim.x) {
    float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
    if (live) {
      r = __ldg(src + c);
      r.x *= inv; r.y *= inv; r.z *= inv; r.w *= inv;
    }
    dst[c] = r;
  }
}

// out[c] += sum_r x[r, c].  block (32, 8): 32 lanes x 8 columns each = 256 columns, 8 row lanes.
__global__ void colsum_bf16_kernel(const __nv_bfloat16* __restrict__ x, long long ld, float* __restrict__ out,
                                   long long rows, int cols) {
  __shared__ float part[8][256];
  const int c0 = blockIdx.x * 256 + threadIdx.x * 8;
  const long long rper = (rows + gridDim.y - 1) / gridDim.y;
  const long long r0 = (long long)blockIdx.y * rper;
  const long long r1 = min(rows, r0 + rper);
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (c0 < cols) {
#pragma unroll 4
    for (long long r = r0 + threadIdx.y; r < r1; r += 8) {
      const uint4 u = *reinterpret_cast<const uint4*>(x + r * ld + c0);
      const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
      acc[0] += a.x; acc[1] += a.y; acc[2] += b.x; acc[3] += b.y;
      acc[4] += c.x; acc[5] += c.y; acc[6] += d.x; acc[7] += d.y;
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) part[threadIdx.y][threadIdx.x * 8 + j] = acc[j];
  __syncthreads();
  const int tid = threadIdx.y * 32 + threadIdx.x;
  const int c = blockIdx.x * 256 + tid;
  if (c < cols) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += part[k][tid];
    atomicAdd(out + c, s);
  }
}

// ------------------------------------------------------------------------------------------------
// Fused cross-entropy forward + backward.  One CTA (256 threads) per batch row.
// ------------------------------------------------------------------------------------------------
constexpr int CE_THREADS = 256;
constexpr int CE_MAXPT = 16;  // up to 4096 classes

__device__ __forceinline__ float block_reduce(float v, bool is_max, float* sh) {
  v = is_max ? warp_max(v) : warp_sum(v);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) sh[warp] = v;
  __syncthreads();
  float r = sh[0];
#pragma unroll
  for (int i = 1; i < CE_THREADS / 32; ++i) r = is_max ? fmaxf(r, sh[i]) : r + sh[i];
  return r;
}

__global__ void __launch_bounds__(CE_THREADS)
ce_kernel(const float* __restrict__ logits, const float* __restrict__ soft, const long long* __restrict__ labels,
          float smoothing, const float* __restrict__ teacher, float alpha, float T,
          float* __restrict__ dlogits, float* __restrict__ row_loss, int B, int C) {
  __shared__ float sh[CE_THREADS / 32];
  const int b = blockIdx.x;
  const float* xr = logits + (long long)b * C;
  float xv[CE_MAXPT];
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < CE_MAXPT; ++i) {
    const int c = threadIdx.x + i * CE_THREADS;
    xv[i] = (c < C) ? xr[c] : -INFINITY;
    mx = fmaxf(mx, xv[i]);
  }
  mx = block_reduce(mx, true, sh);
  float se = 0.f;
#pragma unroll
  for (int i = 0; i < CE_MAXPT; ++i) {
    const int c = threadIdx.x + i * CE_THREADS;
    if (c < C) se += __expf(xv[i] - mx);
  }
  se = block_reduce(se, false, sh);
  const float lse = mx + __logf(se);

  // base term: -sum_c t_c * (x_c - lse)
  const long long label = (soft == nullptr && labels != nullptr) ? labels[b] : -1;
  const float off_v = smoothing / (float)C, on_v = 1.0f - smoothing + off_v;
  float tv[CE_MAXPT];
  float base = 0.f, tsum = 0.f;
#pragma unroll
  for (int i = 0; i < CE_MAXPT; ++i) {
    const int c = threadIdx.x + i * CE_THREADS;
    tv[i] = 0.f;
    if (c < C) {
      tv[i] = soft ? soft[(long long)b * C + c] : ((long long)c == label ? on_v : off_v);
      base -= tv[i] * (xv[i] - lse);
      tsum += tv[i];
    }
  }
  base = block_reduce(base, false, sh);
  tsum = block_reduce(tsum, false, sh);

  float kd = 0.f;
  float lse_s = 0.f, lse_t = 0.f;
  const float invT = 1.0f / T;
  if (teacher != nullptr) {
    const float* zr = teacher + (long long)b * C;
    float zmx = -INFINITY;
    float zv[CE_MAXPT];
#pragma unroll
    for (int i = 0; i < CE_MAXPT; ++i) {
      const int c = threadIdx.x + i * CE_THREADS;
      zv[i] = (c < C) ? zr[c] * invT : -INFINITY;
      zmx = fmaxf(zmx, zv[i]);
    }
    zmx = block_reduce(zmx, true, sh);
    float zs = 0.f, ss = 0.f;
#pragma unroll
    for (int i = 0; i < CE_MAXPT; ++i) {
      const int c = threadIdx.x + i * CE_THREADS;
      if (c < C) {
        zs += __expf(zv[i] - zmx);
        ss += __expf((xv[i] - mx) * invT);
      }
    }
    zs = block_reduce(zs, false, sh);
    ss = block_reduce(ss, false, sh);
    lse_t = zmx + __logf(zs);
    lse_s = mx * invT + __logf(ss);
#pragma unroll
    for (int i = 0; i < CE_MAXPT; ++i) {
      const int c = threadIdx.x + i * CE_THREADS;
      if (c < C) {
        const float lpt = zv[i] - lse_t;
        const float lps = xv[i] * invT - lse_s;
        const float pt = __expf(lpt);
        kd += pt * (lpt - lps);
        // stash p_t - p_s(T) contribution in zv for the gradient pass
        zv[i] = __expf(lps) - pt;
      }
    }
    kd = block_reduce(kd, false, sh);
    const float invB = 1.0f / (float)B;
#pragma unroll
    for (int i = 0; i < CE_MAXPT; ++i) {
      const int c = threadIdx.x + i * CE_THREADS;
      if (c < C) {
        const float p = __expf(xv[i] - lse);
        const float gbase = (p * tsum - tv[i]) * invB;
        dlogits[(long long)b * C + c] = (1.0f - alpha) * gbase + alpha * T * zv[i] * invB;
      }
    }
    if (threadIdx.x == 0) row_loss[b] = (1.0f - alpha) * base + alpha * T * T * kd;
  } else {
    const float invB = 1.0f / (float)B;
#pragma unroll
    for (int i = 0; i < CE_MAXPT; ++i) {
      const int c = threadIdx.x + i * CE_THREADS;
      if (c < C) {
        const float p = __expf(xv[i] - lse);
        dlogits[(long long)b * C + c] = (p * tsum - tv[i]) * invB;
      }
    }
    if (threadIdx.x == 0) row_loss[b] = base;
  }
}

__global__ void mean_rows_kernel(const float* __restrict__ row_loss, float* __restrict__ loss, int B) {
  __shared__ float sh[CE_THREADS / 32];
  float s = 0.f;
  for (int i = threadIdx.x; i < B; i += CE_THREADS) s += row_loss[i];
  s = block_reduce(s, false, sh);
  if (threadIdx.x == 0) loss[0] = s / (float)B;
}

__global__ void scale_cast_kernel(const float* __restrict__ in, const float* __restrict__ scale,
                                  __nv_bfloat16* __restrict__ out, long long n) {
  const float s = scale ? __ldg(scale) : 1.0f;
  const long long i4 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i4 + 3 < n) {
    const float4 v = *reinterpret_cast<const float4*>(in + i4);
    uint2 o;
    o.x = pack_bf16x2(v.x * s, v.y * s);
    o.y = pack_bf16x2(v.z * s, v.w * s);
    *reinterpret_cast<uint2*>(out + i4) = o;
  } else {
    for (long long i = i4; i < n; ++i) out[i] = __float2bfloat16(in[i] * s);
  }
}

// out_bf16[i] = in_f32[i] * rowscale[i / elems_per_group]   (DropPath scale applied to a gradient stream)
__global__ void rowscale_cast_kernel(const float* __restrict__ in, const float* __restrict__ rowscale,
                                     long long elems_per_group, __nv_bfloat16* __restrict__ out, long long n) {
  const long long i4 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i4 >= n) return;
  const float s = rowscale ? __ldg(rowscale + ((n < (1LL << 32) && elems_per_group < (1LL << 32)) ? (long long)((unsigned)i4 / (unsigned)elems_per_group)
                                                                                                  : i4 / elems_per_group))
                           : 1.0f;
  const float4 v = *reinterpret_cast<const float4*>(in + i4);
  uint2 o;
  o.x = pack_bf16x2(v.x * s, v.y * s);
  o.y = pack_bf16x2(v.z * s, v.w * s);
  *reinterpret_cast<uint2*>(out + i4) = o;
}

// ------------------------------------------------------------------------------------------------
// Flat AdamW
// ------------------------------------------------------------------------------------------------
constexpr int ADAMW_MAX_GROUPS = 8;
struct AdamwHyper {
  float lr[ADAMW_MAX_GROUPS];
  float wd[ADAMW_MAX_GROUPS];
  float beta1, beta2, eps, inv_bc1, inv_sqrt_bc2, grad_scale, ema_decay;
  int zero_grad;
};

__global__ void __launch_bounds__(256)
adamw_kernel(float* __restrict__ p, float* __restrict__ g, const __nv_bfloat16* __restrict__ g16,
             const float* __restrict__ gscale_dev, float* __restrict__ m, float* __restrict__ v,
             __nv_bfloat16* __restrict__ shadow, float* __restrict__ ema, long long n,
             const uint8_t* __restrict__ chunk_group, int chunk, const __grid_constant__ AdamwHyper h) {
  // (__grid_constant__: h.lr[grp] is read straight from the parameter bank; without it the dynamic index makes the
  //  compiler copy both arrays to local memory in every thread)
  const long long i4 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i4 >= n) return;
  const int grp = chunk_group ? chunk_group[(unsigned long long)i4 < 0xffffffffull ? (unsigned)i4 / (unsigned)chunk : i4 / chunk] : 0;
  const float lr = h.lr[grp], wd = h.wd[grp];
  float4 pv = *reinterpret_cast<float4*>(p + i4);
  float4 gv;
  if (g16 != nullptr) {   // the gradient as all-reduced in bf16 (data parallel); g is only zeroed below
    const uint2 u = *reinterpret_cast<const uint2*>(g16 + i4);
    const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y);
    gv = make_float4(a.x, a.y, b.x, b.y);
  } else {
    gv = *reinterpret_cast<float4*>(g + i4);
  }
  // 1/world of the gradient mean, times the clip coefficient left on the device by vitk_clip_coef (no host sync)
  const float gscale = gscale_dev != nullptr ? h.grad_scale * __ldg(gscale_dev) : h.grad_scale;
  float4 mv = *reinterpret_cast<float4*>(m + i4);
  float4 vv = *reinterpret_cast<float4*>(v + i4);
  const float decay = 1.0f - lr * wd;
  const float step = lr * h.inv_bc1;
#define VITK_ADAMW_ONE(P, G, M, V)                              \
  {                                                             \
    const float gg = (G) * gscale;                              \
    (P) *= decay;                                               \
    (M) = h.beta1 * (M) + (1.0f - h.beta1) * gg;                \
    (V) = h.beta2 * (V) + (1.0f - h.beta2) * gg * gg;           \
    const float denom = sqrtf(V) * h.inv_sqrt_bc2 + h.eps;      \
    (P) -= step * ((M) / denom);                                \
  }
  VITK_ADAMW_ONE(pv.x, gv.x, mv.x, vv.x)
  VITK_ADAMW_ONE(pv.y, gv.y, mv.y, vv.y)
  VITK_ADAMW_ONE(pv.z, gv.z, mv.z, vv.z)
  VITK_ADAMW_ONE(pv.w, gv.w, mv.w, vv.w)
#undef VITK_ADAMW_ONE
  *reinterpret_cast<float4*>(p + i4) = pv;
  *reinterpret_cast<float4*>(m + i4) = mv;
  *reinterpret_cast<float4*>(v + i4) = vv;
  if (h.zero_grad) *reinterpret_cast<float4*>(g + i4) = make_float4(0.f, 0.f, 0.f, 0.f);
  if (shadow) {
    uint2 o;
    o.x = pack_bf16x2(pv.x, pv.y);
    o.y = pack_bf16x2(pv.z, pv.w);
    *reinterpret_cast<uint2*>(shadow + i4) = o;
  }
  if (ema) {
    float4 e = *reinterpret_cast<float4*>(ema + i4);
    const float d = h.ema_decay;
    e.x = d * e.x + (1.0f - d) * pv.x; e.y = d * e.y + (1.0f - d) * pv.y;
    e.z = d * e.z + (1.0f - d) * pv.z; e.w = d * e.w + (1.0f - d) * pv.w;
    *reinterpret_cast<float4*>(ema + i4) = e;
  }
}

// Sum of squares, DETERMINISTIC: every data-parallel rank must derive bit-identical clip coefficients from bit-identical
// reduced gradients, so there are no floating-point atomics here.  Stage 1: a fixed grid, each block sums its grid-stride
// share in a fixed order and writes one partial; stage 2: one block adds the partials in index order.
constexpr int SUMSQ_BLOCKS = 1024;
template <typename T>
__global__ void __launch_bounds__(CE_THREADS) sumsq_partial_kernel(const T* __restrict__ x, long long n, float* __restrict__ partial) {
  __shared__ float sh[CE_THREADS / 32];
  constexpr int V = 16 / sizeof(T);   // elements per 16-byte load
  float s = 0.f;
  const long long stride = (long long)gridDim.x * blockDim.x * V;
  for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * V; i < n; i += stride) {
    if (i + V - 1 < n) {
      const uint4 u = *reinterpret_cast<const uint4*>(x + i);
      if constexpr (sizeof(T) == 4) {
        const float a = __uint_as_float(u.x), b = __uint_as_float(u.y), c = __uint_as_float(u.z), d = __uint_as_float(u.w);
        s += (a * a + b * b) + (c * c + d * d);
      } else {
        const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
        s += (a.x * a.x + a.y * a.y) + (b.x * b.x + b.y * b.y) + (c.x * c.x + c.y * c.y) + (d.x * d.x + d.y * d.y);
      }
    } else {
      for (long long j = i; j < n; ++j) {
        float v;
        if constexpr (sizeof(T) == 4) v = x[j]; else v = __bfloat162float(x[j]);
        s += v * v;
      }
    }
  }
  s = block_reduce(s, false, sh);
  if (threadIdx.x == 0) partial[blockIdx.x] = s;
}
__global__ void __launch_bounds__(CE_THREADS) sumsq_final_kernel(const float* __restrict__ partial, int nblocks, float* __restrict__ out) {
  __shared__ float sh[CE_THREADS / 32];
  float s = 0.f;
  for (int i = threadIdx.x; i < nblocks; i += CE_THREADS) s += partial[i];
  s = block_reduce(s, false, sh);
  if (threadIdx.x == 0) out[0] += s;
}

inline unsigned blocks_for(long long n, int per) { return (unsigned)((n + per - 1) / per); }

// coef = min(1, max_norm / (sqrt(sumsq) * grad_scale + 1e-6)): torch.nn.utils.clip_grad_norm_'s coefficient for the
// gradient mean (= the all-reduced SUM times grad_scale = 1/world).  Stays on the device; AdamW multiplies it in.
__global__ void clip_coef_kernel(const float* __restrict__ sumsq, float grad_scale, float max_norm, float* __restrict__ coef,
                                 float* __restrict__ norm) {
  const float nrm = sqrtf(sumsq[0]) * grad_scale;
  if (norm) norm[0] = nrm;
  coef[0] = fminf(1.0f, max_norm / (nrm + 1e-6f));
}

__global__ void scale_f32_kernel(float* __restrict__ x, const float* __restrict__ scale, long long n) {
  const float s = __ldg(scale);
  const long long i4 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i4 + 3 < n) {
    float4 v = *reinterpret_cast<float4*>(x + i4);
    v.x *= s; v.y *= s; v.z *= s; v.w *= s;
    *reinterpret_cast<float4*>(x + i4) = v;
  } else {
    for (long long i = i4; i < n; ++i) x[i] *= s;
  }
}

// ---------------------------------------------------------------------------------------------
// DropPath (timm drop_path, called from Block at /root/reference/models/vision_transformer.py:160-161, 172-178): every
// per-sample keep mask of one forward pass in ONE launch.  rs[row, b] = Bernoulli(1 - p[row]) / (1 - p[row]), rows in
// the order the reference draws them (block 0 attention branch, block 0 MLP branch, block 1 ...).  Counter-based
// Philox4x32-10 keyed by (seed, offset): reproducible under torch.manual_seed, no state on the device.
// ---------------------------------------------------------------------------------------------
constexpr int DROPPATH_MAX_ROWS = 128;
struct DropPathProbs { float p[DROPPATH_MAX_ROWS]; };

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

__global__ void droppath_masks_kernel(float* __restrict__ rs, int rows, int B, unsigned long long seed,
                                      unsigned long long offset, const __grid_constant__ DropPathProbs probs) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * B) return;
  const float keep = 1.0f - probs.p[idx / B];
  const uint4 r = philox4x32_10(make_uint4((uint32_t)idx, 0u, (uint32_t)offset, (uint32_t)(offset >> 32)),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const float u = (float)(r.x >> 8) * (1.0f / 16777216.0f);   // uniform in [0, 1)
  rs[idx] = (u < keep) ? (keep > 0.f ? 1.0f / keep : 1.0f) : 0.0f;
}


// ---------------------------------------------------------------------------------------------
// Mixup / CutMix on the device, in place, batch mode of timm.data.Mixup (constructed at
// /root/reference/main.py:622-629, applied at engine.py:259-262): image b is mixed with image B-1-b.
//   mixup : x_b <- x_b * lam + x_{B-1-b} * (1 - lam)          (two roundings, like x.mul_(lam).add_(x.flip(0).mul_(1-lam)))
//   cutmix: x_b[:, yl:yh, xl:xh] <- x_{B-1-b}[:, yl:yh, xl:xh]
// One thread handles the same float4 of both images of a pair, so the update is safe in place.
// ---------------------------------------------------------------------------------------------
__global__ void mixup_batch_kernel(float* __restrict__ x, long long pairs, long long per_img4, int Himg, int W4, float lam,
                                   float om, int use_cutmix, int yl, int yh, int xl, int xh) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= pairs * per_img4) return;
  const long long pr = idx / per_img4, off = idx - pr * per_img4;
  float4* a = reinterpret_cast<float4*>(x) + pr * per_img4 + off;
  float4* b = reinterpret_cast<float4*>(x) + (2 * pairs - 1 - pr) * per_img4 + off;
  float4 va = *a, vb = *b;
  if (!use_cutmix) {
    float4 ra, rb;
    ra.x = __fadd_rn(__fmul_rn(va.x, lam), __fmul_rn(vb.x, om)); rb.x = __fadd_rn(__fmul_rn(vb.x, lam), __fmul_rn(va.x, om));
    ra.y = __fadd_rn(__fmul_rn(va.y, lam), __fmul_rn(vb.y, om)); rb.y = __fadd_rn(__fmul_rn(vb.y, lam), __fmul_rn(va.y, om));
    ra.z = __fadd_rn(__fmul_rn(va.z, lam), __fmul_rn(vb.z, om)); rb.z = __fadd_rn(__fmul_rn(vb.z, lam), __fmul_rn(va.z, om));
    ra.w = __fadd_rn(__fmul_rn(va.w, lam), __fmul_rn(vb.w, om)); rb.w = __fadd_rn(__fmul_rn(vb.w, lam), __fmul_rn(va.w, om));
    *a = ra;
    *b = rb;
  } else {
    const long long row = off / W4;                 // (channel * H + y)
    const int y = (int)(row % Himg), x0 = (int)(off - row * W4) * 4;
    if (y < yl || y >= yh || x0 + 4 <= xl || x0 >= xh) return;
    float4 ra = va, rb = vb;
    if (x0 + 0 >= xl && x0 + 0 < xh) { ra.x = vb.x; rb.x = va.x; }
    if (x0 + 1 >= xl && x0 + 1 < xh) { ra.y = vb.y; rb.y = va.y; }
    if (x0 + 2 >= xl && x0 + 2 < xh) { ra.z = vb.z; rb.z = va.z; }
    if (x0 + 3 >= xl && x0 + 3 < xh) { ra.w = vb.w; rb.w = va.w; }
    *a = ra;
    *b = rb;
  }
}

// soft targets: out[b, c] = v(y_b == c) * lam + v(y_{B-1-b} == c) * (1 - lam), v = on / off value with label smoothing
__global__ void mixup_target_kernel(const long long* __restrict__ labels, float* __restrict__ out, int B, int C, float lam,
                                    float om, float on_value, float off_value) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)B * C) return;
  const int b = (int)(idx / C), c = (int)(idx - (long long)b * C);
  const float y1 = labels[b] == c ? on_value : off_value;
  const float y2 = labels[B - 1 - b] == c ? on_value : off_value;
  out[idx] = __fadd_rn(__fmul_rn(y1, lam), __fmul_rn(y2, om));
}


// ---------------------------------------------------------------------------------------------
// LayerScale (/root/reference/models/vision_transformer.py:80-106), backward side.
//   colscale_bf16: x[r, c] *= gamma[c] in place on the bf16 branch gradient that feeds the branch's dgrad / wgrad
//     (the forward multiplies the branch output by gamma inside the residual GEMM epilogue).
//   layerscale_grad: the branch output y = a W^T + b is never stored, but
//       dgamma_c = sum_r g[r,c] y[r,c] = sum_k W[c,k] (sum_r g[r,c] a[r,k]) + b_c sum_r g[r,c]
//     and the weight / bias gradients of the branch's last Linear, computed from the gamma-scaled gradient, are
//     dW[c,:] = gamma_c * (sum_r g[r,c] a[r,:]), db_c = gamma_c * sum_r g[r,c].  Hence
//       dgamma_c = (sum_k W[c,k] dW[c,k] + b_c db_c) / gamma_c,
//     linear in the (possibly accumulated, possibly all-reduced) dW: it is SET, not added.  One warp per channel.
// ---------------------------------------------------------------------------------------------
__global__ void colscale_bf16_kernel(__nv_bfloat16* __restrict__ x, const float* __restrict__ gamma, long long rows, int dim) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // one 16-byte unit
  const int per_row = dim >> 3;
  if (idx >= rows * per_row) return;
  const int c = (int)(idx % per_row) * 8;
  uint4* p = reinterpret_cast<uint4*>(x) + idx;
  uint4 u = *p;
  const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + c)), g1 = __ldg(reinterpret_cast<const float4*>(gamma + c + 4));
  float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), d = unpack_bf16x2(u.z), e = unpack_bf16x2(u.w);
  u.x = pack_bf16x2(a.x * g0.x, a.y * g0.y);
  u.y = pack_bf16x2(b.x * g0.z, b.y * g0.w);
  u.z = pack_bf16x2(d.x * g1.x, d.y * g1.y);
  u.w = pack_bf16x2(e.x * g1.z, e.y * g1.w);
  *p = u;
}

__global__ void layerscale_grad_kernel(const float* __restrict__ W, const float* __restrict__ dW, const float* __restrict__ b,
                                       const float* __restrict__ db, const float* __restrict__ gamma, float* __restrict__ dgamma,
                                       int C, int K) {
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (c >= C) return;
  const int lane = threadIdx.x & 31;
  const float4* w4 = reinterpret_cast<const float4*>(W + (long long)c * K);
  const float4* d4 = reinterpret_cast<const float4*>(dW + (long long)c * K);
  float acc = 0.f;
  for (int k = lane; k < (K >> 2); k += 32) {
    const float4 w = __ldg(w4 + k), d = d4[k];
    acc += w.x * d.x + w.y * d.y + w.z * d.z + w.w * d.w;
  }
  acc = warp_sum(acc);
  if (lane == 0) {
    if (b != nullptr) acc = fmaf(b[c], db[c], acc);
    const float g = gamma[c];
    dgamma[c] = g != 0.f ? acc / g : 0.f;
  }
}

}  // namespace

extern "C" int vitk_patchify(const float* img, void* patches_bf16, int32_t B, int32_t C, int32_t H, int32_t W,
                             int32_t ps, void* stream) {
  VITK_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0 && ps > 0, VITK_ERR_SHAPE, "patchify: bad shape");
  VITK_REQUIRE(H % ps == 0 && W % ps == 0 && ps % 8 == 0, VITK_ERR_SHAPE,
               "patchify: H=%d W=%d must be multiples of ps=%d and ps a multiple of 8", H, W, ps);
  VITK_REQUIRE(((uintptr_t)img & 15) == 0 && ((uintptr_t)patches_bf16 & 15) == 0, VITK_ERR_ALIGN, "patchify: unaligned");
  const long long total = (long long)B * C * H * (W / 8);
  if (total < (1LL << 32))
    patchify_kernel<unsigned><<<blocks_for(total, 256), 256, 0, (cudaStream_t)stream>>>(img, (__nv_bfloat16*)patches_bf16, B, C, H, W, ps);
  else
    patchify_kernel<long long><<<blocks_for(total, 256), 256, 0, (cudaStream_t)stream>>>(img, (__nv_bfloat16*)patches_bf16, B, C, H, W, ps);
  return vitk_check_launch("patchify");
}

extern "C" int vitk_prefix_rows(float* x, const float* prefix_tok, const float* pos, int32_t B, int32_t N, int32_t D,
                                int32_t prefix, void* stream) {
  VITK_REQUIRE(B > 0 && N > 0 && D > 0 && prefix >= 0 && prefix <= N, VITK_ERR_SHAPE, "prefix_rows: bad shape");
  if (prefix == 0) return VITK_OK;
  const long long total = (long long)B * prefix * D;
  prefix_rows_kernel<<<blocks_for(total, 256), 256, 0, (cudaStream_t)stream>>>(x, prefix_tok, pos, B, N, D, prefix);
  return vitk_check_launch("prefix_rows");
}

extern "C" int vitk_embed_bwd(const float* g, void* gp_bf16, float* dpos, float* dprefix0, float* dprefix1, int32_t B,
                              int32_t N, int32_t D, int32_t prefix, int32_t gw, int32_t gwp, void* stream) {
  VITK_REQUIRE_ALIGNED("embed_bwd", "g", g, 16);
  VITK_REQUIRE_ALIGNED("embed_bwd", "gp", gp_bf16, 8);
  VITK_REQUIRE(B > 0 && N > 0 && D > 0 && D % 4 == 0 && prefix >= 0 && prefix <= 2 && prefix <= N, VITK_ERR_SHAPE,
               "embed_bwd: bad shape (prefix must be 0, 1 or 2)");
  VITK_REQUIRE(gw == 0 || (gw > 0 && gwp >= gw && (N - prefix) % gw == 0), VITK_ERR_SHAPE,
               "embed_bwd: padded layout needs gwp >= gw > 0 and a whole number of patch-grid rows (gw=%d gwp=%d)", gw, gwp);
  const long long total = (long long)N * (D / 4);
  const int bchunks = B >= 32 ? 8 : 1;
  dim3 grid(blocks_for(total, 256), bchunks);
  embed_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(g, (__nv_bfloat16*)gp_bf16, dpos, dprefix0, dprefix1, B, N, D,
                                                           prefix, gw, gwp);
  int rc = vitk_check_launch("embed_bwd");
  if (rc || gp_bf16 == nullptr || gw == 0 || gwp == gw) return rc;
  const long long groups = (long long)B * ((N - prefix) / gw);
  embed_bwd_pad_kernel<<<blocks_for(groups * (gwp - gw) * (D / 4), 256), 256, 0, (cudaStream_t)stream>>>(
      (__nv_bfloat16*)gp_bf16, groups, D, gw, gwp);
  return vitk_check_launch("embed_bwd_pad");
}

extern "C" int vitk_pool_fwd(const float* x, float* pooled, int32_t B, int32_t N, int32_t D, int32_t prefix,
                             int32_t mode, void* stream) {
  VITK_REQUIRE_ALIGNED("pool_fwd", "x", x, 16);
  VITK_REQUIRE_ALIGNED("pool_fwd", "pooled", pooled, 16);
  VITK_REQUIRE(B > 0 && N > prefix && D > 0 && D % 4 == 0, VITK_ERR_SHAPE, "pool_fwd: bad shape");
  VITK_REQUIRE(mode == 0 || mode == 1, VITK_ERR_UNSUPPORTED, "pool_fwd: mode %d (0=avg, 1=token)", mode);
  dim3 grid(blocks_for(D / 4, 64), B), block(64, 4);
  pool_fwd_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(x, pooled, N, D, prefix, mode);
  return vitk_check_launch("pool_fwd");
}

extern "C" int vitk_pool_bwd(const float* dpooled, float* g, int32_t B, int32_t N, int32_t D, int32_t prefix,
                             int32_t mode, void* stream) {
  VITK_REQUIRE_ALIGNED("pool_bwd", "dpooled", dpooled, 16);
  VITK_REQUIRE_ALIGNED("pool_bwd", "g", g, 16);
  VITK_REQUIRE(B > 0 && N > prefix && D > 0 && D % 4 == 0, VITK_ERR_SHAPE, "pool_bwd: bad shape");
  VITK_REQUIRE(mode == 0 || mode == 1, VITK_ERR_UNSUPPORTED, "pool_bwd: mode %d (0=avg, 1=token)", mode);
  VITK_REQUIRE((long long)B * N < (1LL << 31), VITK_ERR_SHAPE, "pool_bwd: B * N must be below 2^31");
  const int threads = (D / 4 + 31) / 32 * 32;   // one float4 per thread up to D = 1024
  pool_bwd_kernel<<<(unsigned)((long long)B * N), threads < 256 ? threads : 256, 0, (cudaStream_t)stream>>>(dpooled, g, B, N, D, prefix, mode);
  return vitk_check_launch("pool_bwd");
}

extern "C" int vitk_colsum_bf16(const void* x_bf16, int64_t ld, float* out, int64_t rows, int32_t cols, void* stream) {
  VITK_REQUIRE_ALIGNED("colsum", "x", x_bf16, 16);
  VITK_REQUIRE(rows >= 0 && cols > 0 && cols % 8 == 0 && ld % 8 == 0, VITK_ERR_SHAPE, "colsum: cols/ld must be multiples of 8");
  if (rows == 0) return VITK_OK;
  const unsigned gx = blocks_for(cols, 256);
  long long gy = (long long)vitk_num_sms() * 4 / gx;
  if (gy < 1) gy = 1;
  const long long maxgy = (rows + 63) / 64;
  if (gy > maxgy) gy = maxgy;
  dim3 grid(gx, (unsigned)gy), block(32, 8);
  colsum_bf16_kernel<<<grid, block, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)x_bf16, ld, out, rows, cols);
  return vitk_check_launch("colsum_bf16");
}

extern "C" int vitk_ce_fwd_bwd(const float* logits, const float* soft_targets, const int64_t* labels, float smoothing,
                               const float* teacher_logits, float kd_alpha, float kd_temp, float* loss, float* dlogits,
                               float* row_loss_scratch, int32_t B, int32_t C, void* stream) {
  VITK_REQUIRE(B > 0 && C > 0 && C <= CE_THREADS * CE_MAXPT, VITK_ERR_SHAPE, "ce: C=%d must be in [1, %d]", C, CE_THREADS * CE_MAXPT);
  VITK_REQUIRE(soft_targets != nullptr || labels != nullptr, VITK_ERR_SHAPE, "ce: need soft_targets or labels");
  VITK_REQUIRE(loss && dlogits && row_loss_scratch, VITK_ERR_SHAPE, "ce: loss/dlogits/scratch required");
  if (teacher_logits != nullptr) VITK_REQUIRE(kd_temp > 0.f, VITK_ERR_SHAPE, "ce: kd_temp must be > 0");
  const float alpha = teacher_logits ? kd_alpha : 0.f;
  ce_kernel<<<B, CE_THREADS, 0, (cudaStream_t)stream>>>(logits, soft_targets, (const long long*)labels, smoothing,
                                                        teacher_logits, alpha, teacher_logits ? kd_temp : 1.f, dlogits,
                                                        row_loss_scratch, B, C);
  int rc = vitk_check_launch("ce");
  if (rc) return rc;
  mean_rows_kernel<<<1, CE_THREADS, 0, (cudaStream_t)stream>>>(row_loss_scratch, loss, B);
  return vitk_check_launch("ce_mean");
}

extern "C" int vitk_scale_cast_bf16(const float* in, const float* scale_dev, void* out_bf16, int64_t n, void* stream) {
  VITK_REQUIRE(n >= 0, VITK_ERR_SHAPE, "scale_cast: n < 0");
  VITK_REQUIRE(((uintptr_t)in & 15) == 0 && ((uintptr_t)out_bf16 & 7) == 0, VITK_ERR_ALIGN, "scale_cast: unaligned");
  if (n == 0) return VITK_OK;
  scale_cast_kernel<<<blocks_for((n + 3) / 4, 256), 256, 0, (cudaStream_t)stream>>>(in, scale_dev, (__nv_bfloat16*)out_bf16, n);
  return vitk_check_launch("scale_cast");
}

extern "C" int vitk_rowscale_cast_bf16(const float* in, const float* rowscale, int64_t elems_per_group, void* out_bf16,
                                       int64_t n, void* stream) {
  VITK_REQUIRE(n >= 0 && n % 4 == 0, VITK_ERR_SHAPE, "rowscale_cast: n must be a non-negative multiple of 4");
  VITK_REQUIRE(rowscale == nullptr || (elems_per_group > 0 && elems_per_group % 4 == 0), VITK_ERR_SHAPE,
               "rowscale_cast: elems_per_group must be a positive multiple of 4");
  VITK_REQUIRE(((uintptr_t)in & 15) == 0 && ((uintptr_t)out_bf16 & 7) == 0, VITK_ERR_ALIGN, "rowscale_cast: unaligned");
  if (n == 0) return VITK_OK;
  rowscale_cast_kernel<<<blocks_for(n / 4, 256), 256, 0, (cudaStream_t)stream>>>(in, rowscale, elems_per_group > 0 ? elems_per_group : 4,
                                                                                 (__nv_bfloat16*)out_bf16, n);
  return vitk_check_launch("rowscale_cast");
}

extern "C" int vitk_cast_bf16(const float* in, void* out_bf16, int64_t n, void* stream) {
  return vitk_scale_cast_bf16(in, nullptr, out_bf16, n, stream);
}

extern "C" int vitk_adamw_flat(float* p, float* g, const void* g_bf16, const float* grad_scale_dev, float* m, float* v,
                               void* shadow_bf16, float* ema, int64_t n, const uint8_t* chunk_group, int32_t chunk,
                               int32_t num_groups, const float* lr, const float* wd, float beta1, float beta2, float eps,
                               int64_t step, float grad_scale, float ema_decay, int32_t zero_grad, void* stream) {
  // float4 accesses to p, g, m, v, ema; 8-byte ones to g_bf16 and shadow.  g is read only without g_bf16, and written
  // only by zero_grad.
  VITK_REQUIRE_ALIGNED("adamw", "p", p, 16);
  if (g_bf16 == nullptr || zero_grad) VITK_REQUIRE_ALIGNED("adamw", "g", g, 16);
  VITK_REQUIRE_ALIGNED("adamw", "g_bf16", g_bf16, 8);
  VITK_REQUIRE_ALIGNED("adamw", "m", m, 16);
  VITK_REQUIRE_ALIGNED("adamw", "v", v, 16);
  VITK_REQUIRE_ALIGNED("adamw", "shadow", shadow_bf16, 8);
  VITK_REQUIRE_ALIGNED("adamw", "ema", ema, 16);
  VITK_REQUIRE(n >= 0 && n % 4 == 0, VITK_ERR_SHAPE, "adamw: n=%lld must be a multiple of 4", (long long)n);
  VITK_REQUIRE(num_groups >= 1 && num_groups <= ADAMW_MAX_GROUPS, VITK_ERR_SHAPE, "adamw: num_groups=%d not in [1,%d]", num_groups, ADAMW_MAX_GROUPS);
  VITK_REQUIRE(chunk_group == nullptr || (chunk > 0 && chunk % 4 == 0), VITK_ERR_SHAPE, "adamw: chunk must be a positive multiple of 4");
  VITK_REQUIRE(step >= 1, VITK_ERR_SHAPE, "adamw: step must be >= 1");
  VITK_REQUIRE(lr && wd, VITK_ERR_SHAPE, "adamw: lr/wd arrays required");
  if (n == 0) return VITK_OK;
  AdamwHyper h;
  for (int i = 0; i < ADAMW_MAX_GROUPS; ++i) {
    h.lr[i] = i < num_groups ? lr[i] : 0.f;
    h.wd[i] = i < num_groups ? wd[i] : 0.f;
  }
  h.beta1 = beta1; h.beta2 = beta2; h.eps = eps;
  const double bc1 = 1.0 - pow((double)beta1, (double)step);
  const double bc2 = 1.0 - pow((double)beta2, (double)step);
  h.inv_bc1 = (float)(1.0 / bc1);
  h.inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
  h.grad_scale = grad_scale; h.ema_decay = ema_decay; h.zero_grad = zero_grad;
  adamw_kernel<<<blocks_for(n / 4, 256), 256, 0, (cudaStream_t)stream>>>(p, g, (const __nv_bfloat16*)g_bf16, grad_scale_dev, m, v,
                                                                          (__nv_bfloat16*)shadow_bf16, ema, n, chunk_group,
                                                                          chunk > 0 ? chunk : 4, h);
  return vitk_check_launch("adamw");
}

extern "C" int vitk_clip_coef(const float* sumsq, float grad_scale, float max_norm, float* coef, float* norm, void* stream) {
  VITK_REQUIRE(sumsq && coef && max_norm > 0.f, VITK_ERR_SHAPE, "clip_coef: bad args");
  clip_coef_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(sumsq, grad_scale, max_norm, coef, norm);
  return vitk_check_launch("clip_coef");
}

extern "C" int vitk_scale_f32(float* x, const float* scale_dev, int64_t n, void* stream) {
  VITK_REQUIRE(n >= 0 && scale_dev, VITK_ERR_SHAPE, "scale_f32: bad args");
  VITK_REQUIRE(((uintptr_t)x & 15) == 0, VITK_ERR_ALIGN, "scale_f32: unaligned");
  if (n == 0) return VITK_OK;
  scale_f32_kernel<<<blocks_for((n + 3) / 4, 256), 256, 0, (cudaStream_t)stream>>>(x, scale_dev, n);
  return vitk_check_launch("scale_f32");
}

// ------------------------------------------------------------------------------------------------
// Dropout masks and the in-place multiplies that go with them (see include/vitk.h)
// ------------------------------------------------------------------------------------------------
// one Philox call -> 4 x 32 random bits -> 8 keep bytes (16 random bits per element: p is honoured to 2^-16)
__global__ void dropout_mask_kernel(uint8_t* __restrict__ mask, long long n, uint32_t thresh, unsigned long long seed,
                                    unsigned long long offset) {
  const long long i8 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i8 * 8 >= n) return;
  const uint4 r = philox4x32_10(make_uint4((uint32_t)i8, (uint32_t)(i8 >> 32), (uint32_t)offset, (uint32_t)(offset >> 32)),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
  uint32_t o[2] = {0u, 0u};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    o[k >> 1] |= ((w[k] & 0xffffu) >= thresh ? 1u : 0u) << (16 * (k & 1));
    o[k >> 1] |= ((w[k] >> 16) >= thresh ? 1u : 0u) << (16 * (k & 1) + 8);
  }
  if (i8 * 8 + 8 <= n) {
    *reinterpret_cast<uint2*>(mask + i8 * 8) = make_uint2(o[0], o[1]);
  } else {
    for (long long j = i8 * 8; j < n; ++j) mask[j] = (uint8_t)((o[(j & 7) >> 2] >> (8 * (j & 3))) & 0xffu);
  }
}

template <typename T, int V>   // V elements per thread: 8 bf16 (16 B) or 4 fp32 (16 B)
__global__ void mask_mul_kernel(T* __restrict__ x, long long ld_x, const uint8_t* __restrict__ mask, long long ld_mask,
                                long long rows, int cols, float scale) {
  const int per_row = cols / V;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * per_row) return;
  const long long r = idx / per_row;
  const int c = (int)(idx - r * per_row) * V;
  const uint8_t* mp = mask + r * ld_mask + c;
  float m[V];
#pragma unroll
  for (int j = 0; j < V; ++j) m[j] = mp[j] ? scale : 0.f;
  if constexpr (V == 8) {
    uint4* px = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(x) + r * ld_x + c);
    uint4 u = *px;
    float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c2 = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
    u.x = pack_bf16x2(a.x * m[0], a.y * m[1]);
    u.y = pack_bf16x2(b.x * m[2], b.y * m[3]);
    u.z = pack_bf16x2(c2.x * m[4], c2.y * m[5]);
    u.w = pack_bf16x2(d.x * m[6], d.y * m[7]);
    *px = u;
  } else {
    float4* px = reinterpret_cast<float4*>(reinterpret_cast<float*>(x) + r * ld_x + c);
    float4 u = *px;
    *px = make_float4(u.x * m[0], u.y * m[1], u.z * m[2], u.w * m[3]);
  }
}

extern "C" int vitk_dropout_mask(uint8_t* mask, int64_t n, float p, uint64_t seed, uint64_t offset, void* stream) {
  VITK_REQUIRE(mask != nullptr && n >= 0 && ((uintptr_t)mask & 15) == 0, VITK_ERR_ALIGN, "dropout_mask: 16-byte aligned mask required");
  VITK_REQUIRE(p >= 0.f && p < 1.f, VITK_ERR_SHAPE, "dropout_mask: p=%f not in [0, 1)", p);
  if (n == 0) return VITK_OK;
  const uint32_t thresh = (uint32_t)(p * 65536.f + 0.5f);   // keep iff a 16-bit uniform >= thresh
  dropout_mask_kernel<<<blocks_for((n + 7) / 8, 256), 256, 0, (cudaStream_t)stream>>>(mask, n, thresh, seed, offset);
  return vitk_check_launch("dropout_mask");
}

extern "C" int vitk_mask_mul_bf16(void* x, int64_t ld_x, const uint8_t* mask, int64_t ld_mask, int64_t rows, int32_t cols,
                                  float scale, void* stream) {
  VITK_REQUIRE(x && mask && rows >= 0 && cols > 0 && cols % 8 == 0 && ld_x % 8 == 0 && ((uintptr_t)x & 15) == 0, VITK_ERR_ALIGN,
               "mask_mul_bf16: cols and ld_x must be multiples of 8, x 16-byte aligned");
  if (rows == 0) return VITK_OK;
  mask_mul_kernel<__nv_bfloat16, 8><<<blocks_for(rows * (cols / 8), 256), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<__nv_bfloat16*>(x), ld_x, mask, ld_mask, rows, cols, scale);
  return vitk_check_launch("mask_mul_bf16");
}

extern "C" int vitk_mask_mul_f32(float* x, int64_t ld_x, const uint8_t* mask, int64_t ld_mask, int64_t rows, int32_t cols,
                                 float scale, void* stream) {
  VITK_REQUIRE(x && mask && rows >= 0 && cols > 0 && cols % 4 == 0 && ld_x % 4 == 0 && ((uintptr_t)x & 15) == 0, VITK_ERR_ALIGN,
               "mask_mul_f32: cols and ld_x must be multiples of 4, x 16-byte aligned");
  if (rows == 0) return VITK_OK;
  mask_mul_kernel<float, 4><<<blocks_for(rows * (cols / 4), 256), 256, 0, (cudaStream_t)stream>>>(x, ld_x, mask, ld_mask, rows, cols,
                                                                                                 scale);
  return vitk_check_launch("mask_mul_f32");
}

extern "C" int vitk_droppath_masks(float* rs, const float* drop_probs, int32_t rows, int32_t B, uint64_t seed, uint64_t offset,
                                   void* stream) {
  VITK_REQUIRE(rs && drop_probs && rows > 0 && rows <= DROPPATH_MAX_ROWS && B > 0, VITK_ERR_SHAPE,
               "droppath_masks: rows=%d (max %d) B=%d", rows, DROPPATH_MAX_ROWS, B);
  DropPathProbs pr;
  for (int i = 0; i < DROPPATH_MAX_ROWS; ++i) pr.p[i] = i < rows ? drop_probs[i] : 0.f;
  for (int i = 0; i < rows; ++i)
    VITK_REQUIRE(pr.p[i] >= 0.f && pr.p[i] <= 1.f, VITK_ERR_SHAPE, "droppath_masks: drop_probs[%d]=%f not in [0,1]", i, pr.p[i]);
  droppath_masks_kernel<<<blocks_for((long long)rows * B, 256), 256, 0, (cudaStream_t)stream>>>(rs, rows, B, seed, offset, pr);
  return vitk_check_launch("droppath_masks");
}

template <typename T>
static int sumsq_launch(const T* x, int64_t n, float* out, float* scratch, void* stream) {
  VITK_REQUIRE(n >= 0 && out && scratch, VITK_ERR_SHAPE, "sumsq: out and a scratch of vitk_sumsq_scratch_floats() fp32 required");
  VITK_REQUIRE(((uintptr_t)x & 15) == 0, VITK_ERR_ALIGN, "sumsq: x must be 16-byte aligned");
  if (n == 0) return VITK_OK;
  sumsq_partial_kernel<T><<<SUMSQ_BLOCKS, CE_THREADS, 0, (cudaStream_t)stream>>>(x, n, scratch);
  int rc = vitk_check_launch("sumsq");
  if (rc) return rc;
  sumsq_final_kernel<<<1, CE_THREADS, 0, (cudaStream_t)stream>>>(scratch, SUMSQ_BLOCKS, out);
  return vitk_check_launch("sumsq_final");
}
extern "C" int32_t vitk_sumsq_scratch_floats(void) { return SUMSQ_BLOCKS; }
extern "C" int vitk_sumsq(const float* x, int64_t n, float* out, float* scratch, void* stream) {
  return sumsq_launch<float>(x, n, out, scratch, stream);
}
extern "C" int vitk_sumsq_bf16(const void* x_bf16, int64_t n, float* out, float* scratch, void* stream) {
  return sumsq_launch<__nv_bfloat16>((const __nv_bfloat16*)x_bf16, n, out, scratch, stream);
}

extern "C" int vitk_mixup_batch(float* x, int32_t B, int32_t C, int32_t H, int32_t W, double lam, int32_t use_cutmix,
                                int32_t yl, int32_t yh, int32_t xl, int32_t xh, void* stream) {
  VITK_REQUIRE(x && B > 0 && C > 0 && H > 0 && W > 0, VITK_ERR_SHAPE, "mixup_batch: bad shape");
  VITK_REQUIRE(B % 2 == 0, VITK_ERR_SHAPE, "mixup_batch: batch size %d must be even", B);
  VITK_REQUIRE(W % 4 == 0 && ((uintptr_t)x & 15) == 0, VITK_ERR_ALIGN, "mixup_batch: W %% 4 == 0 and 16-byte alignment required");
  const long long per_img4 = (long long)C * H * W / 4, pairs = B / 2;
  const long long n = pairs * per_img4;
  mixup_batch_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, pairs, per_img4, H, W / 4, (float)lam, (float)(1.0 - lam), use_cutmix, yl,
                                                                                      yh, xl, xh);
  return vitk_check_launch("mixup_batch");
}

extern "C" int vitk_mixup_target(const int64_t* labels, float* out, int32_t B, int32_t C, double lam, double smoothing,
                                 void* stream) {
  VITK_REQUIRE(labels && out && B > 0 && C > 0, VITK_ERR_SHAPE, "mixup_target: bad shape");
  // lam, 1 - lam and the on / off values are formed in double and rounded once, like the Python scalars of the reference
  const double off_d = smoothing / (double)C;
  const float off_value = (float)off_d;
  const float on_value = (float)(1.0 - smoothing + off_d);
  const long long n = (long long)B * C;
  mixup_target_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>((const long long*)labels, out, B, C, (float)lam, (float)(1.0 - lam), on_value,
                                                                                       off_value);
  return vitk_check_launch("mixup_target");
}

extern "C" int vitk_colscale_bf16(void* x_bf16, const float* gamma, int64_t rows, int32_t dim, void* stream) {
  VITK_REQUIRE(x_bf16 && gamma && rows >= 0 && dim > 0 && dim % 8 == 0, VITK_ERR_SHAPE, "colscale_bf16: bad shape (dim %% 8 == 0)");
  VITK_REQUIRE(((uintptr_t)x_bf16 & 15) == 0 && ((uintptr_t)gamma & 15) == 0, VITK_ERR_ALIGN, "colscale_bf16: 16-byte alignment");
  if (rows == 0) return VITK_OK;
  const long long n = rows * (dim / 8);
  colscale_bf16_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>((__nv_bfloat16*)x_bf16, gamma, rows, dim);
  return vitk_check_launch("colscale_bf16");
}

extern "C" int vitk_layerscale_grad(const float* W, const float* dW, const float* bias, const float* dbias, const float* gamma,
                                    float* dgamma, int32_t C, int32_t K, void* stream) {
  VITK_REQUIRE(W && dW && gamma && dgamma && C > 0 && K > 0 && K % 4 == 0, VITK_ERR_SHAPE, "layerscale_grad: bad shape (K %% 4 == 0)");
  VITK_REQUIRE((bias == nullptr) == (dbias == nullptr), VITK_ERR_SHAPE, "layerscale_grad: bias and dbias go together");
  VITK_REQUIRE(((uintptr_t)W & 15) == 0 && ((uintptr_t)dW & 15) == 0, VITK_ERR_ALIGN, "layerscale_grad: 16-byte alignment");
  layerscale_grad_kernel<<<(unsigned)((C + 7) / 8), 256, 0, (cudaStream_t)stream>>>(W, dW, bias, dbias, gamma, dgamma, C, K);
  return vitk_check_launch("layerscale_grad");
}
