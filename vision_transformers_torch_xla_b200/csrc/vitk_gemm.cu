// vitk_gemm.cu — persistent warp-specialised tcgen05/TMEM bf16 GEMM for sm_100a.
//
//   D[M,N] = opA(A)[M,K] * opB(B)[N,K]^T      (fp32 accumulation in TMEM)
//
// Replaces the library GEMMs dispatched by the reference's nn.Linear / Conv2d-patchify
// call sites (SURVEY §2.4 K1,K4,K6,K7,K8,K10): qkv/proj (timm Attention via
// /root/reference/models/vision_transformer.py:149-159), fc1/fc2 (Mlp, :164-171), head (:618)
// and their dgrad/wgrad in autograd.
//
// Roles (1 CTA / SM, persistent over output tiles):
//   warp 0        TMA producer   (global -> 128B-swizzled smem ring, mbarrier tx-count)
//   warp 1        MMA issuer     (one elected thread: tcgen05.mma 128 x BLOCK_N x 16, cta_group::1)
//   warp 2        TMEM allocator
//   warps 4..     epilogue       (tcgen05.ld accumulator -> fused epilogue -> global); 8 warps, or 16
//                                for the GELU epilogue whose per-element math would otherwise outlast
//                                the K=768 main loop
// Accumulators are double-buffered in TMEM so tile i's epilogue overlaps tile i+1's MMAs.
//
// Operand layouts: "K-major" = stored [rows][K] (K contiguous), "MN-major" = stored [K][rows].
//   fprop  Y  = X  W^T   : A K-major,  B K-major   (W is [N,K] like nn.Linear.weight)
//   dgrad  dX = dY W     : A K-major,  B MN-major  (W itself, no transposed copy)
//   wgrad  dW = dY^T X   : A MN-major, B MN-major  (split-K, fp32 red.add into the grad buffer)
#include <cstring>

#include "vitk_common.cuh"
#include "vitk_internal.h"

namespace {

using namespace vitk;

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;  // 64 bf16 = 128 B = one swizzle row
constexpr int UMMA_K = 16;

struct GemmParams {
  int M, N, K;
  int num_m_tiles, num_n_tiles, num_k_blocks, splits;
  void* out;
  long long ld_out;
  void* aux;
  long long ld_aux;
  const float* bias;
  const float* resid;
  long long ld_resid;
  const float* rowscale;
  int rows_per_group;
  const float* colscale;
  const float* pos;
  int tokens_per_img;
  int prefix;
  int ragged;  // EPI_F32 only: N % 8 != 0 or unaligned rows -> scalar epilogue stores
  float* colsum_out;  // EPI_ATOMIC only: += column sums of A (bias gradient), or null
  // im2col-free patch view of a bf16 NCHW image (see include/vitk.h): which operand, and its geometry
  int a_image, b_image;
  int img_c, img_gh, img_gw, img_gwp, img_ps;
  // dropout keep-mask bytes [M, N] for the GELU / RESID epilogues (staged-panel variants), or null
  const uint8_t* mask;
  long long ld_mask;
  float mask_scale;
};

// One [8 patch rows][64 columns] piece of the patch matrix of an NCHW image (patch 16) = one TMA box (px, gx, y, bc) =
// (16, 8, 4, 1): four image rows of eight neighbouring patches of one channel.  With the 32-byte swizzle (a swizzle
// WIDER than the box's inner dimension would pad every 32-byte row to the swizzle span: tools/tma_probe.cu) it lands
// as [py 4][gx' 8][32 B] = four 256-byte atoms, which tcgen05 reads either as a K-major SW32 tile (8 rows x one 16-wide
// k-step per atom: the forward's A operand) or as an MN-major SW32 tile (8 k-rows x 16 columns per atom: the weight
// gradient's B operand).  Columns gx' >= gw of a patch-grid row and groups past the last image are zero-filled by TMA.
// A run of `n` consecutive 8-row groups starting at group `first` (= row / 8 of the padded row order (b, gy, gx')), all
// for the same 64 columns starting at col0 (c, py, px), box j going to dst + j * dst_stride.  Issued by ONE lane: the
// (image, grid row, part) of the first group costs two divisions, the others follow by increments (a division per box
// made the producer, not the tensor core, the limit: 25 us per 256 x 256 tile).
template <bool CTA2>
__device__ __forceinline__ void tma_load_patch_boxes(uint8_t* dst, uint32_t dst_stride, const CUtensorMap* tm, uint64_t* bar,
                                                     uint32_t bar_addr, const GemmParams& p, int first, int n, int col0) {
  const int per_row = p.img_gwp >> 3;                    // 8-patch groups per patch-grid row
  const int bgy = first / per_row;
  int part = first - bgy * per_row;
  int b = bgy / p.img_gh;
  int gy = bgy - b * p.img_gh;
  const int c = col0 >> 8, py0 = (col0 & 255) >> 4;      // patch 16: 256 columns per channel, 16 per image row
  for (int j = 0; j < n; ++j) {
    // (a group past the last image has b >= B: the bc coordinate is out of range and the box is zero-filled)
    if constexpr (CTA2) tma_load_4d_2cta(dst, tm, bar_addr, 0, part * 8, gy * 16 + py0, b * p.img_c + c);
    else tma_load_4d(dst, tm, bar, 0, part * 8, gy * 16 + py0, b * p.img_c + c);
    dst += dst_stride;
    if (++part == per_row) {
      part = 0;
      if (++gy == p.img_gh) { gy = 0; ++b; }
    }
  }
}

// EPI_PATCH: matrix row -> (output token row, pos_embed row), or orow < 0 for a pad row of an image operand
__device__ __forceinline__ void patch_row_map(const GemmParams& p, int row, long long& orow, int& prow) {
  int b = row / p.tokens_per_img;
  int t = row - b * p.tokens_per_img;
  orow = -1;
  prow = 0;
  if (row >= p.M) return;
  if (p.a_image) {   // padded rows (b, gy, gx'): gx' >= gw are zero padding, not tokens
    const int grp = row / p.img_gwp, gx = row - grp * p.img_gwp;
    if (gx >= p.img_gw) return;
    b = grp / p.img_gh;
    t = (grp - b * p.img_gh) * p.img_gw + gx;
  }
  orow = (long long)b * (p.tokens_per_img + p.prefix) + p.prefix + t;
  prow = p.prefix + t;
}

// Epilogue staging: every epilogue warp owns a private [32 rows][32 columns] panel in smem (4 KB for fp32
// columns, 2 KB for bf16) through which accumulator rows (thread = row) are transposed into row-contiguous
// order, so that every global load/store instruction touches whole 64/128-byte row segments.
template <int EPI>
constexpr uint32_t kStgBytes = (EPI == EPI_BF16) ? 2048u : 4096u;
// GELU / x GELU' epilogues with 64 columns per epilogue warp leave (and, for the aux operand, enter) through TMA:
// two [32 rows][64 B] panels per warp in the 64-byte-swizzle layout (see the epilogue branch of gemm_kernel).
template <int EPI, int PART_N>
constexpr bool kTmaEpi = (EPI == EPI_GELU || EPI == EPI_DGELU) && PART_N == 64;
// Residual epilogue through TMA: every epilogue warp owns a ring of three [32 rows][128 B] fp32 panels (128-byte
// swizzle).  The residual panels of the warp's tile sequence are loaded up to two panels ahead (across tile
// boundaries: the tile schedule is static), the sum is formed in place and leaves by a TMA store, so the epilogue
// issues no global loads / stores and keeps 1.5-2 panels per warp in flight instead of one.  (The single-CTA
// 256-column tile has no room for the rings next to three operand stages and keeps the register-prefetch path.)
// The rings take 96 KB, i.e. two of the six operand stages of the 256-wide CTA-pair tile: a win for the short-K,
// HBM-bound projection (K = 768: 123 -> 81 us per launch inside the training step) and a loss for the MMA-bound fc2
// (K = 3072: 183 -> 197 us), so the dispatcher picks this variant (internal epilogue code EPI_RESID_TMA) for K <= 1536.
constexpr int EPI_RESID_TMA = 100;
// bf16 epilogue through TMA (internal code): pairs of 32-column chunks leave as ONE [32 rows][128 B] box, so that every
// row segment reaching L2 is a whole line and the epilogue issues no global stores; taken whenever the warp's share of
// the tile is a multiple of 64 columns (BLOCK_N 128 and 256; the entry checks make every bf16 output TMA-compatible)
constexpr int EPI_BF16_TMA = 101;
constexpr int kResidTmaMaxK = 1536;
template <int EPI, int BLOCK_N, bool CTA2>
constexpr bool kTmaResid = (EPI == EPI_RESID_TMA);
constexpr int kResidBufs = 3;
template <int EPI, int BLOCK_N, bool CTA2>
constexpr uint32_t kStgBytesFor = kTmaResid<EPI, BLOCK_N, CTA2> ? kResidBufs * 4096u : kStgBytes<EPI>;
static_assert(kStgBytes<EPI_BF16_TMA> == 4096u, "one [32][128 B] panel per epilogue warp");

// CTA2: a pair of CTAs (cluster of 2, one TPC) computes a 256 x BLOCK_N tile with tcgen05.mma.cta_group::2.
// Each CTA stages its own 128 rows of A but only HALF of the B tile, so per-SM operand traffic from L2 (and smem
// write bandwidth) drops from 48 KB to 32 KB per 64-wide k-block at BLOCK_N = 256.
template <int BLOCK_N, int EW, uint32_t STG_BYTES, bool CTA2>
struct TileCfg {
  static constexpr int B_ROWS = CTA2 ? BLOCK_N / 2 : BLOCK_N;  // rows of the B tile staged by one CTA
  static constexpr uint32_t A_BYTES = BLOCK_M * BLOCK_K * 2;
  static constexpr uint32_t B_BYTES = B_ROWS * BLOCK_K * 2;
  static constexpr uint32_t STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr uint32_t STG_TOTAL = EW * STG_BYTES;
  static constexpr uint32_t SMEM_MAX = 232448;  // 227 KB
  static constexpr int STAGES_FIT = (SMEM_MAX - 1024 - 512 - STG_TOTAL) / STAGE_BYTES;
  static constexpr int STAGES = STAGES_FIT > 6 ? 6 : STAGES_FIT;
  static constexpr uint32_t TMEM_COLS = (2 * BLOCK_N <= 256) ? 256 : 512;
  static constexpr uint32_t SMEM_BYTES = STAGES * STAGE_BYTES + STG_TOTAL + 1024 /*align slack*/ + 512 /*barriers*/;
  static_assert(STAGES >= 3, "not enough shared memory for a 3-stage pipeline");
};

__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c),
               "f"(d)
               : "memory");
}

__device__ __forceinline__ uint4 pack8(const float* v) {
  uint4 u;
  u.x = pack_bf16x2(v[0], v[1]);
  u.y = pack_bf16x2(v[2], v[3]);
  u.z = pack_bf16x2(v[4], v[5]);
  u.w = pack_bf16x2(v[6], v[7]);
  return u;
}

// One 32-column chunk of one accumulator row, for the two epilogues that do not go through a staging panel: the
// ragged fp32 epilogue (scalar stores) and the split-K red.add.  `acc` holds the raw fp32 bits.
template <int EPI>
__device__ __forceinline__ void epilogue_chunk(const GemmParams& p, uint32_t (&acc)[32], int row, int col0) {
  if constexpr (EPI == EPI_F32) {
    // e.g. a 10- or 100-class head: rows are not 16-byte aligned, store scalars
    if (row >= p.M) return;
    float* o = reinterpret_cast<float*>(p.out) + (long long)row * p.ld_out + col0;
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (col0 + j < p.N) o[j] = __uint_as_float(acc[j]) + (p.bias ? __ldg(p.bias + col0 + j) : 0.f);
  } else if constexpr (EPI == EPI_ATOMIC) {
    // number of valid 8-column groups in this chunk (N % 8 == 0 is a host-side requirement)
    const int ngroups = min(4, (p.N - col0) >> 3);
    if (row >= p.M || ngroups <= 0) return;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      if (g >= ngroups) break;
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(acc[g * 8 + j]);
      float* o = reinterpret_cast<float*>(p.out) + (long long)row * p.ld_out + col0 + g * 8;
      red_add_v4(o, v[0], v[1], v[2], v[3]);
      red_add_v4(o + 4, v[4], v[5], v[6], v[7]);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Staged (coalesced) epilogue for one [32 rows x 32 columns] panel per warp.
//   fp32 panel: row pitch 128 B, 8 units of 16 B, unit u of row r lives at slot u ^ (r & 7)
//   bf16 panel: row pitch  64 B, 4 units of 16 B, unit u of row r lives at slot u ^ ((r >> 1) & 3)
// Both are conflict-free for "thread = row" accesses and for "8 (4) lanes per row" accesses.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t stg_f32(int r, int u) { return r * 128 + ((u ^ (r & 7)) << 4); }
__device__ __forceinline__ uint32_t stg_b16(int r, int u) { return r * 64 + ((u ^ ((r >> 1) & 3)) << 4); }

// global (row-contiguous) <-> staging, fp32: 8 instructions, each covering 4 rows x 128 B.  All loads of a panel
// are issued before the first dependent store (the compiler cannot prove smem/global do not alias).
template <bool LOAD>
__device__ __forceinline__ void panel_io_f32(uint8_t* stg, float* g, long long ld, int row0, int col0, int M, int N,
                                             int lane) {
  const int u = lane & 7, c = col0 + u * 4;
  float4 t[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int rr = i * 4 + (lane >> 3);
    const bool ok = (row0 + rr < M) && (c < N);
    if constexpr (LOAD) {
      if (ok) t[i] = __ldcs(reinterpret_cast<const float4*>(g + (long long)(row0 + rr) * ld + c));
    } else {
      t[i] = *reinterpret_cast<const float4*>(stg + stg_f32(rr, u));
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int rr = i * 4 + (lane >> 3);
    const bool ok = (row0 + rr < M) && (c < N);
    if constexpr (LOAD) {
      if (ok) *reinterpret_cast<float4*>(stg + stg_f32(rr, u)) = t[i];
    } else {
      if (ok) *reinterpret_cast<float4*>(g + (long long)(row0 + rr) * ld + c) = t[i];
    }
  }
}
// The same transfer split in two, so that the residual panel of the NEXT iteration is in flight (in registers) while
// the current panel is processed: global -> registers (issue), registers -> staging (once the buffer is free).
__device__ __forceinline__ void panel_ldg_f32(float4 (&t)[8], const float* g, long long ld, int row0, int col0, int M, int N,
                                              int lane) {
  const int u = lane & 7, c = col0 + u * 4;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int rr = i * 4 + (lane >> 3);
    t[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if ((row0 + rr < M) && (c < N)) t[i] = __ldcs(reinterpret_cast<const float4*>(g + (long long)(row0 + rr) * ld + c));
  }
}
__device__ __forceinline__ void panel_sts_f32(uint8_t* stg, const float4 (&t)[8], int lane) {
  const int u = lane & 7;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int rr = i * 4 + (lane >> 3);
    *reinterpret_cast<float4*>(stg + stg_f32(rr, u)) = t[i];
  }
}
// global <-> staging, bf16: 4 instructions, each covering 8 rows x 64 B
template <bool LOAD>
__device__ __forceinline__ void panel_io_b16(uint8_t* stg, __nv_bfloat16* g, long long ld, int row0, int col0, int M,
                                             int N, int lane) {
  const int u = lane & 3, c = col0 + u * 8;
  uint4 t[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int rr = i * 8 + (lane >> 2);
    const bool ok = (row0 + rr < M) && (c < N);
    if constexpr (LOAD) {
      if (ok) t[i] = __ldcs(reinterpret_cast<const uint4*>(g + (long long)(row0 + rr) * ld + c));
    } else {
      t[i] = *reinterpret_cast<const uint4*>(stg + stg_b16(rr, u));
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int rr = i * 8 + (lane >> 2);
    const bool ok = (row0 + rr < M) && (c < N);
    if constexpr (LOAD) {
      if (ok) *reinterpret_cast<uint4*>(stg + stg_b16(rr, u)) = t[i];
    } else {
      if (ok) *reinterpret_cast<uint4*>(g + (long long)(row0 + rr) * ld + c) = t[i];
    }
  }
}
__device__ __forceinline__ void row_put_b16(uint8_t* stg, int r, const float* v) {
#pragma unroll
  for (int u = 0; u < 4; ++u) *reinterpret_cast<uint4*>(stg + stg_b16(r, u)) = pack8(v + u * 8);
}
__device__ __forceinline__ void row_put_f32(uint8_t* stg, int r, const float* v) {
#pragma unroll
  for (int u = 0; u < 8; ++u)
    *reinterpret_cast<float4*>(stg + stg_f32(r, u)) = make_float4(v[u * 4], v[u * 4 + 1], v[u * 4 + 2], v[u * 4 + 3]);
}

// Dropout in the epilogue: this thread's 32 keep bytes (row `row`, columns col0 .. col0 + 31) -> v[j] *= keep ? scale : 0.
// Rows >= M and columns >= N are never stored, so they read as "drop" instead of touching memory.
__device__ __forceinline__ void load_keep_mask(const GemmParams& p, int row, int col0, uint32_t (&w)[8]) {
  const uint32_t* mp = reinterpret_cast<const uint32_t*>(p.mask + (long long)row * p.ld_mask + col0);
#pragma unroll
  for (int u = 0; u < 8; ++u) w[u] = (row < p.M && col0 + u * 4 < p.N) ? __ldg(mp + u) : 0u;
}
__device__ __forceinline__ void apply_keep_mask(const uint32_t (&w)[8], float scale, float (&v)[32]) {
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = ((w[j >> 2] >> ((j & 3) * 8)) & 0xffu) ? v[j] * scale : 0.f;
}

// `acc`: this thread's row (lane) of the panel, 32 fp32 accumulators.  row0 = first row of the warp's 32 rows.
template <int EPI>
__device__ __forceinline__ void epilogue_panel(const GemmParams& p, uint32_t (&acc)[32], uint8_t* stg, int lane,
                                               int row0, int col0, float rs) {
  float v[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(acc[j]);
  if constexpr (EPI != EPI_DGELU) {
    if (p.bias != nullptr) {
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        if (col0 + j < p.N) {
          const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + j));
          v[j] += b.x; v[j + 1] += b.y; v[j + 2] += b.z; v[j + 3] += b.w;
        }
      }
    }
  }
  if constexpr (EPI == EPI_BF16) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] *= rs;
    row_put_b16(stg, lane, v);
    __syncwarp();
    panel_io_b16<false>(stg, reinterpret_cast<__nv_bfloat16*>(p.out), p.ld_out, row0, col0, p.M, p.N, lane);
    __syncwarp();
  } else if constexpr (EPI == EPI_GELU) {
    // out = gelu(h), aux = gelu'(h): the backward epilogue (EPI_DGELU) is then a plain multiply
    float gd[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) gelu_fwd_bwd(v[j], v[j], gd[j]);
    if (p.mask != nullptr) {   // Mlp.drop1: the mask rides in the saved derivative too, the backward multiply stays as it is
      uint32_t w[8];
      load_keep_mask(p, row0 + lane, col0, w);
      apply_keep_mask(w, p.mask_scale, v);
      apply_keep_mask(w, p.mask_scale, gd);
    }
    row_put_b16(stg, lane, v);
    __syncwarp();
    panel_io_b16<false>(stg, reinterpret_cast<__nv_bfloat16*>(p.out), p.ld_out, row0, col0, p.M, p.N, lane);
    __syncwarp();
    row_put_b16(stg, lane, gd);
    __syncwarp();
    panel_io_b16<false>(stg, reinterpret_cast<__nv_bfloat16*>(p.aux), p.ld_aux, row0, col0, p.M, p.N, lane);
    __syncwarp();
  } else if constexpr (EPI == EPI_F32) {
    row_put_f32(stg, lane, v);
    __syncwarp();
    panel_io_f32<false>(stg, reinterpret_cast<float*>(p.out), p.ld_out, row0, col0, p.M, p.N, lane);
    __syncwarp();
  } else if constexpr (EPI == EPI_PATCH) {
    // acc + bias goes through the panel; on the way out every row adds its pos_embed row and lands on its token row
    // (8 lanes per row: 128-byte row segments for the pos_embed loads and the stores)
    row_put_f32(stg, lane, v);
    __syncwarp();
    const int u = lane & 7, c = col0 + u * 4;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int rr = i * 4 + (lane >> 3);
      long long orow;
      int prow;
      patch_row_map(p, row0 + rr, orow, prow);
      if (orow >= 0 && c < p.N) {
        float4 t = *reinterpret_cast<const float4*>(stg + stg_f32(rr, u));
        const float4 a = __ldg(reinterpret_cast<const float4*>(p.pos + (long long)prow * p.N + c));
        t.x += a.x; t.y += a.y; t.z += a.z; t.w += a.w;
        *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + orow * p.ld_out + c) = t;
      }
    }
    __syncwarp();
  } else if constexpr (EPI == EPI_RESID) {
    // the residual panel was loaded (coalesced) into the staging buffer by the caller before the TMEM wait
    if (p.mask != nullptr) {   // proj_drop / Mlp.drop2: on the branch (acc + bias), before LayerScale, DropPath and the residual
      uint32_t w[8];
      load_keep_mask(p, row0 + lane, col0, w);
      apply_keep_mask(w, p.mask_scale, v);
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      float4 cs = make_float4(rs, rs, rs, rs);
      if (p.colscale != nullptr && col0 + u * 4 < p.N) {
        const float4 cc = __ldg(reinterpret_cast<const float4*>(p.colscale + col0 + u * 4));
        cs.x *= cc.x; cs.y *= cc.y; cs.z *= cc.z; cs.w *= cc.w;
      }
      float4* sp = reinterpret_cast<float4*>(stg + stg_f32(lane, u));
      const float4 a = *sp;
      *sp = make_float4(fmaf(v[u * 4], cs.x, a.x), fmaf(v[u * 4 + 1], cs.y, a.y), fmaf(v[u * 4 + 2], cs.z, a.z),
                        fmaf(v[u * 4 + 3], cs.w, a.w));
    }
    __syncwarp();
    panel_io_f32<false>(stg, reinterpret_cast<float*>(p.out), p.ld_out, row0, col0, p.M, p.N, lane);
    __syncwarp();
  } else if constexpr (EPI == EPI_DGELU) {
    // out = acc * aux, aux = gelu'(h) (already staged by the caller)
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const uint4 du = *reinterpret_cast<const uint4*>(stg + stg_b16(lane, u));
      const float2 d0 = unpack_bf16x2(du.x), d1 = unpack_bf16x2(du.y), d2 = unpack_bf16x2(du.z), d3 = unpack_bf16x2(du.w);
      float* w = v + u * 8;
      w[0] *= d0.x * rs; w[1] *= d0.y * rs; w[2] *= d1.x * rs; w[3] *= d1.y * rs;
      w[4] *= d2.x * rs; w[5] *= d2.y * rs; w[6] *= d3.x * rs; w[7] *= d3.y * rs;
    }
    __syncwarp();
    row_put_b16(stg, lane, v);
    __syncwarp();
    panel_io_b16<false>(stg, reinterpret_cast<__nv_bfloat16*>(p.out), p.ld_out, row0, col0, p.M, p.N, lane);
    __syncwarp();
  }
}

template <int EPI>
constexpr bool kStaged = (EPI == EPI_BF16 || EPI == EPI_GELU || EPI == EPI_F32 || EPI == EPI_RESID || EPI == EPI_DGELU ||
                          EPI == EPI_PATCH);


// ROLES_HI: the three control warps (TMA, MMA, TMEM) take the HIGHEST warp ids.  The sub-partition issue arbiter
// favours higher warp ids (B300_MICROARCH.md: "hi-wid-first"), and a starved single-thread MMA issuer costs far
// more than a delayed epilogue instruction.
template <int BLOCK_N, bool A_MN, bool B_MN, int EPI, int EW, bool CTA2>
__global__ void __launch_bounds__(128 + EW * 32, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
            const __grid_constant__ CUtensorMap tmOut, const __grid_constant__ CUtensorMap tmAux, const GemmParams p) {
  constexpr uint32_t STG_BYTES = kStgBytesFor<EPI, BLOCK_N, CTA2>;
  using Cfg = TileCfg<BLOCK_N, EW, STG_BYTES, CTA2>;
  constexpr bool TMA_RESID = kTmaResid<EPI, BLOCK_N, CTA2>;
  constexpr bool TMA_BF16 = (EPI == EPI_BF16_TMA);
  constexpr int STAGES = Cfg::STAGES;
  constexpr bool ROLES_HI = true;
  constexpr int TILE_M = CTA2 ? 2 * BLOCK_M : BLOCK_M;
  constexpr int ACC_STAGES = 2;
  // wgrad with a fused bias gradient (EPI_ATOMIC, A MN-major): the otherwise idle epilogue warps are a second
  // consumer of every smem stage.  Once the MMAs of a stage have retired (mma_done) they add up the columns of the
  // A tile (= dY) straight out of shared memory and only then hand the slot back to the TMA producer.
  constexpr bool CS = (EPI == EPI_ATOMIC) && A_MN;
  // CTA pairs: each CTA stages half of the B tile.  MN-major B is loaded in 64-column chunks (BLOCK_N / 2 must be a
  // multiple of 64); K-major B is one box of BLOCK_N / 2 rows, so 192 works there too (96 rows per CTA)
  static_assert(!CTA2 || (BLOCK_N % 128 == 0) || (BLOCK_N == 192 && !B_MN), "CTA pairs need BLOCK_N in {128, 256} (192: K-major B only)");
  constexpr int PARTS = EW / 4;             // column partitions of the tile among epilogue warps
  constexpr int PART_N = BLOCK_N / PARTS;   // columns per epilogue warp
  static_assert(BLOCK_N % PARTS == 0 && PART_N % 32 == 0, "tile does not split into 32-column chunks per epilogue warp");

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* stg_base = smem + STAGES * Cfg::STAGE_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(stg_base + Cfg::STG_TOTAL);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* mma_done = tmem_empty + 2;  // [STAGES], used when CS
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mma_done + STAGES);
  uint64_t* aux_bar = mma_done + STAGES + 1;  // [EW] kTmaEpi x GELU': aux panels of the epilogue warp have landed

  const int hw_warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // logical warp: 0 = TMA, 1 = MMA, 2 = TMEM alloc, 3 = idle, 4.. = epilogue
  const int warp = ROLES_HI ? (hw_warp < EW ? hw_warp + 4 : hw_warp - EW) : hw_warp;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      // CTA2: the leader's barrier collects its own arrive.expect_tx plus the peer producer's remote arrive
      mbar_init(&full_bar[s], CTA2 ? 2 : 1);
      mbar_init(&empty_bar[s], CS ? EW : 1);  // CS: the epilogue warps release the slot after their column sums
      mbar_init(&mma_done[s], 1);
    }
    for (int s = 0; s < (TMA_RESID ? EW * kResidBufs : EW); ++s) mbar_init(&aux_bar[s], 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], CTA2 ? 2 * EW : EW);  // CTA2: epilogue warps of BOTH CTAs release the leader
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    if constexpr (CTA2) {
      tmem_alloc_2cta(tmem_slot, Cfg::TMEM_COLS);
      tmem_relinquish_2cta();
    } else {
      tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
      tmem_relinquish();
    }
  }
  if constexpr (CS) {
    for (int i = threadIdx.x; i < BLOCK_M; i += blockDim.x) reinterpret_cast<float*>(stg_base)[i] = 0.f;
  }
  tc_fence_before();
  if constexpr (CTA2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int total_units = p.num_m_tiles * p.num_n_tiles * p.splits;
  const uint32_t rank = CTA2 ? cluster_ctarank() : 0u;   // 0 = leader of the pair
  const int unit0 = CTA2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int ustride = CTA2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;

  if (warp == 0) {
    // ------------------------------ TMA producer ------------------------------
    // the whole warp runs the loops (uniform control flow keeps addresses / coordinates in uniform registers);
    // one elected lane issues the copies
    {
      int stage = 0;
      uint32_t phase = 0;
      for (int unit = unit0; unit < total_units; unit += ustride) {
        const int split = unit % p.splits;
        const int tile = unit / p.splits;
        const int n_blk = tile % p.num_n_tiles;
        const int m_blk = tile / p.num_n_tiles;
        const int kb0 = (int)(((long long)split * p.num_k_blocks) / p.splits);
        const int kb1 = (int)(((long long)(split + 1) * p.num_k_blocks) / p.splits);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (elect_one()) {
          uint8_t* sA = smem + stage * Cfg::STAGE_BYTES;
          uint8_t* sB = sA + Cfg::A_BYTES;
          const int a_row = m_blk * TILE_M + (int)rank * BLOCK_M;
          const int b_row = n_blk * BLOCK_N + (int)rank * Cfg::B_ROWS;
          if constexpr (CTA2) {
            // both CTAs credit their bytes to the LEADER's barrier (same smem offset, peer bit cleared)
            if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * Cfg::STAGE_BYTES);
            else mbar_arrive_remote(&full_bar[stage], 0);
            const uint32_t bar = smem_u32(&full_bar[stage]) & 0xFEFFFFFFu;
            if constexpr (!A_MN) {
              if (p.a_image) {
                tma_load_patch_boxes<true>(sA, 1024, &tmA, nullptr, bar, p, a_row / 8, BLOCK_M / 8, kb * BLOCK_K);
              } else {
                tma_load_2d_2cta(sA, &tmA, bar, kb * BLOCK_K, a_row);
              }
            } else {
#pragma unroll
              for (int c = 0; c < BLOCK_M / 64; ++c)
                tma_load_2d_2cta(sA + c * (BLOCK_K * 128), &tmA, bar, a_row + c * 64, kb * BLOCK_K);
            }
            if constexpr (!B_MN) {
              tma_load_2d_2cta(sB, &tmB, bar, kb * BLOCK_K, b_row);
            } else {
#pragma unroll
              for (int c = 0; c < Cfg::B_ROWS / 64; ++c) {
                if (p.b_image) {   // [8 k-row groups][B_ROWS / 64 column chunks][1 KB box]
                  tma_load_patch_boxes<true>(sB + c * 1024, (Cfg::B_ROWS / 64) * 1024, &tmB, nullptr, bar, p,
                                             kb * (BLOCK_K / 8), BLOCK_K / 8, b_row + c * 64);
                } else {
                  tma_load_2d_2cta(sB + c * (BLOCK_K * 128), &tmB, bar, b_row + c * 64, kb * BLOCK_K);
                }
              }
            }
          } else {
            mbar_arrive_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES);
            if constexpr (!A_MN) {
              if (p.a_image) {
                tma_load_patch_boxes<false>(sA, 1024, &tmA, &full_bar[stage], 0u, p, a_row / 8, BLOCK_M / 8, kb * BLOCK_K);
              } else {
                tma_load_2d(sA, &tmA, &full_bar[stage], kb * BLOCK_K, a_row);
              }
            } else {
#pragma unroll
              for (int c = 0; c < BLOCK_M / 64; ++c)
                tma_load_2d(sA + c * (BLOCK_K * 128), &tmA, &full_bar[stage], a_row + c * 64, kb * BLOCK_K);
            }
            if constexpr (!B_MN) {
              tma_load_2d(sB, &tmB, &full_bar[stage], kb * BLOCK_K, b_row);
            } else {
#pragma unroll
              for (int c = 0; c < BLOCK_N / 64; ++c) {
                if (p.b_image) {
                  tma_load_patch_boxes<false>(sB + c * 1024, (BLOCK_N / 64) * 1024, &tmB, &full_bar[stage], 0u, p,
                                              kb * (BLOCK_K / 8), BLOCK_K / 8, b_row + c * 64);
                } else {
                  tma_load_2d(sB + c * (BLOCK_K * 128), &tmB, &full_bar[stage], b_row + c * 64, kb * BLOCK_K);
                }
              }
            }
          }
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------ MMA issuer ------------------------------
    if (rank == 0) {  // CTA2: only the leader CTA issues (for both CTAs); whole warp loops, one elected lane issues
      constexpr uint32_t idesc = umma_idesc(TILE_M, BLOCK_N, 1 /*bf16*/, A_MN, B_MN);
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      // Descriptors are built once; per stage / per k-step only the 14-bit start-address field moves
      // (units of 16 B, never carries out of the field: smem < 256 KB).
      const uint32_t s0 = smem_u32(smem);
      // an image operand (32-byte-swizzle boxes, see tma_load_patch_boxes): A K-major = [16 row groups][4 k-steps][256 B],
      // B MN-major = [8 k-row groups][column chunks of 64][4 x 256 B]
      constexpr uint32_t B_SBO_IMG = (Cfg::B_ROWS / 64) * 1024;
      const uint64_t adesc0 = A_MN ? umma_desc_mnmajor(s0, BLOCK_K * 128)
                                   : (p.a_image ? umma_desc_kmajor_sw32(s0, 1024) : umma_desc_kmajor(s0));
      const uint64_t bdesc0 = B_MN ? (p.b_image ? umma_desc_mnmajor_sw32(s0 + Cfg::A_BYTES, 256, B_SBO_IMG)
                                                : umma_desc_mnmajor(s0 + Cfg::A_BYTES, BLOCK_K * 128))
                                   : umma_desc_kmajor(s0 + Cfg::A_BYTES);
      // K-major: 16 elements = 32 B inside the 128 B swizzle row.  MN-major: 16 k-rows = 2 swizzle atoms = 2048 B.
      // Image operands: one k-step = the next 256-byte atom (A), or two 8-k-row groups further (B).
      const uint32_t A_KSTEP = (A_MN ? 2048 : (p.a_image ? 256 : 32)) >> 4;
      const uint32_t B_KSTEP = (B_MN ? (p.b_image ? 2 * B_SBO_IMG : 2048) : 32) >> 4;
      for (int unit = unit0; unit < total_units; unit += ustride) {
        const int split = unit % p.splits;
        const int kb0 = (int)(((long long)split * p.num_k_blocks) / p.splits);
        const int kb1 = (int)(((long long)(split + 1) * p.num_k_blocks) / p.splits);
        mbar_wait(&tmem_empty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BLOCK_N;
        uint32_t accum = 0;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint64_t soff = (uint64_t)(stage * (Cfg::STAGE_BYTES >> 4));
          // once these MMAs retire: free the smem slot (in both CTAs), or (CS) wake the column-sum warps that free it
          uint64_t* done_bar = CS ? &mma_done[stage] : &empty_bar[stage];
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
              if constexpr (CTA2) umma_bf16_ss_2cta(d_tmem, adesc0 + soff + k * A_KSTEP, bdesc0 + soff + k * B_KSTEP, idesc, (k > 0) ? 1u : accum);
              else umma_bf16_ss(d_tmem, adesc0 + soff + k * A_KSTEP, bdesc0 + soff + k * B_KSTEP, idesc, (k > 0) ? 1u : accum);
            }
            if constexpr (CTA2) umma_commit_2cta_mc(done_bar, 3); else umma_commit(done_bar);
          }
          __syncwarp();
          accum = 1;
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        // accumulator complete -> epilogue (of both CTAs)
        if (elect_one()) {
          if constexpr (CTA2) umma_commit_2cta_mc(&tmem_full[as], 3); else umma_commit(&tmem_full[as]);
        }
        __syncwarp();
        if (++as == ACC_STAGES) { as = 0; aphase ^= 1; }
      }
    }
  } else if (warp >= 4) {
    // ------------------------------ epilogue ------------------------------
    const int ew = warp - 4;
    const int quad = hw_warp & 3;    // TMEM lane quadrant this (hardware) warp may access
    const int part = ew >> 2;        // column partition of the tile
    int as = 0;
    uint32_t aphase = 0;
    int cstage = 0;
    uint32_t cphase = 0;
    [[maybe_unused]] uint32_t tphase = 0;   // kTmaEpi x GELU': parity of this warp's aux barrier
    // TMA_RESID: this warp's panel sequence q = 0, 1, ... runs over its tiles (NP panels each); panel q lives in ring
    // buffer q % 3 and is announced on res_bar[q % 3]
    [[maybe_unused]] uint64_t* res_bar = aux_bar + ew * kResidBufs;
    [[maybe_unused]] uint8_t* ring = stg_base + ew * STG_BYTES;
    [[maybe_unused]] int rq = 0;            // sequence number of the panel being processed
    [[maybe_unused]] int rbuf = 0;          // rq % kResidBufs
    [[maybe_unused]] uint32_t rphase = 0;   // (rq / kResidBufs) & 1
    [[maybe_unused]] auto resid_issue = [&](int qq) {   // one elected lane: fetch the residual panel qq of the sequence
      constexpr int NP = PART_N / 32;
      const int u = unit0 + (qq / NP) * ustride;
      if (u >= total_units) return;
      const int nb = u % p.num_n_tiles, mb = u / p.num_n_tiles;
      const int b = qq % kResidBufs;
      mbar_arrive_expect_tx(&res_bar[b], 4096);
      tma_load_2d(ring + b * 4096, &tmAux, &res_bar[b], nb * BLOCK_N + part * PART_N + (qq % NP) * 32,
                  mb * TILE_M + (int)rank * BLOCK_M + quad * 32);
    };
    if constexpr (TMA_RESID) {
      if (elect_one()) {
        resid_issue(0);
        resid_issue(1);
      }
      __syncwarp();
    }
    for (int unit = unit0; unit < total_units; unit += ustride) {
      const int tile = unit / p.splits;
      const int n_blk = tile % p.num_n_tiles;
      const int m_blk = tile / p.num_n_tiles;
      const int row = m_blk * TILE_M + (int)rank * BLOCK_M + quad * 32 + lane;
      // The accumulator stage goes back to the MMA warp as soon as this warp has READ its last column out of TMEM:
      // the rest of the epilogue (math, staging, stores) then overlaps the MMAs of the tile after next.
      bool released = false;
      auto release_acc = [&]() {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (CTA2 && rank != 0) mbar_arrive_remote(&tmem_empty[as], 0);
          else mbar_arrive(&tmem_empty[as]);
        }
        released = true;
      };
      if constexpr (CS) {
        // second consumer of the smem ring: per k-block wait for the MMAs, (n_blk == 0 tiles only) add this thread's
        // 8 columns x 4 k-rows of the swizzled MN-major A tile, then release the slot to the producer
        const int split = unit % p.splits;
        const int kb0 = (int)(((long long)split * p.num_k_blocks) / p.splits);
        const int kb1 = (int)(((long long)(split + 1) * p.num_k_blocks) / p.splits);
        const bool colsum = p.colsum_out != nullptr && n_blk == 0;
        const int et = ew * 32 + lane;   // 0..255
        const int m8 = et & 15;          // 8-column group of the 128 tile rows (MN index)
        const int kg = et >> 4;          // k rows kg, kg+16, kg+32, kg+48
        float cs[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&mma_done[cstage], cphase);
          if (colsum) {
            const uint8_t* sA = smem + cstage * Cfg::STAGE_BYTES + (m8 >> 3) * (BLOCK_K * 128);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int k = kg + i * 16;
              const uint4 u = *reinterpret_cast<const uint4*>(sA + k * 128 + (((m8 & 7) ^ (k & 7)) << 4));
              const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
              cs[0] += a.x; cs[1] += a.y; cs[2] += b.x; cs[3] += b.y;
              cs[4] += c.x; cs[5] += c.y; cs[6] += d.x; cs[7] += d.y;
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&empty_bar[cstage]);
          if (++cstage == STAGES) { cstage = 0; cphase ^= 1; }
        }
        if (colsum) {
          float* red = reinterpret_cast<float*>(stg_base);  // [BLOCK_M], zero on entry
#pragma unroll
          for (int j = 0; j < 8; ++j) atomicAdd(red + m8 * 8 + j, cs[j]);
          asm volatile("bar.sync 1, %0;" ::"n"(EW * 32) : "memory");
          if (et < BLOCK_M) {
            const int r = m_blk * TILE_M + (int)rank * BLOCK_M + et;
            if (r < p.M) atomicAdd(p.colsum_out + r, red[et]);
            red[et] = 0.f;
          }
          asm volatile("bar.sync 1, %0;" ::"n"(EW * 32) : "memory");
        }
      }
      float rs = 1.0f;
      if constexpr (EPI == EPI_BF16 || EPI == EPI_BF16_TMA || EPI == EPI_RESID || EPI == EPI_RESID_TMA || EPI == EPI_DGELU) {
        if (p.rowscale != nullptr && row < p.M) rs = __ldg(p.rowscale + row / p.rows_per_group);
      }
      if constexpr (kTmaEpi<EPI, PART_N>) {
        // ---- TMA-staged epilogue: no global loads / stores, no bounds predicates (the tensor maps clip) ----
        // x GELU': one [32 rows][128 B] panel, 16-byte chunk u of row r at u ^ (r & 7) (128-byte swizzle);
        // GELU: two [32 rows][64 B] panels (gelu, gelu'), unit u of row r at u ^ ((r >> 1) & 3) (64-byte swizzle)
        uint8_t* buf0 = stg_base + ew * STG_BYTES;
        [[maybe_unused]] uint8_t* buf1 = buf0 + 2048;
        const int row0 = m_blk * TILE_M + (int)rank * BLOCK_M + quad * 32;
        const int colp = n_blk * BLOCK_N + part * PART_N;
        const uint32_t tacc = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + as * BLOCK_N + part * PART_N;
        if constexpr (EPI == EPI_DGELU) {
          // aux = gelu'(h) of this warp's [32 rows][64 columns] is fetched while the tile's MMAs still run: ONE box of
          // 128-byte rows (128-byte swizzle: chunk u of row r at u ^ (r & 7)), multiplied in place and stored as one box,
          // so every row segment that reaches L2 is a whole line (with two 64-byte boxes per row the L2 write hit
          // rate was exactly 50 %: every line arrived in two halves)
          if (elect_one()) {
            tma_store_wait_read();   // the previous tile's output panel has left the buffer
            mbar_arrive_expect_tx(&aux_bar[ew], 4096);
            tma_load_2d(buf0, &tmAux, &aux_bar[ew], colp, row0);
          }
          __syncwarp();
          mbar_wait(&tmem_full[as], aphase);
          tc_fence_after();
          uint32_t acc0[32], acc1[32];
          tmem_ld_32x32(tacc, acc0);
          tmem_ld_32x32(tacc + 32, acc1);
          mbar_wait(&aux_bar[ew], tphase);
          tmem_ld_wait();
          release_acc();
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            uint4* slot = reinterpret_cast<uint4*>(buf0 + lane * 128 + ((u ^ (lane & 7)) << 4));
            const uint4 du = *slot;
            const float2 d0 = unpack_bf16x2(du.x), d1 = unpack_bf16x2(du.y), d2 = unpack_bf16x2(du.z), d3 = unpack_bf16x2(du.w);
            const uint32_t* a = (u < 4 ? acc0 : acc1) + (u & 3) * 8;
            uint4 o;
            o.x = pack_bf16x2(__uint_as_float(a[0]) * (d0.x * rs), __uint_as_float(a[1]) * (d0.y * rs));
            o.y = pack_bf16x2(__uint_as_float(a[2]) * (d1.x * rs), __uint_as_float(a[3]) * (d1.y * rs));
            o.z = pack_bf16x2(__uint_as_float(a[4]) * (d2.x * rs), __uint_as_float(a[5]) * (d2.y * rs));
            o.w = pack_bf16x2(__uint_as_float(a[6]) * (d3.x * rs), __uint_as_float(a[7]) * (d3.y * rs));
            *slot = o;   // in place: every thread rewrites exactly the 128 bytes it read
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (elect_one()) {
            tma_store_2d(&tmOut, buf0, colp, row0);
            tma_store_commit();
          }
          __syncwarp();
          tphase ^= 1;
        } else {
          // bias of this warp's 64 columns -> L1 while the MMAs run
          if (p.bias != nullptr && lane < 2) asm volatile("prefetch.global.L1 [%0];" ::"l"(p.bias + colp + lane * 32));
          mbar_wait(&tmem_full[as], aphase);
          tc_fence_after();
#pragma unroll 1
          for (int hf = 0; hf < 2; ++hf) {
            const int col0 = colp + hf * 32;
            uint32_t acc[32];
            tmem_ld_32x32(tacc + hf * 32, acc);
            float4 bb[8];
#pragma unroll
            for (int j = 0; j < 8; ++j)
              bb[j] = (p.bias != nullptr && col0 + j * 4 < p.N) ? __ldg(reinterpret_cast<const float4*>(p.bias + col0) + j)
                                                               : make_float4(0.f, 0.f, 0.f, 0.f);
            tmem_ld_wait();
            if (hf == 1) release_acc();
            uint32_t act[16], der[16];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float a0, a1, a2, a3, g0, g1, g2, g3;
              gelu_fwd_bwd(__uint_as_float(acc[j * 4 + 0]) + bb[j].x, a0, g0);
              gelu_fwd_bwd(__uint_as_float(acc[j * 4 + 1]) + bb[j].y, a1, g1);
              gelu_fwd_bwd(__uint_as_float(acc[j * 4 + 2]) + bb[j].z, a2, g2);
              gelu_fwd_bwd(__uint_as_float(acc[j * 4 + 3]) + bb[j].w, a3, g3);
              act[j * 2] = pack_bf16x2(a0, a1);
              act[j * 2 + 1] = pack_bf16x2(a2, a3);
              der[j * 2] = pack_bf16x2(g0, g1);
              der[j * 2 + 1] = pack_bf16x2(g2, g3);
            }
            // the panels of the previous half (or tile) must have been read by the TMA unit before they are overwritten
            if (elect_one()) tma_store_wait_read();
            __syncwarp();
#pragma unroll
            for (int u = 0; u < 4; ++u)
              *reinterpret_cast<uint4*>(buf0 + stg_b16(lane, u)) = make_uint4(act[u * 4], act[u * 4 + 1], act[u * 4 + 2], act[u * 4 + 3]);
#pragma unroll
            for (int u = 0; u < 4; ++u)
              *reinterpret_cast<uint4*>(buf1 + stg_b16(lane, u)) = make_uint4(der[u * 4], der[u * 4 + 1], der[u * 4 + 2], der[u * 4 + 3]);
            fence_proxy_async_smem();
            __syncwarp();
            if (elect_one()) {
              tma_store_2d(&tmOut, buf0, col0, row0);
              tma_store_2d(&tmAux, buf1, col0, row0);
              tma_store_commit();
            }
            __syncwarp();
          }
        }
      } else if constexpr (TMA_BF16) {
        static_assert(PART_N % 64 == 0, "128-byte boxes are 64 bf16 columns wide");
        const int row0 = m_blk * TILE_M + (int)rank * BLOCK_M + quad * 32;
        uint8_t* buf = stg_base + ew * STG_BYTES;   // [32 rows][128 B], 16-byte chunk u of row r at u ^ (r & 7)
        mbar_wait(&tmem_full[as], aphase);
        tc_fence_after();
#pragma unroll 1
        for (int c = 0; c < PART_N / 64; ++c) {
          const int col_in_tile = part * PART_N + c * 64;
          const int col0 = n_blk * BLOCK_N + col_in_tile;
          const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + as * BLOCK_N + col_in_tile;
          uint32_t acc0[32], acc1[32];
          tmem_ld_32x32(taddr, acc0);
          tmem_ld_32x32(taddr + 32, acc1);
          tmem_ld_wait();
          if (c + 1 == PART_N / 64) release_acc();
          uint4 o[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const uint32_t* a = (u < 4 ? acc0 : acc1) + (u & 3) * 8;
            float4 b0 = make_float4(0.f, 0.f, 0.f, 0.f), b1 = b0;
            if (p.bias != nullptr && col0 + u * 8 < p.N) {
              b0 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + u * 8));
              b1 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + u * 8 + 4));
            }
            o[u].x = pack_bf16x2((__uint_as_float(a[0]) + b0.x) * rs, (__uint_as_float(a[1]) + b0.y) * rs);
            o[u].y = pack_bf16x2((__uint_as_float(a[2]) + b0.z) * rs, (__uint_as_float(a[3]) + b0.w) * rs);
            o[u].z = pack_bf16x2((__uint_as_float(a[4]) + b1.x) * rs, (__uint_as_float(a[5]) + b1.y) * rs);
            o[u].w = pack_bf16x2((__uint_as_float(a[6]) + b1.z) * rs, (__uint_as_float(a[7]) + b1.w) * rs);
          }
          // the previous box must have been read by the TMA unit before the panel is overwritten
          if (elect_one()) tma_store_wait_read();
          __syncwarp();
#pragma unroll
          for (int u = 0; u < 8; ++u) *reinterpret_cast<uint4*>(buf + lane * 128 + ((u ^ (lane & 7)) << 4)) = o[u];
          fence_proxy_async_smem();
          __syncwarp();
          if (elect_one()) {
            tma_store_2d(&tmOut, buf, col0, row0);
            tma_store_commit();
          }
          __syncwarp();
        }
      } else if constexpr (TMA_RESID) {
        const int row0 = m_blk * TILE_M + (int)rank * BLOCK_M + quad * 32;
        mbar_wait(&tmem_full[as], aphase);
        tc_fence_after();
#pragma unroll 1
        for (int c = 0; c < PART_N / 32; ++c) {
          const int col_in_tile = part * PART_N + c * 32;
          const int col0 = n_blk * BLOCK_N + col_in_tile;
          const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + as * BLOCK_N + col_in_tile;
          uint32_t acc[32];
          tmem_ld_32x32(taddr, acc);
          mbar_wait(&res_bar[rbuf], rphase);
          // panel rq + 2 goes into the buffer panel rq - 1 left by a TMA store issued one iteration ago
          if (elect_one()) {
            tma_store_wait_read();
            resid_issue(rq + 2);
          }
          __syncwarp();
          tmem_ld_wait();
          if (c + 1 == PART_N / 32) release_acc();
          uint8_t* buf = ring + rbuf * 4096;
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            float4 cs = make_float4(rs, rs, rs, rs);
            float4 bb = make_float4(0.f, 0.f, 0.f, 0.f);
            if (col0 + u * 4 < p.N) {
              if (p.bias != nullptr) bb = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + u * 4));
              if (p.colscale != nullptr) {
                const float4 cc = __ldg(reinterpret_cast<const float4*>(p.colscale + col0 + u * 4));
                cs.x *= cc.x; cs.y *= cc.y; cs.z *= cc.z; cs.w *= cc.w;
              }
            }
            float4* sp = reinterpret_cast<float4*>(buf + lane * 128 + ((u ^ (lane & 7)) << 4));
            const float4 a = *sp;
            *sp = make_float4(fmaf(__uint_as_float(acc[u * 4]) + bb.x, cs.x, a.x), fmaf(__uint_as_float(acc[u * 4 + 1]) + bb.y, cs.y, a.y),
                              fmaf(__uint_as_float(acc[u * 4 + 2]) + bb.z, cs.z, a.z), fmaf(__uint_as_float(acc[u * 4 + 3]) + bb.w, cs.w, a.w));
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (elect_one()) {
            tma_store_2d(&tmOut, buf, col0, row0);
            tma_store_commit();
          }
          __syncwarp();
          ++rq;
          if (++rbuf == kResidBufs) { rbuf = 0; rphase ^= 1; }
        }
      } else if constexpr (kStaged<EPI>) {
        uint8_t* stg = stg_base + ew * STG_BYTES;
        const int row0 = m_blk * TILE_M + (int)rank * BLOCK_M + quad * 32;
        const bool ragged = (EPI == EPI_F32) && p.ragged;
        // second operand of the first panel is fetched while the MMAs are still running; for the residual epilogue
        // panel c + 1 is in flight (registers) while panel c is processed
        [[maybe_unused]] float4 rnext[8];
        if constexpr (EPI == EPI_RESID)
          panel_ldg_f32(rnext, p.resid, p.ld_resid, row0, n_blk * BLOCK_N + part * PART_N, p.M, p.N, lane);
        if constexpr (EPI == EPI_DGELU)
          panel_io_b16<true>(stg, reinterpret_cast<__nv_bfloat16*>(p.aux), p.ld_aux, row0, n_blk * BLOCK_N + part * PART_N, p.M, p.N, lane);
        mbar_wait(&tmem_full[as], aphase);
        tc_fence_after();
#pragma unroll 1
        for (int c = 0; c < PART_N / 32; ++c) {
          const int col_in_tile = part * PART_N + c * 32;
          const int col0 = n_blk * BLOCK_N + col_in_tile;
          const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + as * BLOCK_N + col_in_tile;
          uint32_t acc[32];
          tmem_ld_32x32(taddr, acc);
          if constexpr (EPI == EPI_RESID) {
            if (!ragged) {
              panel_sts_f32(stg, rnext, lane);
              if (c + 1 < PART_N / 32) panel_ldg_f32(rnext, p.resid, p.ld_resid, row0, col0 + 32, p.M, p.N, lane);
            }
          }
          tmem_ld_wait();
          if (c + 1 == PART_N / 32) release_acc();
          if (ragged) {
            epilogue_chunk<EPI>(p, acc, row, col0);
          } else {
            if constexpr (EPI == EPI_RESID || EPI == EPI_DGELU) {
              if constexpr (EPI == EPI_DGELU) {
                if (c > 0)
                  panel_io_b16<true>(stg, reinterpret_cast<__nv_bfloat16*>(p.aux), p.ld_aux, row0, col0, p.M, p.N, lane);
              }
              __syncwarp();
            }
            epilogue_panel<EPI>(p, acc, stg, lane, row0, col0, rs);
          }
        }
      } else {
        mbar_wait(&tmem_full[as], aphase);
        tc_fence_after();
#pragma unroll 1
        for (int c = 0; c < PART_N / 32; ++c) {
          const int col_in_tile = part * PART_N + c * 32;
          const uint32_t taddr =
              tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + as * BLOCK_N + col_in_tile;
          uint32_t acc[32];
          tmem_ld_32x32(taddr, acc);
          tmem_ld_wait();
          if (c + 1 == PART_N / 32) release_acc();
          epilogue_chunk<EPI>(p, acc, row, n_blk * BLOCK_N + col_in_tile);
        }
      }
      if (!released) release_acc();
      if (++as == ACC_STAGES) { as = 0; aphase ^= 1; }
    }
    if constexpr (kTmaEpi<EPI, PART_N> || TMA_RESID || TMA_BF16) {
      if (elect_one()) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // smem must outlive the bulk stores
      __syncwarp();
    }
  }

  tc_fence_before();
  if constexpr (CTA2) cluster_sync_all(); else __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    if constexpr (CTA2) tmem_dealloc_2cta(tmem_base, Cfg::TMEM_COLS);
    else tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// number of images behind an image operand: its rows are (b, gy, gx') groups of img_gwp
inline long long image_batch(const vitk_gemm_args* a) {
  const long long rows = a->a_image ? a->M : a->K;
  const long long per_img = (long long)(a->img_h / a->img_patch) * a->img_gwp;
  return per_img > 0 ? (rows + per_img - 1) / per_img : 0;
}

int pick_splits(int tiles, int num_k_blocks, int slots, int block_n) {
  // Split-K factor of a weight gradient.  Cost model fitted to measurements (profiles/r02_wgrad_splits.txt): a CTA pair
  // runs its units one after the other; a unit costs its k-blocks plus the red.add epilogue of its fp32 tile, which is
  // NOT hidden behind the next unit's main loop and is worth ~45 k-blocks for a 256 x 256 tile (17-20 us on B200):
  //     time(s) ~ waves(s) * (ceil(k_blocks / s) + 45 * block_n / 256),   waves(s) = ceil(tiles * s / slots)
  // (round 1 charged 0.4 % of a wave per split, which sent ViT-L's 64-tile fc weight gradients to 8 splits:
  //  273 / 293 us against 225 / 220 us with one).
  const int epi = 45 * block_n / 256;
  int best = 1;
  long long best_cost = -1;
  for (int s = 1; s <= 32 && s <= num_k_blocks; ++s) {
    const long long waves = ((long long)tiles * s + slots - 1) / slots;
    const long long cost = waves * ((num_k_blocks + s - 1) / s + epi);
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = s; }
  }
  return best;
}

template <int BLOCK_N, bool A_MN, bool B_MN, int EPI, bool CTA2>
int launch_gemm(const vitk_gemm_args* a, cudaStream_t stream) {
  // 16 epilogue warps for the GELU epilogues (~20 instructions per element); 8 elsewhere.  With BLOCK_N = 192 and
  // 16 warps a warp's share is 48 columns, which is not a whole number of 32-column panels -> keep 8 there.
  constexpr int EW = ((EPI == EPI_GELU || EPI == EPI_DGELU) && BLOCK_N != 192) ? 16 : 8;
  using Cfg = TileCfg<BLOCK_N, EW, kStgBytesFor<EPI, BLOCK_N, CTA2>, CTA2>;
  constexpr int TILE_M = CTA2 ? 2 * BLOCK_M : BLOCK_M;
  CUtensorMap tmA, tmB;
  int rc;
  // the patch view of an NCHW image (patch 16): dims (px, gx, y, b*c) with strides (1, 16, W, H*W) elements, boxes of
  // (16 px, 8 patches, 4 image rows, 1) in the 32-byte swizzle
  auto image_map = [&](CUtensorMap* tm, const void* img) {
    return vitk_make_tmap_4d(tm, img, 2, 16, (uint64_t)(a->img_w / 16), (uint64_t)a->img_h,
                             (uint64_t)((long long)a->img_c * image_batch(a)), 16, (uint64_t)a->img_w,
                             (uint64_t)a->img_h * a->img_w, 16u, 8u, 4u, 1u, 32);
  };
  if (a->a_image) rc = image_map(&tmA, a->A);
  else if (!A_MN) rc = vitk_make_tmap_2d(&tmA, a->A, 2, a->K, a->M, a->lda, BLOCK_K, BLOCK_M);
  else            rc = vitk_make_tmap_2d(&tmA, a->A, 2, a->M, a->K, a->lda, 64, BLOCK_K);
  if (rc) return rc;
  if (a->b_image) rc = image_map(&tmB, a->B);
  else if (!B_MN) rc = vitk_make_tmap_2d(&tmB, a->B, 2, a->K, a->N, a->ldb, BLOCK_K, Cfg::B_ROWS);
  else            rc = vitk_make_tmap_2d(&tmB, a->B, 2, a->N, a->K, a->ldb, 64, BLOCK_K);
  if (rc) return rc;

  CUtensorMap tmOut, tmAux;
  memset(&tmOut, 0, sizeof(tmOut));
  memset(&tmAux, 0, sizeof(tmAux));
  if (EPI == EPI_BF16_TMA) {
    rc = vitk_make_tmap_2d(&tmOut, a->out, 2, a->N, a->M, a->ld_out, 64, 32);
    if (rc) return rc;
  }
  if (kTmaResid<EPI, BLOCK_N, CTA2>) {
    rc = vitk_make_tmap_2d(&tmOut, a->out, 4, a->N, a->M, a->ld_out, 32, 32);
    if (rc) return rc;
    rc = vitk_make_tmap_2d(&tmAux, a->resid, 4, a->N, a->M, a->ld_resid, 32, 32);
    if (rc) return rc;
  }
  if (kTmaEpi<EPI, BLOCK_N / (EW / 4)>) {
    if (EPI == EPI_DGELU) {   // [32 rows][128 B] boxes, 128-byte swizzle
      rc = vitk_make_tmap_2d(&tmOut, a->out, 2, a->N, a->M, a->ld_out, 64, 32);
      if (rc) return rc;
      rc = vitk_make_tmap_2d(&tmAux, a->aux, 2, a->N, a->M, a->ld_aux, 64, 32);
    } else {                  // [32 rows][64 B] boxes, 64-byte swizzle
      rc = vitk_make_tmap_2d_sw64(&tmOut, a->out, 2, a->N, a->M, a->ld_out, 32, 32);
      if (rc) return rc;
      rc = vitk_make_tmap_2d_sw64(&tmAux, a->aux, 2, a->N, a->M, a->ld_aux, 32, 32);
    }
    if (rc) return rc;
  }

  const int sms = vitk_num_sms();
  const int slots = CTA2 ? sms / 2 : sms;
  GemmParams p;
  p.M = a->M; p.N = a->N; p.K = a->K;
  p.num_m_tiles = (a->M + TILE_M - 1) / TILE_M;
  p.num_n_tiles = (a->N + BLOCK_N - 1) / BLOCK_N;
  p.num_k_blocks = (a->K + BLOCK_K - 1) / BLOCK_K;
  p.splits = 1;
  if (EPI == EPI_ATOMIC) {
    p.splits = a->splits > 0 ? a->splits : pick_splits(p.num_m_tiles * p.num_n_tiles, p.num_k_blocks, slots, BLOCK_N);
    if (p.splits > p.num_k_blocks) p.splits = p.num_k_blocks;
  }
  p.out = a->out; p.ld_out = a->ld_out;
  p.aux = a->aux; p.ld_aux = a->ld_aux;
  p.bias = a->bias;
  p.resid = a->resid; p.ld_resid = a->ld_resid;
  p.rowscale = a->rowscale; p.rows_per_group = a->rows_per_group > 0 ? a->rows_per_group : 1;
  p.colscale = a->colscale;
  p.pos = a->pos; p.tokens_per_img = a->tokens_per_img > 0 ? a->tokens_per_img : 1;
  p.prefix = a->prefix;
  p.ragged = (EPI == EPI_F32 && (a->N % 8 != 0 || a->ld_out % 4 != 0)) ? 1 : 0;
  p.colsum_out = (EPI == EPI_ATOMIC && A_MN) ? a->colsum_out : nullptr;
  p.mask = a->mask; p.ld_mask = a->ld_mask; p.mask_scale = a->mask_scale;
  p.a_image = (a->a_image && !A_MN) ? 1 : 0;
  p.b_image = (a->b_image && B_MN) ? 1 : 0;
  p.img_c = a->img_c; p.img_ps = a->img_patch > 0 ? a->img_patch : 16; p.img_gwp = a->img_gwp > 0 ? a->img_gwp : 16;
  p.img_gh = a->img_h / p.img_ps; p.img_gw = a->img_w / p.img_ps;
  if (p.img_gh < 1) p.img_gh = 1;

  auto kern = gemm_kernel<BLOCK_N, A_MN, B_MN, EPI, EW, CTA2>;
  static bool attr_set = false;  // per-instantiation
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM_BYTES);
    if (e != cudaSuccess)
      return vitk_set_error(VITK_ERR_CUDA, "gemm: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    attr_set = true;
  }
  const int units = p.num_m_tiles * p.num_n_tiles * p.splits;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)((units < slots ? units : slots) * (CTA2 ? 2 : 1)));
  cfg.blockDim = dim3(128 + EW * 32);
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CTA2 ? 2 : 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, tmA, tmB, tmOut, tmAux, p);
  if (e != cudaSuccess) return vitk_set_error(VITK_ERR_CUDA, "gemm: launch failed: %s", cudaGetErrorString(e));
  return vitk_check_launch("gemm");
}

template <int BLOCK_N, bool CTA2>
int dispatch2(const vitk_gemm_args* a, cudaStream_t stream) {
  const bool amn = a->a_mn_major != 0, bmn = a->b_mn_major != 0;
  constexpr bool PAIR192 = CTA2 && BLOCK_N == 192;   // built for the forward (K-major B) epilogues only
  if (a->epilogue == EPI_ATOMIC) {
    if constexpr (!PAIR192) {
      if (amn && bmn) return launch_gemm<BLOCK_N, true, true, EPI_ATOMIC, CTA2>(a, stream);
      if (!amn && !bmn) return launch_gemm<BLOCK_N, false, false, EPI_ATOMIC, CTA2>(a, stream);
    }
    return vitk_set_error(VITK_ERR_UNSUPPORTED, "gemm: EPI_ATOMIC needs both operands in the same major");
  }
  if (!amn && !bmn) {
    switch (a->epilogue) {
      case EPI_BF16:
        if constexpr (BLOCK_N % 128 == 0) return launch_gemm<BLOCK_N, false, false, EPI_BF16_TMA, CTA2>(a, stream);
        else return launch_gemm<BLOCK_N, false, false, EPI_BF16, CTA2>(a, stream);
      case EPI_GELU:  return launch_gemm<BLOCK_N, false, false, EPI_GELU, CTA2>(a, stream);
      case EPI_RESID:
        // TMA needs 16-byte aligned bases and row pitches: the entry checks require them of out, resid, ld_out, ld_resid and N
        if constexpr (CTA2 || BLOCK_N < 256) {
          if (a->K <= kResidTmaMaxK && a->mask == nullptr)   // the dropout mask lives in the staged-panel epilogue
            return launch_gemm<BLOCK_N, false, false, EPI_RESID_TMA, CTA2>(a, stream);
        }
        return launch_gemm<BLOCK_N, false, false, EPI_RESID, CTA2>(a, stream);
      case EPI_F32:   return launch_gemm<BLOCK_N, false, false, EPI_F32, CTA2>(a, stream);
      case EPI_PATCH: return launch_gemm<BLOCK_N, false, false, EPI_PATCH, CTA2>(a, stream);
    }
  } else if (!amn && bmn) {
    if constexpr (!PAIR192) {
    switch (a->epilogue) {
      case EPI_BF16:
        if constexpr (BLOCK_N % 128 == 0) return launch_gemm<BLOCK_N, false, true, EPI_BF16_TMA, CTA2>(a, stream);
        else return launch_gemm<BLOCK_N, false, true, EPI_BF16, CTA2>(a, stream);
      case EPI_DGELU: return launch_gemm<BLOCK_N, false, true, EPI_DGELU, CTA2>(a, stream);
      case EPI_F32:   return launch_gemm<BLOCK_N, false, true, EPI_F32, CTA2>(a, stream);
    }
    }
  }
  return vitk_set_error(VITK_ERR_UNSUPPORTED, "gemm: unsupported layout/epilogue combination (a_mn=%d b_mn=%d epi=%d)",
                        (int)amn, (int)bmn, a->epilogue);
}

template <int BLOCK_N>
int dispatch(const vitk_gemm_args* a, cudaStream_t stream) {
  // CTA pairs pay off once there are enough 256-row tiles to go round; tiny problems keep 128-row tiles
  if constexpr (BLOCK_N != 192) {
    if (a->M >= 256) return dispatch2<BLOCK_N, true>(a, stream);
  } else {
    // 256 x 192 pair tiles exist for the forward layouts (both operands K-major, not split-K)
    if (a->M >= 256 && !a->a_mn_major && !a->b_mn_major && a->epilogue != EPI_ATOMIC)
      return dispatch2<BLOCK_N, true>(a, stream);
  }
  return dispatch2<BLOCK_N, false>(a, stream);
}

}  // namespace

extern "C" int vitk_gemm_bf16(const vitk_gemm_args* a, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  VITK_REQUIRE(a != nullptr, VITK_ERR_SHAPE, "gemm: null args");
  VITK_REQUIRE(a->M > 0 && a->N > 0 && a->K > 0, VITK_ERR_SHAPE, "gemm: empty problem M=%d N=%d K=%d", a->M, a->N, a->K);
  VITK_REQUIRE(a->N % 8 == 0 || a->epilogue == EPI_F32, VITK_ERR_SHAPE,
               "gemm: N=%d must be a multiple of 8 (only the fp32 epilogue handles ragged N)", a->N);
  VITK_REQUIRE(a->lda % 8 == 0 && a->ldb % 8 == 0, VITK_ERR_ALIGN, "gemm: lda/ldb must be multiples of 8 elements (16 B)");
  VITK_REQUIRE((reinterpret_cast<uintptr_t>(a->A) & 15) == 0 && (reinterpret_cast<uintptr_t>(a->B) & 15) == 0,
               VITK_ERR_ALIGN, "gemm: A/B must be 16-byte aligned");
  VITK_REQUIRE(a->out != nullptr && (reinterpret_cast<uintptr_t>(a->out) & 15) == 0, VITK_ERR_ALIGN, "gemm: out must be 16-byte aligned");
  VITK_REQUIRE(a->ld_out % 8 == 0 || a->epilogue == EPI_F32, VITK_ERR_ALIGN, "gemm: ld_out must be a multiple of 8");
  // The epilogues read bias, colscale, pos and resid with float4 loads (or TMA) and aux with 16-byte loads (or TMA).
  // Checked whatever the epilogue, so that no layout or epilogue choice below depends on a side operand's address.
  const struct { const void* ptr; const char* name; } side[] = {
      {a->bias, "bias"}, {a->colscale, "colscale"}, {a->pos, "pos"}, {a->resid, "resid"}, {a->aux, "aux"}};
  for (const auto& s : side)
    VITK_REQUIRE((reinterpret_cast<uintptr_t>(s.ptr) & 15) == 0, VITK_ERR_ALIGN, "gemm: %s must be 16-byte aligned", s.name);
  if (a->epilogue == EPI_GELU || a->epilogue == EPI_DGELU)
    VITK_REQUIRE(a->aux != nullptr && a->ld_aux % 8 == 0, VITK_ERR_ALIGN, "gemm: aux pointer/ld required for GELU epilogues");
  if (a->epilogue == EPI_RESID)
    VITK_REQUIRE(a->resid != nullptr && a->ld_resid % 4 == 0, VITK_ERR_ALIGN, "gemm: resid pointer/ld required");
  if (a->epilogue == EPI_PATCH)
    VITK_REQUIRE(a->pos != nullptr && a->tokens_per_img > 0, VITK_ERR_SHAPE, "gemm: pos/tokens_per_img required");

  if (a->a_image || a->b_image) {
    const int ps = a->img_patch, gwp = a->img_gwp;
    VITK_REQUIRE(ps == 16, VITK_ERR_UNSUPPORTED, "gemm: image operand: patch %d (built for 16)", ps);
    VITK_REQUIRE(a->img_c > 0 && a->img_h > 0 && a->img_w > 0 && a->img_h % ps == 0 && a->img_w % ps == 0 && a->img_w % 8 == 0,
                 VITK_ERR_SHAPE, "gemm: image operand: bad geometry C=%d H=%d W=%d patch=%d", a->img_c, a->img_h, a->img_w, ps);
    VITK_REQUIRE(gwp > 0 && gwp % 8 == 0 && gwp >= a->img_w / ps && gwp < a->img_w / ps + 8, VITK_ERR_SHAPE,
                 "gemm: image operand: img_gwp=%d must be the patch-grid width %d rounded up to a multiple of 8", gwp, a->img_w / ps);
    VITK_REQUIRE(!(a->a_image && a->b_image), VITK_ERR_UNSUPPORTED, "gemm: only one operand can be an image");
    if (a->a_image)
      VITK_REQUIRE(!a->a_mn_major && a->K == a->img_c * ps * ps && a->M % gwp == 0, VITK_ERR_SHAPE,
                   "gemm: a_image needs K-major A, K = C * patch^2 and M a multiple of img_gwp");
    if (a->b_image)
      VITK_REQUIRE(a->b_mn_major && a->N == a->img_c * ps * ps && a->K % gwp == 0, VITK_ERR_SHAPE,
                   "gemm: b_image needs MN-major B, N = C * patch^2 and K a multiple of img_gwp");
  }

  if (a->mask != nullptr) {
    VITK_REQUIRE(a->epilogue == EPI_GELU || a->epilogue == EPI_RESID, VITK_ERR_UNSUPPORTED,
                 "gemm: a dropout mask goes with the GELU and RESID epilogues (epilogue=%d)", a->epilogue);
    VITK_REQUIRE(a->ld_mask % 4 == 0 && a->ld_mask >= a->N && (reinterpret_cast<uintptr_t>(a->mask) & 3) == 0, VITK_ERR_ALIGN,
                 "gemm: mask must be 4-byte aligned with ld_mask a multiple of 4 and >= N");
    VITK_REQUIRE(a->mask_scale > 0.f, VITK_ERR_SHAPE, "gemm: mask_scale = 1 / (1 - p) must be positive");
  }
  int bn = a->block_n;
  if (bn == 0) {
    // 256-wide pair tiles are the most efficient ones, even with a partly empty last column of tiles, as long as that
    // costs <= 15 % extra MMA work (ViT-S qkv, N = 1152 = 4.5 x 256: 48.6 us against 57.0 us with 6 x 192 pair tiles,
    // profiles/r02_gemm_tile_width.txt); beyond that an exact 192 / 128 split wins (N = 384: 41-42 us against 48.3 us)
    const int n256 = (a->N + 255) / 256 * 256;
    if (a->N % 256 == 0 || (a->N > 512 && n256 * 100 <= a->N * 115)) bn = 256;
    else if (a->N % 192 == 0) bn = 192;
    else if (a->N % 128 == 0) bn = 128;
    else bn = (a->N > 192) ? 256 : (a->N > 128 ? 192 : 128);
  }
  // GELU with a dropout mask: 256-wide tiles take the TMA-staged GELU epilogue, which has no mask path
  if (a->mask != nullptr && a->epilogue == EPI_GELU && bn == 256) bn = 192;
  switch (bn) {
    case 256: return dispatch<256>(a, stream);
    case 192: return dispatch<192>(a, stream);
    case 128: return dispatch<128>(a, stream);
  }
  return vitk_set_error(VITK_ERR_UNSUPPORTED, "gemm: block_n=%d not in {128,192,256}", bn);
}
