// vitk_attn.cu — multi-head attention forward / backward on tcgen05 tensor cores (sm_100a).
//
// Replaces F.scaled_dot_product_attention(q, k, v) (dropout 0, no mask, scale = hd^-0.5) at the
// timm Attention call site constructed by /root/reference/models/vision_transformer.py:149-159
// (witness of the same math in-tree: /root/reference/models/eva.py:146-194).
//
// Layout: qkv bf16 [B, N, 3, H, 64] exactly as the qkv Linear writes it; out / dout bf16
// [B, N, H*64]; lse fp32 [B, H, N].  Tiles are staged by TMA straight out of those tensors (3-D
// tensor maps, rows past N are zero-filled by the TMA unit) into 128-byte-swizzled smem, S / dP /
// O / dK / dV / dQ accumulate in TMEM, and thread t of the CTA owns row t of every 128-row tile
// (TMEM lane == row), so the softmax needs no cross-thread reduction at all.
//
// The same smem bytes serve as a K-major operand ([rows][64 contiguous] = rows x K) and as an
// MN-major operand (K rows x 64 contiguous MN) — only the UMMA descriptor differs — which is how
// P / dS feed P*V, P^T*dO, dS^T*Q and dS*K without any transposes.
#include "vitk_common.cuh"
#include "vitk_internal.h"

namespace {
using namespace vitk;

constexpr int HD = 64;
constexpr int TILE = 128;
constexpr uint32_t TILE_BYTES = TILE * HD * 2;  // 16 KB: [128 rows][128 B]
constexpr int ATTN_MAX_N = 33 * TILE;           // N <= 4224: 1024 px at patch 16 (N = 4097) with room for prefix tokens
constexpr float LOG2E = 1.4426950408889634f;

__device__ __forceinline__ uint32_t roundup16(int v) { return (uint32_t)((v + 15) & ~15); }

// Phase timeline for tuning (vitk_debug_set_trace): attn_fwd4 / attn_fwd6 / attn_bwd4 stamp clock64() into a device buffer.
long long* g_trace_buf = nullptr;

// Store 8 consecutive bf16 (one 16-byte unit `u8` of row `r`) into a [chunk][128 rows][128 B] swizzled tile.
__device__ __forceinline__ void st_swz(uint8_t* tile, int r, int col8, uint4 val) {
  const int chunk = col8 >> 3;  // 64-column chunk
  const int u = col8 & 7;       // 16-byte unit inside the 128-byte row
  uint8_t* p = tile + chunk * TILE_BYTES + r * 128 + ((u ^ (r & 7)) << 4);
  *reinterpret_cast<uint4*>(p) = val;
}

// Compiler-level scheduling fence over 32 registers: everything that produces r[] is emitted before, everything that
// consumes it after (no instruction is generated).
__device__ __forceinline__ void pin32(uint32_t (&r)[32]) {
  asm volatile("" : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
               "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]),
               "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]),
               "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31]));
}

// Wide heads (64 < head_dim <= 80, my_vit_xs: 72): every operand is [64-column tile][tail tile] (2 x 16 KB, the tail
// holding columns 64 .. 127 of the head with everything >= head_dim zero-filled by TMA).  As a K-major operand the tail
// adds one k-step (columns 64 .. 79) to Q K^T; as an MN-major operand it is the second 64-wide chunk of V (dO, Q, K), of
// which an MMA with N = 80 reads the first 16 columns.  Accumulators over the head dimension have 80 columns.
constexpr int HDW_MAX = 80;

// one operand box (+ its tail for wide heads) of head slot `slot`, rows row0 .., image b
template <bool WIDE>
__device__ __forceinline__ void load_head_tiles(uint8_t* dst, const CUtensorMap* tm, uint64_t* bar, int slot, int row0, int b) {
  tma_load_head(dst, tm, bar, slot, row0, b);
  if (WIDE) tma_load_head_col(dst + TILE_BYTES, tm, bar, HD, slot, row0, b);
}

// one accumulator row (columns 0..31 in a, 32..63 in b) -> bf16; only the first `hd` (multiple of 8) columns exist
__device__ __forceinline__ void store_row_bf16_64(__nv_bfloat16* dst, const uint32_t (&a)[32], const uint32_t (&b)[32], int hd) {
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    if (g * 8 >= hd) break;
    uint4 u;
    u.x = pack_bf16x2(__uint_as_float(a[g * 8 + 0]), __uint_as_float(a[g * 8 + 1]));
    u.y = pack_bf16x2(__uint_as_float(a[g * 8 + 2]), __uint_as_float(a[g * 8 + 3]));
    u.z = pack_bf16x2(__uint_as_float(a[g * 8 + 4]), __uint_as_float(a[g * 8 + 5]));
    u.w = pack_bf16x2(__uint_as_float(a[g * 8 + 6]), __uint_as_float(a[g * 8 + 7]));
    *reinterpret_cast<uint4*>(dst + g * 8) = u;
  }
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    if (32 + g * 8 >= hd) break;
    uint4 u;
    u.x = pack_bf16x2(__uint_as_float(b[g * 8 + 0]), __uint_as_float(b[g * 8 + 1]));
    u.y = pack_bf16x2(__uint_as_float(b[g * 8 + 2]), __uint_as_float(b[g * 8 + 3]));
    u.z = pack_bf16x2(__uint_as_float(b[g * 8 + 4]), __uint_as_float(b[g * 8 + 5]));
    u.w = pack_bf16x2(__uint_as_float(b[g * 8 + 6]), __uint_as_float(b[g * 8 + 7]));
    *reinterpret_cast<uint4*>(dst + 32 + g * 8) = u;
  }
}

// ================================================================================================
// Forward, warp-specialised persistent kernel for 128 < N <= 256 (224-px ViT / DeiT: N = 197 / 198).
//
// The softmax, not the tensor core, bounds attention at head_dim 64 (one MUFU.EX2 per 256 MMA flops; measured
// 15.6 ex2/clk/SM, tools/ubench_tmem.cu), so the kernel is organised to keep the MUFU pipe fed:
//   * one CTA per SM loops over (b, h) items; warp 18 prefetches Q/K/V of the next item by TMA (2 smem stages);
//   * group g (warps 8g..8g+7) owns q tile g and TMEM slot g (256 columns).  Two threads share a score row
//     (TMEM lane = row, halves split the kv columns at a 16-column boundary), so each scheduler always has
//     two softmax warps per group;  warp 16+g issues that group's MMAs, so the two groups run out of phase and
//     one group's exps overlap the other's MMA / TMEM round trips;
//   * the whole score row (<= 256 columns) is in TMEM, so the softmax is two passes over it (max, then exp) with no
//     rescaling; P is written back over S in TMEM as packed bf16 and feeds O = P V as the TMEM A operand
//     (no shared-memory round trip, no proxy fence).
// Slot layout (columns): S [0, n_eff) | P_lo [0, 8 k0) | P_hi [16 k0, 16 k0 + 8 k1) | O [192, 256)
// smem: 2 stages x (Q0 Q1 K0 K1 V0 V1) | max / sum exchange | barriers
// ================================================================================================
struct Fwd3Smem {
  static constexpr uint32_t STAGE = 6 * TILE_BYTES;
  static constexpr uint32_t XCH_OFF = 2 * STAGE;                      // float [2 groups][max, sum][2 halves][128]
  static constexpr uint32_t BAR_OFF = XCH_OFF + 2 * 2 * 2 * 128 * 4;
  static constexpr uint32_t BYTES = BAR_OFF + 256;
};

// ================================================================================================
// attn_fwd4: the kernel built on the structure above with ONE thread per score row.
// 11 warps: group g = warps 4g..4g+3 (thread = score row of q tile g), warp 8 + g issues group g's MMAs, warp 10 is
// the TMA producer.  With 168 registers per thread the score row is processed in 32-column chunks that are
// double-buffered in registers and fully unrolled (the structure of the backward's P phase, which sustains ~10 cycles
// per exp per warp; a 16-column rolled loop with two threads per row needed ~29), there is no max / sum
// exchange and no named barrier, and P is one contiguous run of packed columns [0, n_eff / 2) written in place
// behind the read pointer.
// ================================================================================================
constexpr int FWD4_THREADS = 11 * 32;

__global__ void __launch_bounds__(FWD4_THREADS, 1)
attn_fwd4_kernel(const __grid_constant__ CUtensorMap tm_qkv, const __grid_constant__ CUtensorMap tm_out, float* __restrict__ lse,
                 int B, int N, int H, float scale, long long* trace) {
  using L = Fwd3Smem;
#define FWD4_STAMP(base, ev) do { if (trace != nullptr && blockIdx.x == 0 && lane == 0 && (n == 2 || n == 3)) trace[(base) + 8 * (n - 2) + (ev)] = clock64(); } while (0)
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* stage_full = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);  // [2] TMA -> MMA warps
  uint64_t* stage_empty = stage_full + 2;                                  // [2] MMA warps -> TMA
  uint64_t* s_full = stage_empty + 2;                                      // [g] MMA -> group: S ready
  uint64_t* p_full = s_full + 2;                                           // [g] group -> MMA: P written
  uint64_t* o_full = p_full + 2;                                           // [g] MMA -> group: O ready
  uint64_t* slot_free = o_full + 2;                                        // [g] group -> MMA: O read out
  uint64_t* o_staged = slot_free + 2;                                      // [g] group -> MMA: bf16 O tile in smem
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_staged + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int items = B * H;
  const uint32_t n_eff = roundup16(N);
  const int KS = (int)n_eff / 16;           // k-steps of P V
  const int nch = ((int)n_eff + 31) / 32;   // 32-column chunks of the score row (the last one may be half)

  if ((smem_u32(smem) & 1023u) != 0) __trap();
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&stage_full[i], 1);
      mbar_init(&stage_empty[i], 4);   // per MMA warp: Q/K/V reads retired + its group's O staging tile stored
      mbar_init(&s_full[i], 1);
      mbar_init(&p_full[i], 4);        // one arrival per softmax warp
      mbar_init(&o_full[i], 1);
      mbar_init(&slot_free[i], 4);
      mbar_init(&o_staged[i], 4);
    }
    fence_mbar_init();
  }
  if (warp == 10) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 10) {
    // ------------------------------ TMA producer ------------------------------
    if (lane == 0) {
      tma_prefetch_desc(&tm_qkv);
      int n = 0;
      for (int it = blockIdx.x; it < items; it += gridDim.x, ++n) {
        const int st = n & 1;
        const int h = it % H, b = it / H;
        mbar_wait(&stage_empty[st], ((n >> 1) & 1) ^ 1);
        uint8_t* base = smem + st * L::STAGE;
        mbar_arrive_expect_tx(&stage_full[st], L::STAGE);
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          tma_load_head(base + t * TILE_BYTES, &tm_qkv, &stage_full[st], h, t * TILE, b);
          tma_load_head(base + (2 + t) * TILE_BYTES, &tm_qkv, &stage_full[st], H + h, t * TILE, b);
          tma_load_head(base + (4 + t) * TILE_BYTES, &tm_qkv, &stage_full[st], 2 * H + h, t * TILE, b);
        }
      }
    }
  } else if (warp >= 8) {
    // ------------------------------ MMA issuer of group g (uniform control flow, one elected lane issues) ------------------------------
    const int g = warp - 8;
    const uint32_t idesc_s = umma_idesc(TILE, n_eff, 1, false, false);
    const uint32_t idesc_o = umma_idesc(TILE, HD, 1, false, true);  // A = P (TMEM, K-major), B = V MN-major
    const uint32_t slot = tmem_base + g * 256;
    auto store_o = [&](int m, int item) {
      const int st = m & 1;
      mbar_wait(&o_staged[g], m & 1);
      if (elect_one()) {
        tma_store_head(&tm_out, smem + st * L::STAGE + g * TILE_BYTES, item % H, g * TILE, item / H);  // rows >= N clipped
        tma_store_commit_and_wait_read();
        mbar_arrive(&stage_empty[st]);
      }
      __syncwarp();
    };
    int n = 0;
    for (int it = blockIdx.x; it < items; it += gridDim.x, ++n) {
      const int st = n & 1;
      const uint32_t sbase = smem_u32(smem + st * L::STAGE);
      const uint32_t sQ = sbase + g * TILE_BYTES, sK = sbase + 2 * TILE_BYTES, sV = sbase + 4 * TILE_BYTES;
      mbar_wait(&stage_full[st], (n >> 1) & 1);
      FWD4_STAMP(32 + 16 * g, 0);
      if (n > 0) mbar_wait(&slot_free[g], (n - 1) & 1);
      else if (g == 1) mbar_wait(&p_full[0], 0);   // group 1 starts half an item late
      FWD4_STAMP(32 + 16 * g, 1);
      tc_fence_after();
      const uint64_t qdesc = umma_desc_kmajor(sQ), kdesc = umma_desc_kmajor(sK);
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < HD / 16; ++k) umma_bf16_ss(slot, qdesc + (uint64_t)(k * 2), kdesc + (uint64_t)(k * 2), idesc_s, k > 0);
        umma_commit(&s_full[g]);
      }
      __syncwarp();
      FWD4_STAMP(32 + 16 * g, 2);
      if (n > 0) store_o(n - 1, it - (int)gridDim.x);   // nothing else to do until this group's P arrives
      mbar_wait(&p_full[g], n & 1);
      FWD4_STAMP(32 + 16 * g, 3);
      tc_fence_after();
      const uint64_t vdesc = umma_desc_mnmajor(sV, TILE_BYTES);
      if (elect_one()) {
        for (int ks = 0; ks < KS; ++ks) umma_bf16_ts(slot + 192, slot + 8 * ks, vdesc + (uint64_t)(ks * 128), idesc_o, ks > 0);
        umma_commit(&o_full[g]);
        umma_commit(&stage_empty[st]);  // this group's reads of Q_g / K / V have retired
      }
      __syncwarp();
      FWD4_STAMP(32 + 16 * g, 4);
    }
    if (n > 0) {
      store_o(n - 1, blockIdx.x + (n - 1) * (int)gridDim.x);
      if (elect_one()) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // smem must outlive the store
      __syncwarp();
    }
  } else {
    // ------------------------------ softmax group g: 128 threads, thread = score row ------------------------------
    const int g = warp >> 2, quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const uint32_t slot = tmem_base + g * 256 + (static_cast<uint32_t>(quarter * 32) << 16);
    const int qn = g == 0 ? min(TILE, N) : N - TILE;   // valid rows of this q tile
    const bool active = quarter * 32 < qn;             // warp-uniform: some row of this warp is real
    const float c2 = scale * LOG2E;
    const int q = g * TILE + r;
    int n = 0;
    for (int it = blockIdx.x; it < items; it += gridDim.x, ++n) {
      mbar_wait(&s_full[g], n & 1);
      tc_fence_after();
      if (quarter == 0) FWD4_STAMP(16 * g, 0);
      uint32_t ra[32], rb[32];
      float mx = 0.f, l = 1.f;
      if (active) {
        // ---- pass 1: row maximum ----
        float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
        auto mx_chunk = [&](const uint32_t (&v)[32], int c) {
          if (c * 32 + 32 <= N) {
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              m0 = fmaxf(m0, __uint_as_float(v[i]));
              m1 = fmaxf(m1, __uint_as_float(v[i + 1]));
              m2 = fmaxf(m2, __uint_as_float(v[i + 2]));
              m3 = fmaxf(m3, __uint_as_float(v[i + 3]));
            }
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (c * 32 + i < N) m0 = fmaxf(m0, __uint_as_float(v[i]));
          }
        };
        // (four chunks in flight per round trip do not help: with the other group's exps queued in the same MIO
        // pipe a tcgen05.ld takes ~700 cycles here against ~40 on an idle SM, and the extra registers cost more)
        tmem_ld_32x32(slot, ra);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < 8; c += 2) {
          if (c < nch) {
            if (c + 1 < nch) tmem_ld_32x32(slot + (c + 1) * 32, rb);
            mx_chunk(ra, c);
            if (c + 1 < nch) {
              tmem_ld_wait();
              if (c + 2 < nch) tmem_ld_32x32(slot + (c + 2) * 32, ra);
              mx_chunk(rb, c + 1);
              if (c + 2 < nch) tmem_ld_wait();
            }
          }
        }
        mx = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
        if (quarter == 0) FWD4_STAMP(16 * g, 1);

        // ---- pass 2: P = exp2(S * c2 - mx * c2) -> packed bf16, written back over S behind the read pointer ----
        const float mc = mx * c2;
        float s0 = 0.f, s1 = 0.f;
        auto p_chunk = [&](const uint32_t (&v)[32], int c) {
          uint32_t pk[16];
          if (c * 32 + 32 <= N) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float e0 = ex2_approx(fmaf(__uint_as_float(v[2 * i]), c2, -mc));
              const float e1 = ex2_approx(fmaf(__uint_as_float(v[2 * i + 1]), c2, -mc));
              s0 += e0;
              s1 += e1;
              pk[i] = pack_bf16x2(e0, e1);
            }
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              float e0 = ex2_approx(fmaf(__uint_as_float(v[2 * i]), c2, -mc));
              float e1 = ex2_approx(fmaf(__uint_as_float(v[2 * i + 1]), c2, -mc));
              e0 = (c * 32 + 2 * i < N) ? e0 : 0.f;
              e1 = (c * 32 + 2 * i + 1 < N) ? e1 : 0.f;
              s0 += e0;
              s1 += e1;
              pk[i] = pack_bf16x2(e0, e1);
            }
          }
          tmem_st_32x16(slot + c * 16, pk);
        };
        tmem_ld_32x32(slot, ra);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < 8; c += 2) {
          if (c < nch) {
            if (c + 1 < nch) tmem_ld_32x32(slot + (c + 1) * 32, rb);
            p_chunk(ra, c);
            if (c + 1 < nch) {
              tmem_ld_wait();
              if (c + 2 < nch) tmem_ld_32x32(slot + (c + 2) * 32, ra);
              p_chunk(rb, c + 1);
              if (c + 2 < nch) tmem_ld_wait();
            }
          }
        }
        tmem_st_wait();
        l = s0 + s1;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[g]);
      if (quarter == 0) FWD4_STAMP(16 * g, 3);

      // ---- O = P V ----
      mbar_wait(&o_full[g], n & 1);
      tc_fence_after();
      if (quarter == 0) FWD4_STAMP(16 * g, 5);
      if (active) {
        tmem_ld_32x32(slot + 192, ra);
        tmem_ld_32x32(slot + 224, rb);
        tmem_ld_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&slot_free[g]);
      if (quarter == 0) FWD4_STAMP(16 * g, 6);
      // normalised bf16 row -> the (dead) Q_g tile of this item's stage, 128-byte swizzled -> TMA store by the MMA warp
      const int st = n & 1;
      uint8_t* stg = smem + st * L::STAGE + g * TILE_BYTES;
      if (active) {
        const int h = it % H, b = it / H;
        const float inv = 1.0f / l;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const uint32_t(&o)[32] = u < 4 ? ra : rb;
          const int e = (u & 3) * 8;
          uint4 v4;
          v4.x = pack_bf16x2(__uint_as_float(o[e + 0]) * inv, __uint_as_float(o[e + 1]) * inv);
          v4.y = pack_bf16x2(__uint_as_float(o[e + 2]) * inv, __uint_as_float(o[e + 3]) * inv);
          v4.z = pack_bf16x2(__uint_as_float(o[e + 4]) * inv, __uint_as_float(o[e + 5]) * inv);
          v4.w = pack_bf16x2(__uint_as_float(o[e + 6]) * inv, __uint_as_float(o[e + 7]) * inv);
          st_swz(stg, r, u, v4);
        }
        if (q < N && lse) lse[((long long)b * H + h) * N + q] = mx * scale + __logf(l);
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&o_staged[g]);
      if (quarter == 0) FWD4_STAMP(16 * g, 7);
    }
  }
#undef FWD4_STAMP

  tc_fence_before();
  __syncthreads();
  if (warp == 10) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

int launch_fwd4(const CUtensorMap& tm, const CUtensorMap& tm_out, float* lse, int B, int N, int H, float scale, cudaStream_t s) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(attn_fwd4_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Fwd3Smem::BYTES);
    if (e != cudaSuccess) return vitk_set_error(VITK_ERR_CUDA, "attn_fwd4: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    attr_set = true;
  }
  const int items = B * H;
  const int grid = items < vitk_num_sms() ? items : vitk_num_sms();
  attn_fwd4_kernel<<<grid, FWD4_THREADS, Fwd3Smem::BYTES, s>>>(tm, tm_out, lse, B, N, H, scale, g_trace_buf);
  return vitk_check_launch("attn_fwd4");
}

// ================================================================================================
// attn_fwd6: flash-style kv-loop forward for 256 < N <= 640 (ViT-L/16 at 384 px: N = 577), the roles of attn_fwd4 with the
// score MMA taken OFF the softmax's critical path.
// Work item = (b, h, round): in round r group g owns q tile 2r + g (one thread per score row); both groups walk the same
// K_j / V_j tiles, which stream through a 4-stage TMA ring shared by the two groups.  Per kv tile the 128 score columns of a
// row are read out of TMEM ONCE into registers (max and exp both work from there); P goes back to TMEM as packed bf16 and
// feeds O += P V_j as the TMEM A operand; O stays in TMEM across the kv loop and is rescaled in place (tcgen05.ld / st,
// only when some row of the warp raised its maximum).
// Its predecessor (attn_fwd5, removed) kept S and P in the SAME TMEM columns, so S_{j+1} = Q K_{j+1}^T could only be issued
// after P_j had been written, and both groups ended up in phase (timeline in profiles/r02_ncu_attn_fwd6.txt): ~2 700 cycles
// of two groups fighting for the MUFU pipe, then ~1 350 cycles in which both wait for the P V / S hop and nobody issues an
// exp.  Here P has its own columns:
//   TMEM per group (256 columns): S [0,128) fp32 | P [128,192) packed bf16 | O [192,256) fp32
// and the MMA warp issues S_{k+1} as soon as the softmax group has S_k in REGISTERS (s_read) — across kv tiles, q tiles
// and work items (Q is double-buffered), so the next score tile is always waiting in TMEM when a group finishes a step
// and the MUFU pipe never idles on an MMA round trip.  P V_k is issued when P_k is written; the group waits for it
// (pv_done) only before it touches P or O again, one whole max phase later.
// Work item = (b, h, round): group g owns q tile 2 round + g; when the number of q tiles is odd the last round's second
// tile does not exist: its group keeps the barrier protocol (and the shared K/V ring) going but issues no MMA and no exp.
// Every softmax warp executes every wait, also when none of its rows is real: a warp that ran ahead would deliver its
// arrival for step k + 1 into phase k of a barrier.
// smem: Q[g][2] (also the O staging tiles) | 4 x (K_j V_j) | barriers = 192 KB
// ================================================================================================
constexpr int FWD6_THREADS = 12 * 32;   // softmax g0 | softmax g1 | MMA g0, MMA g1, TMA, idle

struct Fwd6Smem {
  static constexpr uint32_t Q_OFF = 0;                       // [g][buf]
  static constexpr uint32_t KV_OFF = 4 * TILE_BYTES;
  static constexpr int STAGES = 4;
  static constexpr uint32_t BAR_OFF = KV_OFF + STAGES * 2 * TILE_BYTES;
  static constexpr uint32_t BYTES = BAR_OFF + 256;
};

__global__ void __launch_bounds__(FWD6_THREADS, 1)
attn_fwd6_kernel(const __grid_constant__ CUtensorMap tm_qkv, const __grid_constant__ CUtensorMap tm_out, float* __restrict__ lse,
                 int B, int N, int H, float scale, long long* trace) {
  using L = Fwd6Smem;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* q_full = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);  // [2 g + buf] TMA -> MMA g: Q tile landed
  uint64_t* q_empty = q_full + 4;                                      // [2 g + buf] MMA g -> TMA: O tile stored, buffer reusable
  uint64_t* kv_full = q_empty + 4;                                     // [4] TMA -> MMA warps
  uint64_t* kv_empty = kv_full + L::STAGES;                            // [4] both MMA warps -> TMA
  uint64_t* s_full = kv_empty + L::STAGES;                             // [g] MMA -> group: S_k in TMEM
  uint64_t* s_read = s_full + 2;                                       // [g] group -> MMA: S_k in registers
  uint64_t* p_full = s_read + 2;                                       // [g] group -> MMA: P_k written, O rescaled
  uint64_t* pv_done = p_full + 2;                                      // [g] MMA -> group: P V_k retired
  uint64_t* o_free = pv_done + 2;                                      // [g] group -> MMA: O read out
  uint64_t* o_staged = o_free + 2;                                     // [g] group -> MMA: bf16 O tile in smem
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_staged + 2);
  volatile uint32_t* half_step = tmem_slot + 1;   // set once: group 0 is half way through its first step

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int QT = (N + TILE - 1) / TILE;     // q tiles == kv tiles
  const int R = (QT + 1) / 2;               // rounds per (b, h)
  const int items = B * H * R;

  if ((smem_u32(smem) & 1023u) != 0) __trap();
  if (threadIdx.x == 0) {
    for (int i = 0; i < 4; ++i) {
      mbar_init(&q_full[i], 1);
      mbar_init(&q_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&s_read[i], 4);
      mbar_init(&p_full[i], 4);
      mbar_init(&pv_done[i], 1);
      mbar_init(&o_free[i], 4);
      mbar_init(&o_staged[i], 4);
    }
    for (int i = 0; i < L::STAGES; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_empty[i], 2);
    }
    *half_step = 0;
    fence_mbar_init();
  }
  if (warp == 10) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp >= 8) {
    // 168 registers per thread at launch (384 threads): the control warpgroup gives back (168 - 56) x 128, exactly what the
    // two softmax warpgroups take ((224 - 168) x 256); an increase that the pool cannot cover never returns
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
  }
  if (warp == 11) {
    // idle: completes the control warpgroup (setmaxnreg is a warpgroup-wide instruction)
  } else if (warp == 10) {
    // ------------------------------ TMA producer ------------------------------
    if (lane == 0) {
      tma_prefetch_desc(&tm_qkv);
      int k = 0;
      for (int it = blockIdx.x, n = 0; it < items; it += gridDim.x, ++n) {
        const int r = it % R, bh = it / R, h = bh % H, b = bh / H;
        for (int g = 0; g < 2; ++g) {
          const int qt = 2 * r + g, qb = 2 * g + (n & 1);
          mbar_wait(&q_empty[qb], ((n >> 1) & 1) ^ 1);
          if (qt < QT) {
            mbar_arrive_expect_tx(&q_full[qb], TILE_BYTES);
            tma_load_head(smem + L::Q_OFF + qb * TILE_BYTES, &tm_qkv, &q_full[qb], h, qt * TILE, b);
          } else {
            mbar_arrive(&q_full[qb]);   // no such q tile: the group only keeps the protocol going
          }
        }
        for (int j = 0; j < QT; ++j, ++k) {
          const int st = k % L::STAGES;
          mbar_wait(&kv_empty[st], ((k / L::STAGES) & 1) ^ 1);
          uint8_t* base = smem + L::KV_OFF + st * 2 * TILE_BYTES;
          mbar_arrive_expect_tx(&kv_full[st], 2 * TILE_BYTES);
          tma_load_head(base, &tm_qkv, &kv_full[st], H + h, j * TILE, b);
          tma_load_head(base + TILE_BYTES, &tm_qkv, &kv_full[st], 2 * H + h, j * TILE, b);
        }
      }
    }
  } else if (warp >= 8) {
    // ------------------------------ MMA issuer of group g (uniform control flow, one elected lane issues) ------------------------------
    const int g = warp - 8;   // warps 8, 9
    const uint32_t slot = tmem_base + g * 256;
    const uint32_t idesc_o = umma_idesc(TILE, HD, 1, false, true);  // A = P (TMEM, K-major), B = V MN-major
    const uint32_t n_last = roundup16(N - (QT - 1) * TILE);
    const uint32_t idesc_full = umma_idesc(TILE, TILE, 1, false, false), idesc_last = umma_idesc(TILE, n_last, 1, false, false);
    const uint64_t qdesc0 = umma_desc_kmajor(smem_u32(smem + L::Q_OFF + 2 * g * TILE_BYTES));
    const uint64_t kdesc0 = umma_desc_kmajor(smem_u32(smem + L::KV_OFF));
    const uint64_t vdesc0 = umma_desc_mnmajor(smem_u32(smem + L::KV_OFF + TILE_BYTES), TILE_BYTES);
    constexpr uint64_t STAGE_STEP = (2 * TILE_BYTES) >> 4, QBUF_STEP = TILE_BYTES >> 4;
    const int n_items = (items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int total = n_items * QT;   // steps of this group; step k = (item n, kv tile j) uses ring tile k
    auto real_tile = [&](int n) { return 2 * ((int)(blockIdx.x + n * gridDim.x) % R) + g < QT; };
    auto issue_s = [&](int k, int n, int j, bool real) {   // S_k = Q_n K_j^T (operands already waited for)
      const uint64_t qd = qdesc0 + (uint64_t)(n & 1) * QBUF_STEP, kd = kdesc0 + (uint64_t)(k % L::STAGES) * STAGE_STEP;
      const uint32_t ids = (j == QT - 1) ? idesc_last : idesc_full;
      if (elect_one()) {
        if (real) {
#pragma unroll
          for (int c = 0; c < HD / 16; ++c) umma_bf16_ss(slot, qd + (uint64_t)(c * 2), kd + (uint64_t)(c * 2), ids, c > 0);
        }
        umma_commit(&s_full[g]);
      }
      __syncwarp();
    };
    int n = 0, j = 0;
    bool real = real_tile(0);
    mbar_wait(&q_full[2 * g], 0);
    mbar_wait(&kv_full[0], 0);
    // Two groups that start together stay together (they share the schedulers evenly) and then also END their steps
    // together: the hand-over between steps (P stores landing, the last S chunk arriving, the row maximum) issues no exp,
    // and in step the MUFU pipe idles through it twice per step.  Group 1 therefore starts half a step late; after that
    // neither group ever waits for the other, so the offset stays.
    if (g == 1)
      while (*half_step == 0) __nanosleep(64);
    tc_fence_after();
    issue_s(0, 0, 0, real);
    for (int k = 0; k < total; ++k) {
      const bool last = j == QT - 1;
      const int n1 = last ? n + 1 : n, j1 = last ? 0 : j + 1;
      bool real1 = real;
      if (k + 1 < total) {
        // S_{k+1} goes out as soon as the group holds S_k in registers: it is ready long before the group asks for it
        if (last) {
          real1 = real_tile(n1);
          mbar_wait(&q_full[2 * g + (n1 & 1)], (n1 >> 1) & 1);
        }
        mbar_wait(&kv_full[(k + 1) % L::STAGES], ((k + 1) / L::STAGES) & 1);
        mbar_wait(&s_read[g], k & 1);
        tc_fence_after();
        issue_s(k + 1, n1, j1, real1);
      }
      mbar_wait(&p_full[g], k & 1);
      if (j == 0 && n > 0) mbar_wait(&o_free[g], (n - 1) & 1);   // the previous q tile's O has been read out
      tc_fence_after();
      {
        const int st = k % L::STAGES;
        const int ksteps = (int)(last ? n_last : (uint32_t)TILE) / 16;
        const uint64_t vd = vdesc0 + (uint64_t)st * STAGE_STEP;
        if (elect_one()) {
          if (real)
            for (int ks = 0; ks < ksteps; ++ks)
              umma_bf16_ts(slot + 192, slot + 128 + 8 * ks, vd + (uint64_t)(ks * 128), idesc_o, (j > 0 || ks > 0));
          umma_commit(&kv_empty[st]);
          umma_commit(&pv_done[g]);
        }
        __syncwarp();
      }
      if (last) {
        // bf16 O tile (staged by the group in its dead Q buffer) -> global; then the buffer may be reloaded
        mbar_wait(&o_staged[g], n & 1);
        if (elect_one()) {
          if (real) {
            const int it = (int)(blockIdx.x + n * gridDim.x);
            const int r = it % R, bh = it / R;
            tma_store_head(&tm_out, smem + L::Q_OFF + (2 * g + (n & 1)) * TILE_BYTES, bh % H, (2 * r + g) * TILE, bh / H);  // rows >= N clipped
            tma_store_commit_and_wait_read();
          }
          mbar_arrive(&q_empty[2 * g + (n & 1)]);
        }
        __syncwarp();
      }
      n = n1;
      j = j1;
      real = real1;
    }
    if (elect_one()) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // smem must outlive the store
    __syncwarp();
  } else {
    // ------------------------------ softmax group g: 128 threads, thread = score row ------------------------------
    // Software pipeline over the steps of the group (across kv tiles, q tiles and work items): while the exps of step k
    // are issued chunk by chunk out of registers, the freed registers are refilled with S_{k+1} (tcgen05.ld is slow when
    // the MUFU queue is busy — ~700 cycles against ~40 — so a load phase of its own would leave the warp with nothing to
    // issue); at the end of the step the loads have landed, S_{k+1} is handed back to the MMA warp and its row maximum is
    // taken, so the next step starts with its exps.
    asm volatile("setmaxnreg.inc.sync.aligned.u32 224;");
    const int g = warp >> 2, quarter = warp & 3;
    const int rr = quarter * 32 + lane;
    const uint32_t slot = tmem_base + g * 256 + (static_cast<uint32_t>(quarter * 32) << 16);
    const float c2 = scale * LOG2E;
    const int n_items = (items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int total = n_items * QT;
    auto tile_rows = [&](int n) { return min(TILE, N - (2 * ((int)(blockIdx.x + n * gridDim.x) % R) + g) * TILE); };   // <= 0: no such q tile
    uint32_t sv[4][32];
    auto load_chunk = [&](int c) { tmem_ld_32x32(slot + c * 32, sv[c]); };
    auto row_max = [&](int kvn, int nch, float run) {
      float m0 = run, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        if (c < nch) {
          if (c * 32 + 32 <= kvn) {
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              m0 = fmaxf(m0, __uint_as_float(sv[c][i]));
              m1 = fmaxf(m1, __uint_as_float(sv[c][i + 1]));
              m2 = fmaxf(m2, __uint_as_float(sv[c][i + 2]));
              m3 = fmaxf(m3, __uint_as_float(sv[c][i + 3]));
            }
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (c * 32 + i < kvn) m0 = fmaxf(m0, __uint_as_float(sv[c][i]));
          }
        }
      }
      return fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
    };
    float m = -INFINITY, l = 0.f, m_new = -INFINITY, alpha = 0.f;
    bool active = quarter * 32 < tile_rows(0);   // warp-uniform
    {   // prologue: S_0 into registers, its maximum
      const int kvn = min(TILE, N), nch = ((int)roundup16(kvn) + 31) / 32;
      mbar_wait(&s_full[g], 0);
      tc_fence_after();
      if (active) {
#pragma unroll
        for (int c = 0; c < 4; ++c)
          if (c < nch) load_chunk(c);
        tmem_ld_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_read[g]);
      if (active) {
        m_new = row_max(kvn, nch, m);
        alpha = 0.f;
      }
    }
    int k = 0;
    for (int n = 0; n < n_items; ++n) {
      const int it = (int)(blockIdx.x + n * gridDim.x);
      const int r = it % R, bh = it / R, h = bh % H, b = bh / H;
      const int qt = 2 * r + g;
      const bool stamp = trace != nullptr && blockIdx.x == 0 && quarter == 0 && lane == 0 && n == 1;
      uint8_t* stg = smem + L::Q_OFF + (2 * g + (n & 1)) * TILE_BYTES;
      bool active1 = active;
      for (int j = 0; j < QT; ++j, ++k) {
        const int kvn = min(TILE, N - j * TILE);
        const int nch = ((int)roundup16(kvn) + 31) / 32;
        const bool has_next = k + 1 < total;
        const int j1 = (j == QT - 1) ? 0 : j + 1;
        const int kvn1 = min(TILE, N - j1 * TILE);
        const int nch1 = ((int)roundup16(kvn1) + 31) / 32;
        if (j == QT - 1 && has_next) active1 = quarter * 32 < tile_rows(n + 1);
        if (stamp && j < 5) trace[16 * g + 3 * j] = clock64();
        const float mc = m_new * c2;
        float s0 = 0.f, s1 = 0.f;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          if (active && c < nch) {
            uint32_t pk[16];
            if (c * 32 + 32 <= kvn) {
              // all 32 exps first, their consumers afterwards: a warp issues in order, and a sum scheduled two
              // instructions behind its MUFU.EX2 stalls the warp (and every exp behind it) for the MUFU latency
#pragma unroll
              for (int i = 0; i < 32; ++i) sv[c][i] = __float_as_uint(ex2_approx(fmaf(__uint_as_float(sv[c][i]), c2, -mc)));
              pin32(sv[c]);
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const float e0 = __uint_as_float(sv[c][2 * i]), e1 = __uint_as_float(sv[c][2 * i + 1]);
                s0 += e0;
                s1 += e1;
                pk[i] = pack_bf16x2(e0, e1);
              }
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                float e0 = ex2_approx(fmaf(__uint_as_float(sv[c][2 * i]), c2, -mc));
                float e1 = ex2_approx(fmaf(__uint_as_float(sv[c][2 * i + 1]), c2, -mc));
                e0 = (c * 32 + 2 * i < kvn) ? e0 : 0.f;
                e1 = (c * 32 + 2 * i + 1 < kvn) ? e1 : 0.f;
                s0 += e0;
                s1 += e1;
                pk[i] = pack_bf16x2(e0, e1);
              }
            }
            // P V_{k-1} reads P and accumulates into O: it has retired before either is touched (it was issued a whole
            // hand-over and 32 exps ago); every warp takes this wait (below for the warps without rows)
            if (c == 0 && j > 0) {
              mbar_wait(&pv_done[g], (k - 1) & 1);
              tc_fence_after();
            }
            tmem_st_32x16(slot + 128 + c * 16, pk);
          }
          if (c == 0 && j > 0 && !active) mbar_wait(&pv_done[g], (k - 1) & 1);
          if (c == 1 && k == 0 && g == 0 && quarter == 0 && lane == 0) *half_step = 1;
          // refill the registers this step is done with from S_{k+1} (issued by the MMA warp when S_k was handed back)
          // (S_{k+1} takes ~800 cycles from the hand-over to its commit: waiting for it after two chunks, not one)
          if (has_next && c >= 2) {
            if (c == 2) {
              mbar_wait(&s_full[g], (k + 1) & 1);
              tc_fence_after();
              if (active1 && 0 < nch1) load_chunk(0);
              if (active1 && 1 < nch1) load_chunk(1);
            }
            if (active1 && c < nch1) load_chunk(c);
          }
        }
        if (active) {
          l = fmaf(l, alpha, s0 + s1);
          // O <- alpha * O before P V_k accumulates into it (only if some row of the warp raised its maximum)
          if (j > 0 && __any_sync(0xffffffffu, m_new > m)) {   // warp-uniform: set together in the hand-over
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              uint32_t o0[32];
              tmem_ld_32x32(slot + 192 + hh * 32, o0);
              tmem_ld_wait();
#pragma unroll
              for (int u = 0; u < 2; ++u) {
                uint32_t t16[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) t16[i] = __float_as_uint(__uint_as_float(o0[u * 16 + i]) * alpha);
                tmem_st_32x16(slot + 192 + hh * 32 + u * 16, t16);
              }
            }
          }
          m = m_new;
          tmem_st_wait();
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&p_full[g]);
        if (stamp && j < 5) trace[16 * g + 3 * j + 1] = clock64();

        if (j == QT - 1) {
          // ---- O read-out, normalisation, staging (the loads of the next q tile's S_0 are in flight meanwhile) ----
          mbar_wait(&pv_done[g], k & 1);
          tc_fence_after();
          uint32_t ra[32];
          const float inv = 1.0f / l;
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            if (active) {
              tmem_ld_32x32(slot + 192 + hh * 32, ra);
              tmem_ld_wait();
            }
            if (hh == 1) {
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive(&o_free[g]);
            }
            if (active) {
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const int e = u * 8;
                uint4 v4;
                v4.x = pack_bf16x2(__uint_as_float(ra[e + 0]) * inv, __uint_as_float(ra[e + 1]) * inv);
                v4.y = pack_bf16x2(__uint_as_float(ra[e + 2]) * inv, __uint_as_float(ra[e + 3]) * inv);
                v4.z = pack_bf16x2(__uint_as_float(ra[e + 4]) * inv, __uint_as_float(ra[e + 5]) * inv);
                v4.w = pack_bf16x2(__uint_as_float(ra[e + 6]) * inv, __uint_as_float(ra[e + 7]) * inv);
                st_swz(stg, rr, hh * 4 + u, v4);
              }
            }
          }
          if (active) {
            const int q = qt * TILE + rr;
            if (q < N && lse) lse[((long long)b * H + h) * N + q] = m * scale + __logf(l);
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(&o_staged[g]);
          m = -INFINITY;
          l = 0.f;
        }

        if (has_next) {
          if (active1) tmem_ld_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&s_read[g]);   // the MMA warp may overwrite S with S_{k+2}
          if (active1) {
            // the reference of a row is its running maximum (rescale whenever some row of the warp raised it)
            m_new = row_max(kvn1, nch1, m);
            if (__any_sync(0xffffffffu, (m_new - m) * c2 > 0.f)) {
              alpha = ex2_approx((m - m_new) * c2);   // 0 on the first kv tile of a q tile (m = -inf)
            } else {
              m_new = m;
              alpha = 1.f;
            }
          }
        }
        if (stamp && j < 5) trace[16 * g + 3 * j + 2] = clock64();
      }
      active = active1;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 10) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

int launch_fwd6(const CUtensorMap& tm, const CUtensorMap& tm_out, float* lse, int B, int N, int H, float scale, cudaStream_t s) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(attn_fwd6_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Fwd6Smem::BYTES);
    if (e != cudaSuccess) return vitk_set_error(VITK_ERR_CUDA, "attn_fwd6: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    attr_set = true;
  }
  const int QT = (N + TILE - 1) / TILE;
  const int items = B * H * ((QT + 1) / 2);
  const int grid = items < vitk_num_sms() ? items : vitk_num_sms();
  attn_fwd6_kernel<<<grid, FWD6_THREADS, Fwd6Smem::BYTES, s>>>(tm, tm_out, lse, B, N, H, scale, g_trace_buf);
  return vitk_check_launch("attn_fwd6");
}

// D[b, h, n] = sum_d O[b, n, h, d] * dO[b, n, h, d]: one warp per token row, fully coalesced 16-byte loads.
// (Computing it inside the backward kernel costs ~10k cycles of exposed, row-strided global loads per CTA.)
__global__ void attn_dsum_kernel(const __nv_bfloat16* __restrict__ out, const __nv_bfloat16* __restrict__ dout,
                                 float* __restrict__ dsum, long long rows, int N, int H, int hd) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const long long b = row / N;
  const int n = (int)(row - b * N);
  const __nv_bfloat16* op = out + row * (long long)(H * hd);
  const __nv_bfloat16* dp = dout + row * (long long)(H * hd);
  const int u = lane & 7;              // 16-byte chunk of the head: 8 lanes per head, 4 heads per pass
  const bool live = u * 8 < hd;
  for (int h0 = 0; h0 < H; h0 += 4) {
    const int h = h0 + (lane >> 3);
    float s = 0.f;
    if (h < H && live) {
      const uint4 a = __ldg(reinterpret_cast<const uint4*>(op + h * hd) + u), d = __ldg(reinterpret_cast<const uint4*>(dp + h * hd) + u);
      const float2 a0 = unpack_bf16x2(a.x), a1 = unpack_bf16x2(a.y), a2 = unpack_bf16x2(a.z), a3 = unpack_bf16x2(a.w);
      const float2 d0 = unpack_bf16x2(d.x), d1 = unpack_bf16x2(d.y), d2 = unpack_bf16x2(d.z), d3 = unpack_bf16x2(d.w);
      s = a0.x * d0.x + a0.y * d0.y + a1.x * d1.x + a1.y * d1.y + a2.x * d2.x + a2.y * d2.y + a3.x * d3.x + a3.y * d3.y;
    }
    if (h < H && (u + 8) * 8 < hd) {   // head columns 64 .. (wide heads)
      const uint4 a = __ldg(reinterpret_cast<const uint4*>(op + h * hd) + u + 8), d = __ldg(reinterpret_cast<const uint4*>(dp + h * hd) + u + 8);
      const float2 a0 = unpack_bf16x2(a.x), a1 = unpack_bf16x2(a.y), a2 = unpack_bf16x2(a.z), a3 = unpack_bf16x2(a.w);
      const float2 d0 = unpack_bf16x2(d.x), d1 = unpack_bf16x2(d.y), d2 = unpack_bf16x2(d.z), d3 = unpack_bf16x2(d.w);
      s += a0.x * d0.x + a0.y * d0.y + a1.x * d1.x + a1.y * d1.y + a2.x * d2.x + a2.y * d2.y + a3.x * d3.x + a3.y * d3.y;
    }
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    if (u == 0 && h < H) dsum[(b * H + h) * N + n] = s;
  }
}

// ================================================================================================
// Backward, warp-specialised persistent kernel for 128 < N <= 256 (224-px ViT / DeiT: N = 197 / 198).
//
// One CTA per SM loops over (b, h) items.  320 threads:
//   warpgroup w (warps 4w..4w+3) owns q tile w, one thread per row (no cross-thread reductions); per kv tile j it turns
//     S_wj into P (bf16, smem), then dP_wj into dS (bf16, smem, over P) — S and dP share one 128-column TMEM buffer;
//   warp 8 issues every tcgen05.mma (uniform control flow, one elected lane) and alternates between the two
//     warpgroups, so one warpgroup's exp / dS math overlaps the other's GEMMs;
//   warp 9 is the TMA producer: K_0 / V_0 of the next item are prefetched while kv tile 1 is processed, the other
//     six tiles as soon as the last MMA of the item retires.
// No masking anywhere in the inner loops: kv rows >= N are zero-filled by TMA (they only reach discarded dK / dV rows
// and contribute 0 to dQ), q rows >= N have Q = dO = 0 and use lse = D = 0 (finite P, dS = 0).
// dQ / dK / dV rows leave through a warp-private 4 KB staging tile so that every global store instruction writes
// whole 128-byte lines (a thread storing its own row costs one L1 line per lane per instruction).
// TMEM: SdP_0 [0,128) | SdP_1 [128,256) | dV_j [256,320) | dK_j [320,384) | dQ_0 [384,448) | dQ_1 [448,512)
// smem: Q_w dO_w (64K) | K_j V_j (64K) | PdS_0 PdS_1 (64K) | 8 x 4K store staging | barriers
// ================================================================================================
struct Bwd3Smem {
  static constexpr uint32_t QDO_OFF = 0;                       // [w][Q, dO]
  static constexpr uint32_t KV_OFF = 4 * TILE_BYTES;           // [j][K, V]
  static constexpr uint32_t PDS_OFF = 8 * TILE_BYTES;          // [w][2 chunks of 64 kv columns][128 rows][128 B]
  static constexpr uint32_t STG_OFF = 12 * TILE_BYTES;         // [8 warps][32 rows][128 B]
  static constexpr uint32_t BAR_OFF = STG_OFF + 8 * 4096;
  static constexpr uint32_t BYTES = BAR_OFF + 256;
};
constexpr int BWD3_THREADS = 10 * 32;

// ================================================================================================
// attn_bwd4: the ping-pong schedule on the roles and smem / TMEM layout above (128 < N <= 256).
//
// Keeping the two warpgroups in lockstep (both do P, then both wait for the MMAs, then both do dS ...) leaves
// the tensor core idle while the CUDA cores work and vice versa.  Here warpgroup 1 runs half a step behind
// warpgroup 0: while one warpgroup turns S into P (MUFU), the other turns dP into dS (FP32 pipe), and the MMA
// warp serves them alternately in the fixed event order E1..E8 below.  What makes that possible with single
// dV / dK accumulators (TMEM is full) is WHEN they are read out:
//   * warpgroup 0 drains dV_j (and, after kv tile 1, dQ_0) only after its NEXT P phase, just before it hands P over —
//     by then dV_j is final (warpgroup 1's P of the same kv tile came half a step later);
//   * warpgroup 1 drains dK_j (and dQ_1) right after its dS phase, while it waits for its next S anyway.
// Event order of the MMA warp for item n  (X' = item n+1, "final" = tcgen05.commit on the named barrier):
//   E1  P_00  -> dV_0  = P_00^T dO_0,  dP_00                      E5  P_01 -> dV_1  = P_01^T dO_0, dP_01
//   E2a dS_11 of item n-1 -> dK_1 +=, dQ_1 += (final), frees Q_1 dO_1 K_1 V_1      E6  dS_10 -> dK_0 += (final), dQ_1 =, S_11, frees K_0 V_0
//   E2b S_10                                                       E7  dS_01 -> dK_1 =, dQ_0 += (final), frees Q_0 dO_0
//   E3  dS_00 -> dK_0 =, dQ_0 =, S_01                              E8  P_11 -> dV_1 += (final), dP_11;  then S_00'
//   E4  P_10  -> dV_0 += (final), dP_10
// ================================================================================================
__global__ void __launch_bounds__(BWD3_THREADS, 1)
attn_bwd4_kernel(const __grid_constant__ CUtensorMap tm_qkv, const __grid_constant__ CUtensorMap tm_do,
                 const __grid_constant__ CUtensorMap tm_dqkv, const float* __restrict__ dsum, const float* __restrict__ lse,
                 int B, int N, int H, float scale, long long* trace) {
  using L = Bwd3Smem;
  int tslot = 0;
#define BWD4_STAMP(base) do { if (trace != nullptr && blockIdx.x == 0 && n == 2 && lane == 0 && tslot < 32) trace[(base) + tslot++] = clock64(); } while (0)
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bar_q = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);  // [w] TMA -> MMA: Q_w, dO_w landed
  uint64_t* bar_kv = bar_q + 2;                                       // [j] TMA -> MMA: K_j, V_j landed
  uint64_t* empty_kv0 = bar_kv + 2;                                   // MMA -> TMA: K_0, V_0 free
  uint64_t* empty_q0 = empty_kv0 + 1;                                 // MMA -> TMA: Q_0, dO_0 free
  uint64_t* empty_rest = empty_q0 + 1;                                // MMA -> TMA: Q_1, dO_1, K_1, V_1 free
  uint64_t* bar_s = empty_rest + 1;                                   // [w] MMA -> WG: S_wj ready
  uint64_t* bar_p = bar_s + 2;                                        // [w] WG -> MMA: P_wj in smem
  uint64_t* bar_dp = bar_p + 2;                                       // [w] MMA -> WG: dP_wj ready, P_wj consumed
  uint64_t* bar_ds = bar_dp + 2;                                      // [w] WG -> MMA: dS_wj in smem
  uint64_t* bar_dvf = bar_ds + 2;                                     // MMA -> WG0: dV_j final
  uint64_t* bar_dkf = bar_dvf + 1;                                    // MMA -> WG1: dK_j final (j = 1: dQ_1 too)
  uint64_t* bar_dq0f = bar_dkf + 1;                                   // MMA -> WG0: dQ_0 final
  uint64_t* drained_dk = bar_dq0f + 1;                                // WG1 -> MMA: dK_j (and dQ_1) read out
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(drained_dk + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int items = B * H;
  const int G = (int)gridDim.x;
  const uint32_t eff1 = roundup16(N - TILE);   // rows of q tile 1 == columns of kv tile 1, rounded up to the MMA K step

  if ((smem_u32(smem) & 1023u) != 0) __trap();
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bar_q[i], 1);
      mbar_init(&bar_kv[i], 1);
      mbar_init(&bar_s[i], 1);
      mbar_init(&bar_p[i], 4);
      mbar_init(&bar_dp[i], 1);
      mbar_init(&bar_ds[i], 4);
    }
    mbar_init(empty_kv0, 1);
    mbar_init(empty_q0, 1);
    mbar_init(empty_rest, 1);
    mbar_init(bar_dvf, 1);
    mbar_init(bar_dkf, 1);
    mbar_init(bar_dq0f, 1);
    mbar_init(drained_dk, 4);
    fence_mbar_init();
  }
  if (warp == 9) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tm_dv = tmem_base + 256, tm_dk = tmem_base + 320, tm_dq = tmem_base + 384;

  if (warp == 9) {
    // ------------------------------ TMA producer ------------------------------
    if (lane == 0) {
      tma_prefetch_desc(&tm_qkv);
      tma_prefetch_desc(&tm_do);
      int n = 0;
      for (int it = blockIdx.x; it < items; it += G, ++n) {
        const int h = it % H, b = it / H;
        if (n > 0) mbar_wait(empty_kv0, (n - 1) & 1);
        mbar_arrive_expect_tx(&bar_kv[0], 2 * TILE_BYTES);
        tma_load_head(smem + L::KV_OFF, &tm_qkv, &bar_kv[0], H + h, 0, b);
        tma_load_head(smem + L::KV_OFF + TILE_BYTES, &tm_qkv, &bar_kv[0], 2 * H + h, 0, b);
        if (n > 0) mbar_wait(empty_q0, (n - 1) & 1);
        mbar_arrive_expect_tx(&bar_q[0], 2 * TILE_BYTES);
        tma_load_head(smem + L::QDO_OFF, &tm_qkv, &bar_q[0], h, 0, b);
        tma_load_head(smem + L::QDO_OFF + TILE_BYTES, &tm_do, &bar_q[0], h, 0, b);
        if (n > 0) mbar_wait(empty_rest, (n - 1) & 1);
        mbar_arrive_expect_tx(&bar_q[1], 2 * TILE_BYTES);
        tma_load_head(smem + L::QDO_OFF + 2 * TILE_BYTES, &tm_qkv, &bar_q[1], h, TILE, b);
        tma_load_head(smem + L::QDO_OFF + 3 * TILE_BYTES, &tm_do, &bar_q[1], h, TILE, b);
        mbar_arrive_expect_tx(&bar_kv[1], 2 * TILE_BYTES);
        tma_load_head(smem + L::KV_OFF + 2 * TILE_BYTES, &tm_qkv, &bar_kv[1], H + h, TILE, b);
        tma_load_head(smem + L::KV_OFF + 3 * TILE_BYTES, &tm_qkv, &bar_kv[1], 2 * H + h, TILE, b);
      }
    }
  } else if (warp == 8) {
    // ------------------------------ MMA issuer (whole warp runs the program, one elected lane issues) ------------------------------
    const uint32_t sQDO = smem_u32(smem + L::QDO_OFF), sKV = smem_u32(smem + L::KV_OFF), sPDS = smem_u32(smem + L::PDS_OFF);
    const uint32_t idesc_t = umma_idesc(TILE, HD, 1, true, true);    // A, B MN-major: P^T dO, dS^T Q
    const uint32_t idesc_q = umma_idesc(TILE, HD, 1, false, true);   // dS K
    // S_wj = Q_w K_j^T (what == 0) or dP_wj = dO_w V_j^T (what == 1) into SdP_w
    auto issue_qk = [&](int w, int j, int what, uint64_t* bar) {
      const uint32_t n_eff = j == 0 ? (uint32_t)TILE : eff1;
      const uint32_t idesc = umma_idesc(TILE, n_eff, 1, false, false);
      const uint64_t adesc = umma_desc_kmajor(sQDO + (w * 2 + what) * TILE_BYTES);
      const uint64_t bdesc = umma_desc_kmajor(sKV + (j * 2 + what) * TILE_BYTES);
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < HD / 16; ++k) umma_bf16_ss(tmem_base + w * 128, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, k > 0);
        umma_commit(bar);
      }
      __syncwarp();
    };
    // dV_j (+)= P_w^T dO_w  (fin: commit bar_dvf), then dP_wj
    auto issue_dv_dp = [&](int w, int j, bool fin) {
      const uint32_t q_eff = w == 0 ? (uint32_t)TILE : eff1;
      const uint64_t pdesc = umma_desc_mnmajor(sPDS + w * 2 * TILE_BYTES, TILE_BYTES);
      const uint64_t dodesc = umma_desc_mnmajor(sQDO + (w * 2 + 1) * TILE_BYTES, TILE_BYTES);
      if (elect_one()) {
        for (int k = 0; k < (int)q_eff / 16; ++k)
          umma_bf16_ss(tm_dv, pdesc + (uint64_t)(k * 128), dodesc + (uint64_t)(k * 128), idesc_t, (w > 0 || k > 0));
        if (fin) umma_commit(bar_dvf);
      }
      __syncwarp();
      issue_qk(w, j, 1, &bar_dp[w]);
    };
    // dK_j (+)= dS_w^T Q_w ; dQ_w (+)= dS_w K_j
    auto issue_dk_dq = [&](int w, int j) {
      const uint32_t q_eff = w == 0 ? (uint32_t)TILE : eff1;
      const uint32_t n_eff = j == 0 ? (uint32_t)TILE : eff1;
      const uint32_t sDS = sPDS + w * 2 * TILE_BYTES;
      const uint64_t dsdesc_t = umma_desc_mnmajor(sDS, TILE_BYTES);
      const uint64_t qdesc = umma_desc_mnmajor(sQDO + w * 2 * TILE_BYTES, TILE_BYTES);
      const uint64_t dsdesc_k = umma_desc_kmajor(sDS);
      const uint64_t kdesc = umma_desc_mnmajor(sKV + j * 2 * TILE_BYTES, TILE_BYTES);
      if (elect_one()) {
        for (int k = 0; k < (int)q_eff / 16; ++k)
          umma_bf16_ss(tm_dk, dsdesc_t + (uint64_t)(k * 128), qdesc + (uint64_t)(k * 128), idesc_t, (w > 0 || k > 0));
        for (int k = 0; k < (int)n_eff / 16; ++k)
          umma_bf16_ss(tm_dq + w * HD, dsdesc_k + (uint64_t)((k >> 2) * (TILE_BYTES >> 4) + (k & 3) * 2), kdesc + (uint64_t)(k * 128),
                       idesc_q, (j > 0 || k > 0));
      }
      __syncwarp();
    };
    auto commit = [&](uint64_t* bar) {
      if (elect_one()) umma_commit(bar);
      __syncwarp();
    };
    // Two in-order event queues, one per warpgroup, served in arrival order (non-blocking barrier tests): warpgroup 0's
    // queue is  S_00 | E1 | E3 | E5 | E7,  warpgroup 1's is  E2b (S_10) | E4 | E6 | E8 | E2a (of the same item).
    // Warpgroup 1's accumulating MMAs may only follow warpgroup 0's initialising ones (E4 after E1, E6 after E3, E8 after
    // E5, E2a after E7); everything else the two queues need from each other travels through the mbarriers tested here.
    const int nitems = (int)blockIdx.x < items ? (items - (int)blockIdx.x + G - 1) / G : 0;
    int n0 = 0, k0 = 0, n1 = 0, k1 = 0;
    [[maybe_unused]] const int n = 0;
    while (n1 < nitems) {
      if (n0 < nitems) {
        const uint32_t par = n0 & 1;
        bool ready = false;
        switch (k0) {
          case 0: ready = mbar_test(&bar_kv[0], par) && mbar_test(&bar_q[0], par); break;
          case 1: ready = mbar_test(&bar_p[0], 0); break;
          case 2: ready = mbar_test(&bar_ds[0], 0) && (n0 == 0 || mbar_test(drained_dk, 1)) && mbar_test(&bar_kv[1], par); break;
          case 3: ready = mbar_test(&bar_p[0], 1); break;
          default: ready = mbar_test(&bar_ds[0], 1) && mbar_test(drained_dk, 0); break;
        }
        if (ready) {
          tc_fence_after();
          switch (k0) {
            case 0: issue_qk(0, 0, 0, &bar_s[0]); break;
            case 1: issue_dv_dp(0, 0, false); break;
            case 2:
              issue_dk_dq(0, 0);
              issue_qk(0, 1, 0, &bar_s[0]);
              break;
            case 3: issue_dv_dp(0, 1, false); break;
            default:
              issue_dk_dq(0, 1);
              commit(bar_dq0f);
              commit(empty_q0);
              break;
          }
          if (++k0 == 5) { k0 = 0; ++n0; }
        }
      }
      {
        const uint32_t par = n1 & 1;
        const bool ahead = n0 > n1;   // warpgroup 0's queue has finished this item
        bool ready = false;
        switch (k1) {
          case 0: ready = mbar_test(&bar_q[1], par) && mbar_test(&bar_kv[0], par); break;
          case 1: ready = (ahead || k0 > 1) && mbar_test(&bar_p[1], 0); break;
          case 2: ready = (ahead || k0 > 2) && mbar_test(&bar_ds[1], 0); break;
          case 3: ready = (ahead || k0 > 3) && mbar_test(&bar_p[1], 1); break;
          default: ready = ahead && mbar_test(&bar_ds[1], 1); break;
        }
        if (ready) {
          tc_fence_after();
          switch (k1) {
            case 0: issue_qk(1, 0, 0, &bar_s[1]); break;
            case 1: issue_dv_dp(1, 0, true); break;
            case 2:
              issue_dk_dq(1, 0);
              commit(bar_dkf);
              commit(empty_kv0);
              issue_qk(1, 1, 0, &bar_s[1]);
              break;
            case 3: issue_dv_dp(1, 1, true); break;
            default:
              issue_dk_dq(1, 1);
              commit(bar_dkf);
              commit(empty_rest);
              break;
          }
          if (++k1 == 5) { k1 = 0; ++n1; }
        }
      }
    }
  } else {
    // ------------------------------ warpgroup w: rows of q tile w ------------------------------
    const int w = warp >> 2, r = threadIdx.x & 127;
    const uint32_t lane_addr = static_cast<uint32_t>((warp & 3) * 32) << 16;
    const uint32_t tm_sdp = tmem_base + w * 128 + lane_addr;
    uint8_t* sPDS = smem + L::PDS_OFF + w * 2 * TILE_BYTES;
    uint8_t* wst = smem + L::STG_OFF + warp * 4096;
    const int q = w * TILE + r;
    const bool row_ok = q < N;
    const uint32_t q_eff = w == 0 ? (uint32_t)TILE : eff1;
    const bool warp_active = (uint32_t)((warp & 3) * 32) < q_eff;   // some row of this warp is read by the dV / dK MMAs
    const float c2 = scale * LOG2E;
    // this warp's 32 accumulator rows (64 fp32 columns at TMEM column `tcol`) -> rows [row_first, ...) of part `which`
    // (0 = dQ, 1 = dK, 2 = dV) of head h of image b: bf16 into the warp's swizzled 4 KB tile, one TMA store (rows >= N
    // are clipped by the tensor map).  The previous store of this warp has long been read when the next one starts.
    auto drain = [&](uint32_t tcol, int which, int b, int h, int row_first) {
      if (row_first < N) {
        uint32_t a0[32], a1[32];
        tmem_ld_32x32(tcol + lane_addr, a0);
        tmem_ld_32x32(tcol + lane_addr + 32, a1);
        if (elect_one()) tma_store_wait_read();
        __syncwarp();
        tmem_ld_wait();
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const uint32_t(&v)[32] = u < 4 ? a0 : a1;
          const int e = (u & 3) * 8;
          uint4 o;
          o.x = pack_bf16x2(__uint_as_float(v[e + 0]), __uint_as_float(v[e + 1]));
          o.y = pack_bf16x2(__uint_as_float(v[e + 2]), __uint_as_float(v[e + 3]));
          o.z = pack_bf16x2(__uint_as_float(v[e + 4]), __uint_as_float(v[e + 5]));
          o.w = pack_bf16x2(__uint_as_float(v[e + 6]), __uint_as_float(v[e + 7]));
          *reinterpret_cast<uint4*>(wst + lane * 128 + ((u ^ (lane & 7)) << 4)) = o;
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (elect_one()) {
          tma_store_head(&tm_dqkv, wst, which * H + h, row_first, b);
          tma_store_commit();
        }
        __syncwarp();
      }
    };
    int n = 0;
    int pb = 0, ph = 0;   // previous item (warpgroup 0 drains it one P phase late)
    for (int it = blockIdx.x; it < items; it += G, ++n) {
      const int h = it % H, b = it / H;
      float my_lse2 = 0.f, my_ds = 0.f;   // rows >= N: P = 2^S stays finite, dS = 0
      if (row_ok) {
        my_lse2 = lse[((long long)b * H + h) * N + q] * LOG2E;
        my_ds = dsum[((long long)b * H + h) * N + q] * scale;
      }
      for (int j = 0; j < 2; ++j) {
        const uint32_t n_eff = j == 0 ? (uint32_t)TILE : eff1;
        const int nch = (int)(n_eff + 31) / 32;   // 32-column chunks (the last one may be half)

        // ---- S -> P ----
        mbar_wait(&bar_s[w], j);
        tc_fence_after();
        if ((warp & 3) == 0) BWD4_STAMP(32 + 16 * w);
        if (warp_active) {
          uint32_t ra[32], rb[32];
          auto p_chunk = [&](const uint32_t (&v)[32], int c) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              uint32_t pk[4];
#pragma unroll
              for (int i = 0; i < 4; ++i)
                pk[i] = pack_bf16x2(ex2_approx(fmaf(__uint_as_float(v[g * 8 + 2 * i]), c2, -my_lse2)),
                                    ex2_approx(fmaf(__uint_as_float(v[g * 8 + 2 * i + 1]), c2, -my_lse2)));
              st_swz(sPDS, r, c * 4 + g, make_uint4(pk[0], pk[1], pk[2], pk[3]));
            }
          };
          tmem_ld_32x32(tm_sdp, ra);
          tmem_ld_wait();
#pragma unroll
          for (int c = 0; c < 4; c += 2) {
            if (c < nch) {
              if (c + 1 < nch) tmem_ld_32x32(tm_sdp + (c + 1) * 32, rb);
              p_chunk(ra, c);
              if (c + 1 < nch) {
                tmem_ld_wait();
                if (c + 2 < nch) tmem_ld_32x32(tm_sdp + (c + 2) * 32, ra);
                p_chunk(rb, c + 1);
                if (c + 2 < nch) tmem_ld_wait();
              }
            }
          }
        }
        if (w == 0) {
          // deferred read-out: dV of the previous kv tile (and dQ_0 of the previous item) are final by now
          if (j == 1) {
            mbar_wait(bar_dvf, 0);
            tc_fence_after();
            drain(tm_dv, 2, b, h, (warp & 3) * 32);
          } else if (n > 0) {
            mbar_wait(bar_dvf, 1);
            tc_fence_after();
            drain(tm_dv, 2, pb, ph, TILE + (warp & 3) * 32);
          }
        }
        fence_proxy_async_smem();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_p[w]);
        if ((warp & 3) == 0) BWD4_STAMP(32 + 16 * w);

        // ---- dP -> dS (over P) ----
        mbar_wait(&bar_dp[w], j);
        tc_fence_after();
        if ((warp & 3) == 0) BWD4_STAMP(32 + 16 * w);
        if (warp_active) {
          uint32_t ra[32], rb[32];
          auto ds_chunk = [&](const uint32_t (&v)[32], int c) {
            uint4 pall[4];   // all four loads first: the compiler cannot hoist them above the (possibly aliasing) stores
#pragma unroll
            for (int g = 0; g < 4; ++g)
              pall[g] = *reinterpret_cast<const uint4*>(sPDS + ((c * 4 + g) >> 3) * TILE_BYTES + r * 128 + ((((c * 4 + g) & 7) ^ (r & 7)) << 4));
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              uint8_t* slot = sPDS + ((c * 4 + g) >> 3) * TILE_BYTES + r * 128 + ((((c * 4 + g) & 7) ^ (r & 7)) << 4);
              const uint4 pu = pall[g];
              const uint32_t pw[4] = {pu.x, pu.y, pu.z, pu.w};
              uint32_t ds[4];
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float2 pp = unpack_bf16x2(pw[i]);
                ds[i] = pack_bf16x2(pp.x * fmaf(__uint_as_float(v[g * 8 + 2 * i]), scale, -my_ds),
                                    pp.y * fmaf(__uint_as_float(v[g * 8 + 2 * i + 1]), scale, -my_ds));
              }
              *reinterpret_cast<uint4*>(slot) = make_uint4(ds[0], ds[1], ds[2], ds[3]);
            }
          };
          tmem_ld_32x32(tm_sdp, ra);
          tmem_ld_wait();
#pragma unroll
          for (int c = 0; c < 4; c += 2) {
            if (c < nch) {
              if (c + 1 < nch) tmem_ld_32x32(tm_sdp + (c + 1) * 32, rb);
              ds_chunk(ra, c);
              if (c + 1 < nch) {
                tmem_ld_wait();
                if (c + 2 < nch) tmem_ld_32x32(tm_sdp + (c + 2) * 32, ra);
                ds_chunk(rb, c + 1);
                if (c + 2 < nch) tmem_ld_wait();
              }
            }
          }
        }
        fence_proxy_async_smem();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_ds[w]);
        if ((warp & 3) == 0) BWD4_STAMP(32 + 16 * w);

        if (w == 0 && j == 1) {
          // dQ_0 is final once the MMAs fed by this dS retire; read it out while the next item's Q_0 is still loading
          mbar_wait(bar_dq0f, n & 1);
          tc_fence_after();
          drain(tm_dq, 0, b, h, (warp & 3) * 32);
        }
        if (w == 1) {
          // dK_j is final half a step after this warpgroup's dS (it is the second contributor); read it out while
          // waiting for the next S anyway.  After kv tile 1 the same holds for dQ_1.
          mbar_wait(bar_dkf, j);
          tc_fence_after();
          drain(tm_dk, 1, b, h, j * TILE + (warp & 3) * 32);
          if (j == 1) drain(tm_dq + HD, 0, b, h, TILE + (warp & 3) * 32);
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(drained_dk);
          if ((warp & 3) == 0) BWD4_STAMP(32 + 16 * w);
        }
      }
      pb = b;
      ph = h;
    }
    if (w == 0 && n > 0) {   // the last item's deferred read-out
      mbar_wait(bar_dvf, 1);
      tc_fence_after();
      drain(tm_dv, 2, pb, ph, TILE + (warp & 3) * 32);
    }
    if (elect_one()) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // smem must outlive the bulk stores
    __syncwarp();
  }
#undef BWD4_STAMP

  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ================================================================================================
// Backward, streaming: every call but the unmasked 128 < N <= 256 at head_dim <= 64 (attn_bwd4), e.g. N <= 128, ViT-L/16
// at 384 px (N = 577), a keep mask, wide heads.  One CTA per (b, h, kv tile j).
// K_j / V_j stay resident, Q_i / dO_i stream through one smem buffer, dV_j / dK_j accumulate in TMEM over the
// q tiles, and each dQ_ij partial is read out of a TMEM scratch tile.  With more than one kv tile it is red.add'ed into
// an fp32 workspace [B, N, H*64] (the q rows are shared by the T CTAs of a head) that a small kernel then casts into
// dqkv; with one kv tile (dq32 == null) dQ_i0 is final and is stored as bf16 directly.
// TMEM: S [0,128) | dP [128,256) | dV_j [256,320) | dK_j [320,384) | dQ_ij [384,448)
// WIDE (64 < head_dim <= 80, used for every N then): operands are [64-column tile][tail tile] pairs (see HDW_MAX), S and dP
// take one more k-step, dV / dK / dQ have 80 accumulator columns (TMEM: 256 | 336 | 416 .. 496), Q_i / dO_i are single-
// buffered (192 KB of smem otherwise) and the fp32 dQ workspace keeps 80-wide heads.
// ================================================================================================
template <bool WIDE>
struct BwdStreamSmem {
  static constexpr uint32_t OPB = WIDE ? 2 * TILE_BYTES : TILE_BYTES;
  static constexpr int NBUF = WIDE ? 1 : 2;
  static constexpr uint32_t KV_OFF = 0;
  static constexpr uint32_t QDO_OFF = 2 * OPB;                     // [NBUF buffers][Q_i, dO_i]
  static constexpr uint32_t P_OFF = QDO_OFF + NBUF * 2 * OPB;
  static constexpr uint32_t DS_OFF = P_OFF + 2 * TILE_BYTES;
  static constexpr uint32_t BAR_OFF = DS_OFF + 2 * TILE_BYTES;
  static constexpr uint32_t BYTES = BAR_OFF + 128;
};

// accumulator columns 64 .. 79 of a wide head -> bf16 (the first hd - 64 of them exist)
__device__ __forceinline__ void store_row_bf16_tail(__nv_bfloat16* dst, const uint32_t (&a)[16], int n) {
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    if (g * 8 >= n) break;
    uint4 u;
    u.x = pack_bf16x2(__uint_as_float(a[g * 8 + 0]), __uint_as_float(a[g * 8 + 1]));
    u.y = pack_bf16x2(__uint_as_float(a[g * 8 + 2]), __uint_as_float(a[g * 8 + 3]));
    u.z = pack_bf16x2(__uint_as_float(a[g * 8 + 4]), __uint_as_float(a[g * 8 + 5]));
    u.w = pack_bf16x2(__uint_as_float(a[g * 8 + 6]), __uint_as_float(a[g * 8 + 7]));
    *reinterpret_cast<uint4*>(dst + g * 8) = u;
  }
}

// Q_i / dO_i are double-buffered (tile i+1 is loading while tile i is processed), S / dP of tile i+1 are issued right
// behind the dV / dK / dQ MMAs of tile i (their TMEM buffers are free once the threads have read them), so they execute
// while the threads read dQ_ij out.  D = rowsum(O * dO) comes from the workspace (attn_dsum_kernel).
// No masks: kv rows >= N are TMA zero fill (they reach only discarded dK / dV rows and add 0 to dQ); q rows >= N have
// Q = dO = 0 and use lse = D = 0.
template <bool WIDE>
__global__ void __launch_bounds__(128)
attn_bwd_stream_kernel(const __grid_constant__ CUtensorMap tm_qkv, const __grid_constant__ CUtensorMap tm_do,
                       const float* __restrict__ dsum, const float* __restrict__ lse, __nv_bfloat16* __restrict__ dqkv,
                       float* __restrict__ dq32, int N, int H, int hd, float scale, const uint8_t* __restrict__ drop_mask,
                       float drop_scale) {
  // drop_mask (attn_drop): keep bytes [B, H, N, N] or null: dV sees P m / keep, dS = P (dP m / keep - D)
  using L = BwdStreamSmem<WIDE>;
  constexpr int HDW = WIDE ? HDW_MAX : HD;   // accumulator columns of dV / dK / dQ, head pitch of the dQ workspace
  constexpr int NBUF = L::NBUF;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bar_kv = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);
  uint64_t* bar_q = bar_kv + 1;     // [2]
  uint64_t* bar_sp = bar_q + 2;
  uint64_t* bar_mma = bar_sp + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_mma + 1);

  const int warp = threadIdx.x >> 5;
  const int j = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int nt = (N + TILE - 1) / TILE;
  const int kvn = min(TILE, N - j * TILE);
  const uint32_t n_eff = roundup16(kvn);
  const int nchunks = (int)(n_eff + 31) / 32;

  if ((smem_u32(smem) & 1023u) != 0) __trap();
  if (dq32 == nullptr && gridDim.x > 1) __trap();   // a direct bf16 dQ store is final only with one kv tile
  if (threadIdx.x == 32) {
    mbar_init(bar_kv, 1);
    mbar_init(&bar_q[0], 1);
    mbar_init(&bar_q[1], 1);
    mbar_init(bar_sp, 1);
    mbar_init(bar_mma, 1);
    fence_mbar_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tm_s = tmem_base, tm_dp = tmem_base + 128, tm_dv = tmem_base + 256, tm_dk = tm_dv + HDW;
  const uint32_t tm_dq = tm_dk + HDW;
  const uint32_t lane_addr = static_cast<uint32_t>(warp * 32) << 16;
  const int r = threadIdx.x;
  const float c2 = scale * LOG2E;
  uint8_t* sP = smem + L::P_OFF;
  uint8_t* sDS = smem + L::DS_OFF;
  const uint32_t sK = smem_u32(smem + L::KV_OFF), sV = sK + L::OPB;
  const uint32_t sQDO = smem_u32(smem + L::QDO_OFF);
  const uint32_t sP_u = smem_u32(sP), sDS_u = smem_u32(sDS);
  const uint32_t idesc = umma_idesc(TILE, n_eff, 1, false, false);
  const uint64_t kd = umma_desc_kmajor(sK), vd = umma_desc_kmajor(sV), k_mn = umma_desc_mnmajor(sK, TILE_BYTES);
  const uint64_t kd_t = umma_desc_kmajor(sK + TILE_BYTES), vd_t = umma_desc_kmajor(sV + TILE_BYTES);   // WIDE: head columns 64 .. 79
  auto buf_of = [&](int i) { return NBUF == 2 ? (i & 1) : 0; };
  auto phase_of = [&](int i) { return NBUF == 2 ? ((i >> 1) & 1) : (i & 1); };

  auto load_q = [&](int i) {   // thread 0 only
    const int buf = buf_of(i);
    mbar_arrive_expect_tx(&bar_q[buf], 2 * L::OPB);
    load_head_tiles<WIDE>(smem + L::QDO_OFF + buf * 2 * L::OPB, &tm_qkv, &bar_q[buf], h, i * TILE, b);
    load_head_tiles<WIDE>(smem + L::QDO_OFF + buf * 2 * L::OPB + L::OPB, &tm_do, &bar_q[buf], h, i * TILE, b);
  };
  // S = Q_i K_j^T and dP = dO_i V_j^T (warp 0, uniform control flow, one elected lane)
  auto issue_s_dp = [&](int i) {
    const uint32_t sQ = sQDO + buf_of(i) * 2 * L::OPB, sDO = sQ + L::OPB;
    const uint64_t qd = umma_desc_kmajor(sQ), dod = umma_desc_kmajor(sDO);
    const uint64_t qd_t = umma_desc_kmajor(sQ + TILE_BYTES), dod_t = umma_desc_kmajor(sDO + TILE_BYTES);
    mbar_wait(&bar_q[buf_of(i)], phase_of(i));
    tc_fence_after();
    if (elect_one()) {
#pragma unroll
      for (int k = 0; k < HD / 16; ++k) umma_bf16_ss(tm_s, qd + (uint64_t)(k * 2), kd + (uint64_t)(k * 2), idesc, k > 0);
      if (WIDE) umma_bf16_ss(tm_s, qd_t, kd_t, idesc, true);
#pragma unroll
      for (int k = 0; k < HD / 16; ++k) umma_bf16_ss(tm_dp, dod + (uint64_t)(k * 2), vd + (uint64_t)(k * 2), idesc, k > 0);
      if (WIDE) umma_bf16_ss(tm_dp, dod_t, vd_t, idesc, true);
      umma_commit(bar_sp);
    }
    __syncwarp();
  };

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tm_qkv);
    tma_prefetch_desc(&tm_do);
    mbar_arrive_expect_tx(bar_kv, 2 * L::OPB);
    load_head_tiles<WIDE>(smem + L::KV_OFF, &tm_qkv, bar_kv, H + h, j * TILE, b);
    load_head_tiles<WIDE>(smem + L::KV_OFF + L::OPB, &tm_qkv, bar_kv, 2 * H + h, j * TILE, b);
    load_q(0);
    if (NBUF == 2 && nt > 1) load_q(1);
  }
  if (warp == 0) {
    mbar_wait(bar_kv, 0);
    issue_s_dp(0);
  }

  for (int i = 0; i < nt; ++i) {
    const int qn = min(TILE, N - i * TILE);
    const uint32_t q_eff = roundup16(qn);
    const bool row_ok = r < qn;
    const int q = i * TILE + r;
    float my_lse2 = 0.f, my_ds = 0.f;   // rows >= N: P = 2^S stays finite, dS = 0
    if (row_ok) {
      my_lse2 = lse[((long long)b * H + h) * N + q] * LOG2E;
      my_ds = dsum[((long long)b * H + h) * N + q] * scale;
    }
    mbar_wait(bar_sp, i & 1);
    tc_fence_after();
    if ((uint32_t)(warp * 32) < q_eff) {   // warp-uniform: some row of this warp is read by the dV / dK MMAs
      uint32_t sa[32], da[32], sb[32], db[32];
      auto chunk = [&](const uint32_t (&sv)[32], const uint32_t (&dv)[32], int c) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint32_t pk[4], dk[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float e0 = ex2_approx(fmaf(__uint_as_float(sv[g * 8 + 2 * k]), c2, -my_lse2));
            const float e1 = ex2_approx(fmaf(__uint_as_float(sv[g * 8 + 2 * k + 1]), c2, -my_lse2));
            float m0 = 1.f, m1 = 1.f;   // dropout factor of the two elements (mask / keep_prob)
            if (drop_mask != nullptr) {
              const int col = j * TILE + c * 32 + g * 8 + 2 * k;
              const uint8_t* mrow = drop_mask + (((long long)b * H + h) * N + q) * N + col;
              m0 = (row_ok && col < N && mrow[0]) ? drop_scale : 0.f;
              m1 = (row_ok && col + 1 < N && mrow[1]) ? drop_scale : 0.f;
            }
            pk[k] = pack_bf16x2(e0 * m0, e1 * m1);
            dk[k] = pack_bf16x2(e0 * fmaf(__uint_as_float(dv[g * 8 + 2 * k]), scale * m0, -my_ds),
                                e1 * fmaf(__uint_as_float(dv[g * 8 + 2 * k + 1]), scale * m1, -my_ds));
          }
          st_swz(sP, r, c * 4 + g, make_uint4(pk[0], pk[1], pk[2], pk[3]));
          st_swz(sDS, r, c * 4 + g, make_uint4(dk[0], dk[1], dk[2], dk[3]));
        }
      };
      tmem_ld_32x32(tm_s + lane_addr, sa);
      tmem_ld_32x32(tm_dp + lane_addr, da);
      tmem_ld_wait();
#pragma unroll
      for (int c = 0; c < 4; c += 2) {
        if (c < nchunks) {
          if (c + 1 < nchunks) {
            tmem_ld_32x32(tm_s + lane_addr + (c + 1) * 32, sb);
            tmem_ld_32x32(tm_dp + lane_addr + (c + 1) * 32, db);
          }
          chunk(sa, da, c);
          if (c + 1 < nchunks) {
            tmem_ld_wait();
            if (c + 2 < nchunks) {
              tmem_ld_32x32(tm_s + lane_addr + (c + 2) * 32, sa);
              tmem_ld_32x32(tm_dp + lane_addr + (c + 2) * 32, da);
            }
            chunk(sb, db, c + 1);
            if (c + 2 < nchunks) tmem_ld_wait();
          }
        }
      }
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
      const uint32_t sQ = sQDO + buf_of(i) * 2 * L::OPB, sDO = sQ + L::OPB;
      const uint32_t idesc_t = umma_idesc(TILE, HDW, 1, true, true);
      const uint32_t idesc_q = umma_idesc(TILE, HDW, 1, false, true);
      const int qsteps = (int)q_eff / 16;
      // MN-major B operands over the head dimension: the tail tile is their second 64-wide chunk (pitch TILE_BYTES)
      const uint64_t p_mn = umma_desc_mnmajor(sP_u, TILE_BYTES), do_mn = umma_desc_mnmajor(sDO, TILE_BYTES);
      const uint64_t ds_mn = umma_desc_mnmajor(sDS_u, TILE_BYTES), q_mn = umma_desc_mnmajor(sQ, TILE_BYTES);
      const uint64_t ds_k = umma_desc_kmajor(sDS_u);
      if (elect_one()) {
        for (int k = 0; k < qsteps; ++k) umma_bf16_ss(tm_dv, p_mn + (uint64_t)(k * 128), do_mn + (uint64_t)(k * 128), idesc_t, (i > 0 || k > 0));
        for (int k = 0; k < qsteps; ++k) umma_bf16_ss(tm_dk, ds_mn + (uint64_t)(k * 128), q_mn + (uint64_t)(k * 128), idesc_t, (i > 0 || k > 0));
        for (int k = 0; k < (int)n_eff / 16; ++k)
          umma_bf16_ss(tm_dq, ds_k + (uint64_t)((k >> 2) * (TILE_BYTES >> 4) + (k & 3) * 2), k_mn + (uint64_t)(k * 128), idesc_q, k > 0);
        umma_commit(bar_mma);
      }
      __syncwarp();
      // S / dP of the next q tile run while the threads read dQ_ij out (every thread has read S / dP of this tile)
      if (NBUF == 2 && i + 1 < nt) issue_s_dp(i + 1);
    }
    mbar_wait(bar_mma, i & 1);
    tc_fence_after();
    // Q_i / dO_i are no longer read: their buffer takes tile i + 2 (i + 1 when there is one buffer)
    if (threadIdx.x == 0 && i + NBUF < nt) load_q(i + NBUF);
    {
      uint32_t a0[32], a1[32];
      tmem_ld_32x32(tm_dq + lane_addr, a0);
      tmem_ld_32x32(tm_dq + lane_addr + 32, a1);
      tmem_ld_wait();
      __nv_bfloat16* dq_row = dqkv + ((long long)b * N + q) * (3 * H * hd) + h * hd;
      float* dst = dq32 != nullptr ? dq32 + ((long long)b * N + q) * (H * HDW) + h * HDW : nullptr;
      if (row_ok && dst == nullptr) {
        store_row_bf16_64(dq_row, a0, a1, hd);
      } else if (row_ok) {
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + g * 4), "f"(__uint_as_float(a0[g * 4])),
                       "f"(__uint_as_float(a0[g * 4 + 1])), "f"(__uint_as_float(a0[g * 4 + 2])),
                       "f"(__uint_as_float(a0[g * 4 + 3]))
                       : "memory");
          asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + 32 + g * 4), "f"(__uint_as_float(a1[g * 4])),
                       "f"(__uint_as_float(a1[g * 4 + 1])), "f"(__uint_as_float(a1[g * 4 + 2])),
                       "f"(__uint_as_float(a1[g * 4 + 3]))
                       : "memory");
        }
      }
      if (WIDE) {
        uint32_t a2[16];
        tmem_ld_32x16(tm_dq + lane_addr + 64, a2);
        tmem_ld_wait();
        if (row_ok && dst == nullptr) {
          store_row_bf16_tail(dq_row + 64, a2, hd - 64);
        } else if (row_ok) {
#pragma unroll
          for (int g = 0; g < 4; ++g)
            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + 64 + g * 4), "f"(__uint_as_float(a2[g * 4])),
                         "f"(__uint_as_float(a2[g * 4 + 1])), "f"(__uint_as_float(a2[g * 4 + 2])),
                         "f"(__uint_as_float(a2[g * 4 + 3]))
                         : "memory");
        }
      }
    }
    tc_fence_before();
    __syncthreads();  // P / dS / the dQ scratch may be overwritten by the next q tile
    tc_fence_after();
    if (NBUF == 1 && warp == 0 && i + 1 < nt) issue_s_dp(i + 1);   // the single Q / dO buffer has just been reloaded
  }

  {
    uint32_t a0[32], a1[32];
    const int kv = j * TILE + r;
    __nv_bfloat16* dv_row = dqkv + ((long long)b * N + kv) * (3 * H * hd) + (2 * H + h) * hd;
    __nv_bfloat16* dk_row = dqkv + ((long long)b * N + kv) * (3 * H * hd) + (H + h) * hd;
    tmem_ld_32x32(tm_dv + lane_addr, a0);
    tmem_ld_32x32(tm_dv + lane_addr + 32, a1);
    tmem_ld_wait();
    if (kv < N) store_row_bf16_64(dv_row, a0, a1, hd);
    tmem_ld_32x32(tm_dk + lane_addr, a0);
    tmem_ld_32x32(tm_dk + lane_addr + 32, a1);
    tmem_ld_wait();
    if (kv < N) store_row_bf16_64(dk_row, a0, a1, hd);
    if (WIDE) {
      uint32_t t0[16], t1[16];
      tmem_ld_32x16(tm_dv + lane_addr + 64, t0);
      tmem_ld_32x16(tm_dk + lane_addr + 64, t1);
      tmem_ld_wait();
      if (kv < N) {
        store_row_bf16_tail(dv_row + 64, t0, hd - 64);
        store_row_bf16_tail(dk_row + 64, t1, hd - 64);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// dqkv[row, h * hd + c] = bf16(dq32[row, h * pitch + c]) for c < hd: the fp32 dQ workspace keeps the padded heads of the
// tiles (pitch 64, or 80 for wide heads), dqkv is the gradient of the qkv Linear output (row pitch 3 * H * hd)
__global__ void dq_cast_kernel(const float* __restrict__ dq32, __nv_bfloat16* __restrict__ dqkv, long long rows, int H, int hd, int pitch) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int per_row = H * (hd / 8);
  if (idx >= rows * per_row) return;
  const long long row = idx / per_row;
  const int rem = (int)(idx - row * per_row);
  const int h = rem / (hd / 8), c = (rem - h * (hd / 8)) * 8;
  const float* src = dq32 + (row * H + h) * pitch + c;
  const float4 a = *reinterpret_cast<const float4*>(src);
  const float4 b2 = *reinterpret_cast<const float4*>(src + 4);
  uint4 u;
  u.x = pack_bf16x2(a.x, a.y);
  u.y = pack_bf16x2(a.z, a.w);
  u.z = pack_bf16x2(b2.x, b2.y);
  u.w = pack_bf16x2(b2.z, b2.w);
  *reinterpret_cast<uint4*>(dqkv + row * 3 * H * hd + h * hd + c) = u;
}

// ================================================================================================
// Forward, kv-streaming: every call but the unmasked 128 < N at head_dim <= 64 (attn_fwd4 / attn_fwd6), i.e. N <= 128, a
// keep mask at any N up to ATTN_MAX_N, and wide heads (N <= WIDE_MAX_N).
// One CTA per (b, h, 128-row q tile), thread t owns row t; K_j / V_j stream through a FWDS_STAGES-deep TMA ring (a stage
// is refilled as soon as P V_j has retired) and O accumulates in TMEM across kv tiles: before P V_j accumulates into it,
// a warp rescales its rows of O in place if some row raised its maximum.
// Per kv tile: S_j (issued behind P V_{j-1}) -> row max -> wait P V_{j-1} -> refill its stage, rescale O -> exps (+ keep
// mask) -> P -> smem -> P V_j.  Dropout (§4.7): the row sum is taken before the mask, m / keep multiplies the P tile that
// feeds P V, lse is that of the undropped scores.
// Narrow: 112 KB of smem and 256 TMEM columns, so two CTAs share an SM and one's exps overlap the other's MMAs.
// WIDE: operands are [tile][tail] pairs (see HDW_MAX), S takes one more k-step, O has 80 columns; 192 KB of smem.
// ================================================================================================
constexpr int FWDS_STAGES = 2;

template <bool WIDE>
struct FwdStreamSmem {
  static constexpr uint32_t OPB = WIDE ? 2 * TILE_BYTES : TILE_BYTES;   // bytes of one operand tile (+ tail)
  static constexpr uint32_t Q_OFF = 0;
  static constexpr uint32_t KV_OFF = OPB;                                      // [stage][K, V]
  static constexpr uint32_t P_OFF = KV_OFF + FWDS_STAGES * 2 * OPB;
  static constexpr uint32_t BAR_OFF = P_OFF + 2 * TILE_BYTES;
  static constexpr uint32_t BYTES = BAR_OFF + 128;
};

template <bool WIDE>
__global__ void __launch_bounds__(128)
attn_fwd_stream_kernel(const __grid_constant__ CUtensorMap tm_qkv, __nv_bfloat16* __restrict__ out, float* __restrict__ lse,
                       int N, int H, int hd, float scale, const uint8_t* __restrict__ drop_mask, float drop_scale) {
  using L = FwdStreamSmem<WIDE>;
  constexpr int HDW = WIDE ? HDW_MAX : HD;   // accumulator columns of O
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bar_q = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);
  uint64_t* kv_full = bar_q + 1;   // [FWDS_STAGES]
  uint64_t* bar_s = kv_full + FWDS_STAGES;
  uint64_t* bar_o = bar_s + 1;     // completes once per kv tile: P V_j retired
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_o + 1);

  const int warp = threadIdx.x >> 5;
  const int q0 = blockIdx.x * TILE, h = blockIdx.y, b = blockIdx.z;
  const int nkv = (N + TILE - 1) / TILE;

  if ((smem_u32(smem) & 1023u) != 0) __trap();
  if (threadIdx.x == 32) {
    mbar_init(bar_q, 1);
    for (int s = 0; s < FWDS_STAGES; ++s) mbar_init(&kv_full[s], 1);
    mbar_init(bar_s, 1);
    mbar_init(bar_o, 1);
    fence_mbar_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_slot, 256);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_s = tmem_base;         // S_j: 128 columns
  const uint32_t tmem_o = tmem_base + 128;   // O: 64 (80) columns, accumulated over every kv tile

  auto load_kv = [&](int j) {   // thread 0 only
    const int st = j % FWDS_STAGES;
    uint8_t* dst = smem + L::KV_OFF + st * 2 * L::OPB;
    mbar_arrive_expect_tx(&kv_full[st], 2 * L::OPB);
    load_head_tiles<WIDE>(dst, &tm_qkv, &kv_full[st], H + h, j * TILE, b);
    load_head_tiles<WIDE>(dst + L::OPB, &tm_qkv, &kv_full[st], 2 * H + h, j * TILE, b);
  };
  const uint32_t sQ_u = smem_u32(smem + L::Q_OFF);
  // S_j = Q K_j^T (warp 0: uniform control flow, one elected lane)
  auto issue_s = [&](int j) {
    const uint32_t sK_u = smem_u32(smem + L::KV_OFF + (j % FWDS_STAGES) * 2 * L::OPB);
    mbar_wait(&kv_full[j % FWDS_STAGES], (j / FWDS_STAGES) & 1);
    tc_fence_after();
    const uint32_t idesc = umma_idesc(TILE, roundup16(min(TILE, N - j * TILE)), 1, false, false);
    const uint64_t qd = umma_desc_kmajor(sQ_u), kd = umma_desc_kmajor(sK_u);
    if (elect_one()) {
#pragma unroll
      for (int k = 0; k < HD / 16; ++k) umma_bf16_ss(tmem_s, qd + (uint64_t)(k * 2), kd + (uint64_t)(k * 2), idesc, k > 0);
      if (WIDE) umma_bf16_ss(tmem_s, umma_desc_kmajor(sQ_u + TILE_BYTES), umma_desc_kmajor(sK_u + TILE_BYTES), idesc, true);
      umma_commit(bar_s);
    }
    __syncwarp();
  };

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tm_qkv);
    mbar_arrive_expect_tx(bar_q, L::OPB);
    load_head_tiles<WIDE>(smem + L::Q_OFF, &tm_qkv, bar_q, h, q0, b);
    for (int j = 0; j < FWDS_STAGES && j < nkv; ++j) load_kv(j);
  }
  if (warp == 0) {
    mbar_wait(bar_q, 0);
    issue_s(0);
  }

  const uint32_t lane_addr = static_cast<uint32_t>(warp * 32) << 16;
  const int r = threadIdx.x;  // row inside the q tile
  const int qrow = q0 + r;
  const float c2 = scale * LOG2E;
  float m_run = -INFINITY, l_run = 0.f;
  uint8_t* sP = smem + L::P_OFF;
  const uint32_t sP_u = smem_u32(sP);
  const uint8_t* mrow_base = drop_mask != nullptr ? drop_mask + (((long long)b * H + h) * N + qrow) * N : nullptr;

  for (int j = 0; j < nkv; ++j) {
    const int kvn = min(TILE, N - j * TILE);
    const uint32_t n_eff = roundup16(kvn);
    const int nchunks = (int)(n_eff + 31) / 32;
    mbar_wait(bar_s, j & 1);
    tc_fence_after();

    // the row (<= 128 scores) is read from TMEM once, two chunks per round trip
    uint32_t sv[4][32];
    float mx = m_run;
#pragma unroll
    for (int cb = 0; cb < 4; cb += 2) {
      if (cb < nchunks) {
        tmem_ld_32x32(tmem_s + lane_addr + cb * 32, sv[cb]);
        if (cb + 1 < nchunks) tmem_ld_32x32(tmem_s + lane_addr + (cb + 1) * 32, sv[cb + 1]);
        tmem_ld_wait();
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          const int c = cb + cc;
          if (c < nchunks) {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (c * 32 + i < kvn) mx = fmaxf(mx, __uint_as_float(sv[c][i]));
          }
        }
      }
    }
    const float alpha = ex2_approx((m_run - mx) * c2);  // 0 on the first tile (m_run = -inf)
    if (j > 0) {
      // P V_{j-1} has retired: its K / V stage takes tile j - 1 + FWDS_STAGES, P and O may be touched again
      mbar_wait(bar_o, (j - 1) & 1);
      tc_fence_after();
      if (threadIdx.x == 0 && j - 1 + FWDS_STAGES < nkv) load_kv(j - 1 + FWDS_STAGES);
      // O <- alpha * O before P V_j accumulates into it (only if some row of the warp raised its maximum)
      if (__any_sync(0xffffffffu, mx > m_run)) {
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          uint32_t o0[32];
          tmem_ld_32x32(tmem_o + lane_addr + hh * 32, o0);
          tmem_ld_wait();
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            uint32_t t16[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) t16[i] = __float_as_uint(__uint_as_float(o0[u * 16 + i]) * alpha);
            tmem_st_32x16(tmem_o + lane_addr + hh * 32 + u * 16, t16);
          }
        }
        if (WIDE) {
          uint32_t t16[16];
          tmem_ld_32x16(tmem_o + lane_addr + 64, t16);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i) t16[i] = __float_as_uint(__uint_as_float(t16[i]) * alpha);
          tmem_st_32x16(tmem_o + lane_addr + 64, t16);
        }
        tmem_st_wait();
      }
    }
    const float mc = mx * c2;
    float rowsum = 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      if (c < nchunks) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          if ((uint32_t)(c * 32 + g * 8) < n_eff) {
            float p[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float e = ex2_approx(fmaf(__uint_as_float(sv[c][g * 8 + i]), c2, -mc));
              p[i] = (c * 32 + g * 8 + i < kvn) ? e : 0.f;
            }
            uint4 u;
            u.x = pack_bf16x2(p[0], p[1]);
            u.y = pack_bf16x2(p[2], p[3]);
            u.z = pack_bf16x2(p[4], p[5]);
            u.w = pack_bf16x2(p[6], p[7]);
            // the row sum uses the bf16-rounded probabilities so that P*V and l stay consistent
            const float2 a0 = unpack_bf16x2(u.x), a1 = unpack_bf16x2(u.y), a2 = unpack_bf16x2(u.z), a3 = unpack_bf16x2(u.w);
            rowsum += ((a0.x + a0.y) + (a1.x + a1.y)) + ((a2.x + a2.y) + (a3.x + a3.y));
            if (mrow_base != nullptr) {   // the dropped, rescaled probabilities are what multiplies V
              const int col = j * TILE + c * 32 + g * 8;
              const uint8_t* mrow = mrow_base + col;
#pragma unroll
              for (int i = 0; i < 8; ++i) p[i] = (qrow < N && col + i < N && mrow[i]) ? p[i] * drop_scale : 0.f;
              u.x = pack_bf16x2(p[0], p[1]);
              u.y = pack_bf16x2(p[2], p[3]);
              u.z = pack_bf16x2(p[4], p[5]);
              u.w = pack_bf16x2(p[6], p[7]);
            }
            st_swz(sP, r, c * 4 + g, u);
          }
        }
      }
    }
    l_run = l_run * alpha + rowsum;
    m_run = mx;

    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
      const uint32_t idesc = umma_idesc(TILE, HDW, 1, false, true);  // A = P K-major, B = V MN-major (tail = second 64-wide chunk)
      const int ksteps = (int)n_eff / 16;
      const uint32_t sV_u = smem_u32(smem + L::KV_OFF + (j % FWDS_STAGES) * 2 * L::OPB + L::OPB);
      const uint64_t pdesc = umma_desc_kmajor(sP_u), vdesc = umma_desc_mnmajor(sV_u, TILE_BYTES);
      if (elect_one()) {
#pragma unroll 4
        for (int k = 0; k < ksteps; ++k)
          umma_bf16_ss(tmem_o, pdesc + (uint64_t)((k >> 2) * (TILE_BYTES >> 4) + (k & 3) * 2), vdesc + (uint64_t)(k * 128), idesc,
                       j > 0 || k > 0);
        umma_commit(bar_o);
      }
      __syncwarp();
      // every thread has S_j in registers: S_{j+1} runs behind P V_j
      if (j + 1 < nkv) issue_s(j + 1);
    }
  }

  mbar_wait(bar_o, (nkv - 1) & 1);
  tc_fence_after();
  {
    uint32_t a0[32], a1[32], t16[16];
    tmem_ld_32x32(tmem_o + lane_addr, a0);
    tmem_ld_32x32(tmem_o + lane_addr + 32, a1);
    if (WIDE) tmem_ld_32x16(tmem_o + lane_addr + 64, t16);
    tmem_ld_wait();
    if (qrow < N) {
      const float inv = 1.0f / l_run;
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        a0[i] = __float_as_uint(__uint_as_float(a0[i]) * inv);
        a1[i] = __float_as_uint(__uint_as_float(a1[i]) * inv);
      }
      __nv_bfloat16* orow = out + ((long long)b * N + qrow) * (H * hd) + h * hd;
      store_row_bf16_64(orow, a0, a1, hd);
      if (WIDE) {
#pragma unroll
        for (int i = 0; i < 16; ++i) t16[i] = __float_as_uint(__uint_as_float(t16[i]) * inv);
        store_row_bf16_tail(orow + 64, t16, hd - 64);
      }
      if (lse) lse[((long long)b * H + h) * N + qrow] = m_run * scale + __logf(l_run);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

template <bool WIDE>
int launch_fwd_stream(const CUtensorMap& tm, void* out, float* lse, int B, int N, int H, int hd, float scale, cudaStream_t s,
                      const uint8_t* drop_mask, float drop_scale) {
  using L = FwdStreamSmem<WIDE>;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(attn_fwd_stream_kernel<WIDE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L::BYTES);
    if (e != cudaSuccess) return vitk_set_error(VITK_ERR_CUDA, "attn_fwd_stream: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    attr_set = true;
  }
  dim3 grid((N + TILE - 1) / TILE, H, B);
  attn_fwd_stream_kernel<WIDE><<<grid, 128, L::BYTES, s>>>(tm, (__nv_bfloat16*)out, lse, N, H, hd, scale, drop_mask, drop_scale);
  return vitk_check_launch("attn_fwd_stream");
}

// The attention tensors are mapped for TMA as (head_dim, head slot, token, image): a [rows][64] box of one head slot
// arrives as a 128-byte-swizzled tile whose columns >= head_dim are zero-filled (and are clipped again on the way out),
// so head_dim < 64 (my_vit_mini: 48) runs on the same 64-wide tiles; the zero columns add nothing to Q K^T or dO V^T
// and produce zero columns of O / dQ / dK / dV.  A head wider than 64 (my_vit_xs: 72) takes a second box at column 64 (its
// tail tile: columns 64 .. 127, zero from head_dim on).  slots = 3 H for qkv / dqkv, H for out / dout.
int make_head_tmap(CUtensorMap* tm, const void* base, int slots, int hd, int N, int B, int box_rows) {
  return vitk_make_tmap_4d(tm, base, 2, (uint64_t)hd, (uint64_t)slots, (uint64_t)N, (uint64_t)B, (uint64_t)hd,
                           (uint64_t)slots * hd, (uint64_t)N * slots * hd, HD, 1, (uint32_t)box_rows, 1);
}

bool head_dim_ok(int hd) { return hd >= 16 && hd <= HDW_MAX && hd % 8 == 0; }
constexpr int WIDE_MAX_N = 2 * TILE;   // heads wider than 64 (my_vit_xs: N = 197) are built and tested up to 256 tokens

// The backward runs attn_bwd4 for the unmasked 128 < N <= 256 at head_dim <= 64 and the streaming kernel for every other call.
bool use_bwd4(int N, int hd, bool masked) { return N > TILE && N <= 2 * TILE && hd <= HD && !masked; }

// Columns per head of the fp32 dQ accumulator in the backward workspace, 0 when the call needs none: the streaming kernel
// red.adds dQ partials into it when it runs over more than one kv tile.
int dq32_pitch(int N, int hd, bool masked) { return N <= TILE || use_bwd4(N, hd, masked) ? 0 : (hd > HD ? HDW_MAX : HD); }

}  // namespace

static int attn_fwd_impl(const void* qkv, void* out, float* lse, int32_t B, int32_t N, int32_t H, int32_t head_dim, float scale,
                         const uint8_t* drop_mask, float drop_scale, void* stream) {
  VITK_REQUIRE(B > 0 && N > 0 && H > 0, VITK_ERR_SHAPE, "attn_fwd: bad shape B=%d N=%d H=%d", B, N, H);
  VITK_REQUIRE(head_dim_ok(head_dim), VITK_ERR_UNSUPPORTED, "attn_fwd: head_dim=%d (built for multiples of 8 in [16, 80])", head_dim);
  VITK_REQUIRE(N <= ATTN_MAX_N, VITK_ERR_UNSUPPORTED, "attn_fwd: N=%d > %d", N, ATTN_MAX_N);
  VITK_REQUIRE(head_dim <= HD || N <= WIDE_MAX_N, VITK_ERR_UNSUPPORTED, "attn_fwd: head_dim=%d > 64 is built for N <= %d (N=%d)",
               head_dim, WIDE_MAX_N, N);
  VITK_REQUIRE(((uintptr_t)qkv & 15) == 0 && ((uintptr_t)out & 15) == 0, VITK_ERR_ALIGN, "attn_fwd: unaligned");
  const int hd = head_dim;
  CUtensorMap tm, tm_out;
  int rc = make_head_tmap(&tm, qkv, 3 * H, hd, N, B, TILE);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  // the kv-streaming kernel for wide heads, a keep mask and N <= 128; attn_fwd4 (whole score row in TMEM, one thread per
  // row) for 128 < N <= 256; attn_fwd6 (kv loop, score MMA off the softmax's critical path) above that
  if (hd > HD) return launch_fwd_stream<true>(tm, out, lse, B, N, H, hd, scale, s, drop_mask, drop_scale);
  if (drop_mask != nullptr || N <= TILE) return launch_fwd_stream<false>(tm, out, lse, B, N, H, hd, scale, s, drop_mask, drop_scale);
  rc = make_head_tmap(&tm_out, out, H, hd, N, B, TILE);
  if (rc) return rc;
  if (N <= 2 * TILE) return launch_fwd4(tm, tm_out, lse, B, N, H, scale, s);
  return launch_fwd6(tm, tm_out, lse, B, N, H, scale, s);
}

extern "C" int vitk_attn_fwd(const void* qkv, void* out, float* lse, int32_t B, int32_t N, int32_t H, int32_t head_dim,
                             float scale, void* stream) {
  return attn_fwd_impl(qkv, out, lse, B, N, H, head_dim, scale, nullptr, 1.f, stream);
}

extern "C" int vitk_attn_fwd_dropout(const void* qkv, void* out, float* lse, const uint8_t* keep_mask, float keep_scale, int32_t B,
                                     int32_t N, int32_t H, int32_t head_dim, float scale, void* stream) {
  VITK_REQUIRE(keep_mask != nullptr && keep_scale > 0.f, VITK_ERR_SHAPE, "attn_fwd_dropout: keep mask [B, H, N, N] and 1 / (1 - p) required");
  return attn_fwd_impl(qkv, out, lse, B, N, H, head_dim, scale, keep_mask, keep_scale, stream);
}

extern "C" void vitk_debug_set_trace(long long* device_buf) { g_trace_buf = device_buf; }

static int64_t dsum_bytes(int32_t B, int32_t N, int32_t H) {
  return (((int64_t)B * H * N * (int64_t)sizeof(float)) + 255) / 256 * 256;
}

// D = rowsum(O * dO) [B, H, N] fp32, plus the fp32 dQ accumulator [B, N, H, dq32_pitch] (heads padded to the tile width)
extern "C" int64_t vitk_attn_bwd_workspace_bytes(int32_t B, int32_t N, int32_t H, int32_t head_dim) {
  return dsum_bytes(B, N, H) + (int64_t)B * N * H * dq32_pitch(N, head_dim, false) * (int64_t)sizeof(float);
}

extern "C" int64_t vitk_attn_bwd_dropout_workspace_bytes(int32_t B, int32_t N, int32_t H, int32_t head_dim) {
  return dsum_bytes(B, N, H) + (int64_t)B * N * H * dq32_pitch(N, head_dim, true) * (int64_t)sizeof(float);
}

static int attn_bwd_impl(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv, void* workspace, int32_t B,
                         int32_t N, int32_t H, int32_t head_dim, float scale, const uint8_t* drop_mask, float drop_scale,
                         void* stream) {
  VITK_REQUIRE(B > 0 && N > 0 && H > 0, VITK_ERR_SHAPE, "attn_bwd: bad shape B=%d N=%d H=%d", B, N, H);
  VITK_REQUIRE(head_dim_ok(head_dim), VITK_ERR_UNSUPPORTED, "attn_bwd: head_dim=%d (built for multiples of 8 in [16, 80])", head_dim);
  VITK_REQUIRE(N <= ATTN_MAX_N, VITK_ERR_UNSUPPORTED, "attn_bwd: N=%d > %d", N, ATTN_MAX_N);
  VITK_REQUIRE(head_dim <= HD || N <= WIDE_MAX_N, VITK_ERR_UNSUPPORTED, "attn_bwd: head_dim=%d > 64 is built for N <= %d (N=%d)",
               head_dim, WIDE_MAX_N, N);
  VITK_REQUIRE(((uintptr_t)qkv & 15) == 0 && ((uintptr_t)out & 15) == 0 && ((uintptr_t)dout & 15) == 0 && ((uintptr_t)dqkv & 15) == 0,
               VITK_ERR_ALIGN, "attn_bwd: unaligned");
  const int hd = head_dim;
  CUtensorMap tm_qkv, tm_do;
  int rc = make_head_tmap(&tm_qkv, qkv, 3 * H, hd, N, B, TILE);
  if (rc) return rc;
  rc = make_head_tmap(&tm_do, dout, H, hd, N, B, TILE);
  if (rc) return rc;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(attn_bwd4_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Bwd3Smem::BYTES);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(attn_bwd_stream_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BwdStreamSmem<false>::BYTES);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(attn_bwd_stream_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BwdStreamSmem<true>::BYTES);
    if (e != cudaSuccess) return vitk_set_error(VITK_ERR_CUDA, "attn_bwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    attr_set = true;
  }
  cudaStream_t st = (cudaStream_t)stream;
  VITK_REQUIRE(workspace != nullptr && ((uintptr_t)workspace & 15) == 0, VITK_ERR_ALIGN,
               "attn_bwd: needs a 16-byte aligned workspace of vitk_attn_bwd_workspace_bytes()");
  float* dsum = reinterpret_cast<float*>(workspace);
  const long long rows = (long long)B * N;
  attn_dsum_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>((const __nv_bfloat16*)out, (const __nv_bfloat16*)dout, dsum, rows,
                                                               N, H, hd);
  rc = vitk_check_launch("attn_dsum");
  if (rc) return rc;
  if (use_bwd4(N, hd, drop_mask != nullptr)) {
    const int items = B * H;
    const int g3 = items < vitk_num_sms() ? items : vitk_num_sms();
    CUtensorMap tm_dqkv;   // 32-row boxes: one per warp-level read-out of dQ / dK / dV
    rc = make_head_tmap(&tm_dqkv, dqkv, 3 * H, hd, N, B, 32);
    if (rc) return rc;
    attn_bwd4_kernel<<<g3, BWD3_THREADS, Bwd3Smem::BYTES, st>>>(tm_qkv, tm_do, tm_dqkv, dsum, lse, B, N, H, scale, g_trace_buf);
    return vitk_check_launch("attn_bwd4");
  }
  // one CTA per (b, h, kv tile); over more than one kv tile the dQ partials are red.add'ed into the fp32 workspace (156 of
  // the ~820 us per layer at ViT-L/384, B = 64, H = 16, N = 577; ~90 us are the memset / cast / D kernels around it)
  const int pitch = dq32_pitch(N, hd, drop_mask != nullptr);
  float* dq32 = nullptr;
  if (pitch > 0) {
    dq32 = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(workspace) + dsum_bytes(B, N, H));
    cudaError_t e = cudaMemsetAsync(dq32, 0, (size_t)rows * H * pitch * sizeof(float), st);
    if (e != cudaSuccess) return vitk_set_error(VITK_ERR_CUDA, "attn_bwd: memset: %s", cudaGetErrorString(e));
  }
  dim3 grid((N + TILE - 1) / TILE, H, B);
  if (hd > HD)
    attn_bwd_stream_kernel<true><<<grid, 128, BwdStreamSmem<true>::BYTES, st>>>(tm_qkv, tm_do, dsum, lse, (__nv_bfloat16*)dqkv, dq32,
                                                                                N, H, hd, scale, drop_mask, drop_scale);
  else
    attn_bwd_stream_kernel<false><<<grid, 128, BwdStreamSmem<false>::BYTES, st>>>(tm_qkv, tm_do, dsum, lse, (__nv_bfloat16*)dqkv,
                                                                                  dq32, N, H, hd, scale, drop_mask, drop_scale);
  rc = vitk_check_launch("attn_bwd_stream");
  if (rc || pitch == 0) return rc;
  const long long n8 = rows * H * (hd / 8);
  dq_cast_kernel<<<(unsigned)((n8 + 255) / 256), 256, 0, st>>>(dq32, (__nv_bfloat16*)dqkv, rows, H, hd, pitch);
  return vitk_check_launch("attn_bwd_dq_cast");
}

extern "C" int vitk_attn_bwd(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv,
                             void* workspace, int32_t B, int32_t N, int32_t H, int32_t head_dim, float scale,
                             void* stream) {
  return attn_bwd_impl(qkv, out, dout, lse, dqkv, workspace, B, N, H, head_dim, scale, nullptr, 1.f, stream);
}

extern "C" int vitk_attn_bwd_dropout(const void* qkv, const void* out, const void* dout, const float* lse, void* dqkv,
                                     void* workspace, const uint8_t* keep_mask, float keep_scale, int32_t B, int32_t N, int32_t H,
                                     int32_t head_dim, float scale, void* stream) {
  VITK_REQUIRE(keep_mask != nullptr && keep_scale > 0.f, VITK_ERR_SHAPE, "attn_bwd_dropout: keep mask [B, H, N, N] and 1 / (1 - p) required");
  return attn_bwd_impl(qkv, out, dout, lse, dqkv, workspace, B, N, H, head_dim, scale, keep_mask, keep_scale, stream);
}
