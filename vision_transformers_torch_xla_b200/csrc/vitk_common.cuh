// vitk_common.cuh — shared device/host helpers for the vitk sm_100a kernel library.
//
// Everything here is a thin wrapper around one PTX instruction (mbarrier, TMA,
// tcgen05/TMEM) or a host-side utility (error slot, tensor-map encoding).  No
// CUTLASS/CuTe is used: kernels in this library are written directly against
// the sm_100a ISA.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

// ----------------------------------------------------------------------------
// Host side: error reporting across the C ABI (see include/vitk.h)
// ----------------------------------------------------------------------------
enum VitkStatus : int {
  VITK_OK = 0,
  VITK_ERR_SHAPE = -1,
  VITK_ERR_ALIGN = -2,
  VITK_ERR_DTYPE = -3,
  VITK_ERR_CUDA = -4,
  VITK_ERR_DRIVER = -5,
  VITK_ERR_UNSUPPORTED = -6,
};

int vitk_set_error(int code, const char* fmt, ...);
int vitk_check_launch(const char* what);

#define VITK_REQUIRE(cond, code, ...)                   \
  do {                                                  \
    if (!(cond)) return vitk_set_error(code, __VA_ARGS__); \
  } while (0)

// A pointer that a kernel loads or stores as BYTES-wide vectors must be BYTES-aligned (NULL passes).  Entry points check
// these first, ahead of the shape checks and of any early return on an empty problem.
#define VITK_REQUIRE_ALIGNED(fn, name, ptr, bytes)                                                  \
  VITK_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & ((bytes) - 1)) == 0, VITK_ERR_ALIGN, \
               fn ": " name " must be %d-byte aligned", (int)(bytes))

// Encode a 2-D bf16/f32 tiled tensor map with 128-byte swizzle.
//   inner = contiguous dimension (elements), outer = rows, ld = row pitch in elements.
int vitk_make_tmap_2d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t inner,
                      uint64_t outer, uint64_t ld_elems, uint32_t box_inner, uint32_t box_outer);
int vitk_make_tmap_3d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t d0, uint64_t d1,
                      uint64_t d2, uint64_t ld1_elems, uint64_t ld2_elems, uint32_t b0, uint32_t b1,
                      uint32_t b2);
int vitk_make_tmap_4d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t d3,
                      uint64_t ld1_elems, uint64_t ld2_elems, uint64_t ld3_elems, uint32_t b0, uint32_t b1, uint32_t b2,
                      uint32_t b3, int swizzle_bytes = 128);
int vitk_make_tmap_2d_sw64(CUtensorMap* out, const void* base, int elem_bytes, uint64_t inner, uint64_t outer,
                           uint64_t ld_elems, uint32_t box_inner, uint32_t box_outer);
int vitk_num_sms();

// ----------------------------------------------------------------------------
// Device side
// ----------------------------------------------------------------------------
#ifdef __CUDACC__

namespace vitk {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n"
      ".reg .b32 rx;\n"
      ".reg .pred px;\n"
      "elect.sync rx|px, 0xffffffff;\n"
      "selp.b32 %0, 1, 0, px;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---- mbarrier ----------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  // make generic-proxy smem writes visible to the async proxy (TMA / tcgen05 operand reads)
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// non-blocking: has the phase with this parity completed?  (any lane seeing it is enough: completion is monotonic)
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.b32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return __any_sync(0xffffffffu, ok != 0);
}

// ---- TMA -----------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int32_t c0, int32_t c1, int32_t c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// 4-D tile load with the innermost coordinate fixed at 0: the attention tensors are mapped as (head_dim, head slot,
// token, image), so a [128 tokens][64] box of head slot `c1` comes in with the columns >= head_dim zero-filled
__device__ __forceinline__ void tma_load_head(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                              int32_t c1, int32_t c2, int32_t c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
// the same box at inner (head_dim) coordinate c0: the columns 64 .. of a head wider than one 64-column tile
__device__ __forceinline__ void tma_load_head_col(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int32_t c0,
                                                  int32_t c1, int32_t c2, int32_t c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int32_t c0, int32_t c1, int32_t c2, int32_t c3,
                                            int32_t c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3),
      "r"(c4)
      : "memory");
}

// smem tile -> global (bulk async group); rows / columns outside the tensor are clipped
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, const void* smem_src, int32_t c0, int32_t c1, int32_t c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
// the store counterpart of tma_load_head: columns >= head_dim and rows >= N are clipped
__device__ __forceinline__ void tma_store_head(const CUtensorMap* m, const void* smem_src, int32_t c1, int32_t c2, int32_t c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(smem_src)), "r"(0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// commit the stores issued so far and wait until their smem source has been read (it may then be overwritten)
__device__ __forceinline__ void tma_store_commit_and_wait_read() {
  asm volatile("cp.async.bulk.commit_group;\n\tcp.async.bulk.wait_group.read 0;" ::: "memory");
}

// ---- tcgen05 / TMEM --------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_slot)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem], bf16 inputs, fp32 accumulate.  One thread issues.
__device__ __forceinline__ void umma_bf16_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                             uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]: A is read from tensor memory (128 lanes = M rows, two bf16 K-elements per 32-bit
// column, K-major only), e.g. bf16 probabilities written back over the fp32 scores they came from.
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// tf32 variant (fp32 operands in smem, UMMA_K = 8)
__device__ __forceinline__ void umma_tf32_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                             uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread retire.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// 32 lanes x 32 consecutive 32-bit columns: thread i of the warp gets lane (base_lane+i).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}

__device__ __forceinline__ void tmem_ld_32x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
// registers -> TMEM, 32 lanes x 8 consecutive 32-bit columns (mirror of tmem_ld_32x8)
__device__ __forceinline__ void tmem_st_32x8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---- CTA-pair (cta_group::2) variants -------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.aligned;\n\tbarrier.cluster.wait.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t* smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2cta() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A * B with M = 256 split over the CTA pair; issued by the leader CTA only.
__device__ __forceinline__ void umma_bf16_ss_2cta(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                  uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive (once the prior MMAs retire) on the barrier at the same smem offset in every CTA of `cta_mask`.
__device__ __forceinline__ void umma_commit_2cta_mc(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}
// TMA load whose completion bytes are credited to the barrier at address `bar_addr` (a shared::cluster address;
// clearing bit 24 of a CTA-local address names the same offset in the even CTA of the pair).
__device__ __forceinline__ void tma_load_2d_2cta(void* smem_dst, const CUtensorMap* m, uint32_t bar_addr, int32_t c0,
                                                 int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_addr), "r"(c0), "r"(c1)
      : "memory");
}
// 4-D tile loads (the patch view of an NCHW image: vitk_gemm.cu), plain and crediting the pair leader's barrier
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int32_t c0, int32_t c1,
                                            int32_t c2, int32_t c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_2cta(void* smem_dst, const CUtensorMap* m, uint32_t bar_addr, int32_t c0,
                                                 int32_t c1, int32_t c2, int32_t c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_addr), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta) {
  asm volatile(
      "{\n"
      ".reg .b32 ra;\n"
      "mapa.shared::cluster.u32 ra, %0, %1;\n"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(cta)
      : "memory");
}

// ---- UMMA descriptors ---------------------------------------------------------------
// Shared-memory matrix descriptor (sm_100 "version 1"), 128-byte swizzle.
//   bits [0,14)  start address >> 4          bits [16,30) leading byte offset >> 4
//   bits [32,46) stride byte offset >> 4     bits [46,48) version = 1
//   bits [61,64) layout type (2 = SWIZZLE_128B, 4 = SWIZZLE_64B, 6 = SWIZZLE_32B, 0 = none)
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t saddr, uint32_t lbo_bytes,
                                                   uint32_t sbo_bytes, uint32_t layout_type = 2) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(layout_type) << 61;
  return d;
}
// 32-byte-swizzle operand tiles (the patch view of an image, vitk_gemm.cu): 8-row atoms of [8 rows][32 B] (256 B).
//   K-major : rows of 16 bf16 (one k-step); atoms of consecutive 8-row groups `sbo_bytes` apart
//   MN-major: k-rows of 16 bf16 along MN; 16-wide MN chunks `lbo_bytes` apart, 8-k-row groups `sbo_bytes` apart
__device__ __forceinline__ uint64_t umma_desc_kmajor_sw32(uint32_t saddr, uint32_t sbo_bytes) {
  return umma_smem_desc(saddr, 16, sbo_bytes, 6);
}
__device__ __forceinline__ uint64_t umma_desc_mnmajor_sw32(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return umma_smem_desc(saddr, lbo_bytes, sbo_bytes, 6);
}
// K-major operand tile: [rows][64 bf16] rows of 128 B, 8-row swizzle atoms of 1024 B.
__device__ __forceinline__ uint64_t umma_desc_kmajor(uint32_t saddr) {
  return umma_smem_desc(saddr, 0, 1024);
}
// MN-major operand tile: [mn/64 chunks][k rows][64 bf16]; chunk pitch = k_rows * 128 B.
__device__ __forceinline__ uint64_t umma_desc_mnmajor(uint32_t saddr, uint32_t chunk_pitch_bytes) {
  return umma_smem_desc(saddr, chunk_pitch_bytes, 1024);
}

// Instruction descriptor for kind::f16 / kind::tf32 with fp32 accumulation.
//   ab_format: 0 = f16, 1 = bf16, 2 = tf32
__host__ __device__ constexpr uint32_t umma_idesc(uint32_t M, uint32_t N, uint32_t ab_format,
                                                  bool a_mn_major, bool b_mn_major) {
  return (1u << 4)                                  // c_format = F32
         | (ab_format << 7) | (ab_format << 10)     // a_format, b_format
         | ((a_mn_major ? 1u : 0u) << 15) | ((b_mn_major ? 1u : 0u) << 16) |
         ((N >> 3) << 17) | ((M >> 4) << 24);
}

// ---- small numeric helpers ------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float2 unpack_bf16x2(uint32_t u) {
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(v);
}

__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// Exact-erf GELU and its derivative: gelu(h) = h Phi(h), gelu'(h) = Phi(h) + h phi(h).
// Phi(h) = 0.5*(1+erf(h/sqrt2)) via Abramowitz-Stegun 7.1.26 (|erf err| < 1.5e-7) evaluated as
//   Phi(-|h|) = 0.5*erfc(|h|/sqrt2) = t*(a1+t*(a2+t*(a3+t*(a4+t*a5))))*exp(-h^2/2),  t = 1/(1 + p*|h|/sqrt2)
// with the 0.5 folded into the coefficients, one MUFU.RCP + one MUFU.EX2; exp(-h^2/2) is shared with the density.
__device__ __forceinline__ void gelu_fwd_bwd(float h, float& act, float& deriv) {
  const float t = rcp_approx(fmaf(fabsf(h), 0.3275911f * 0.70710678118654752f, 1.0f));
  const float e = ex2_approx(h * h * (-0.5f * 1.4426950408889634f));
  float poly = fmaf(t, 0.5f * 1.061405429f, 0.5f * -1.453152027f);
  poly = fmaf(poly, t, 0.5f * 1.421413741f);
  poly = fmaf(poly, t, 0.5f * -0.284496736f);
  poly = fmaf(poly, t, 0.5f * 0.254829592f);
  const float q = poly * t * e;
  const float cdf = h > 0.f ? 1.0f - q : q;
  act = h * cdf;
  deriv = fmaf(h, e * 0.3989422804014327f, cdf);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace vitk

#endif  // __CUDACC__
