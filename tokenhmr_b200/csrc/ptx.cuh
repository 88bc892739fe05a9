// Thin inline-PTX wrappers for the sm_100a features the engine uses:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld / fences).
// Everything here is sm_100a-only; there is no fallback path.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace thmr {

// Every mbarrier spin is bounded: a wedged pipeline sets this flag and falls
// through (the kernel finishes with garbage and the host reports an error)
// instead of hanging the GPU box.
__device__ unsigned int g_pipeline_timeout = 0;  // single translation unit (tokenhmr_b200.cu)
constexpr uint32_t kSpinLimit = 1u << 24;

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t lane_id() {
  uint32_t l;
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(l));
  return l;
}

// One lane of a converged warp.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xFFFFFFFF;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// Make generic-proxy smem writes visible to the async proxy (TMA / tcgen05.mma operand reads).
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Non-blocking probe (no hardware suspend window, unlike try_wait): for pollers that multiplex several barriers.
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait; returns false (and raises the global flag) on timeout.
__device__ __forceinline__ bool mbar_wait(uint64_t* bar, uint32_t parity) {
#pragma unroll 1   // the compiler otherwise unrolls every spin loop x4: pure instruction-cache pressure
  for (uint32_t it = 0; it < kSpinLimit; ++it) {
    if (mbar_try_wait(bar, parity)) return true;
  }
  atomicExch(&g_pipeline_timeout, 1u);
  return false;
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2D tiled load global -> shared, completion on an mbarrier (complete_tx bytes).
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int32_t c0,
                                            int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int32_t c0,
                                            int32_t c1, int32_t c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1),
        "r"(c2)
      : "memory");
}
// 2D tiled store shared -> global (bulk group completion).
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(uint32_t* p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ---------------------------------------------------------------- packed fp32 (fma.rn.f32x2 = SASS FFMA2, IEEE per lane)
__device__ __forceinline__ uint64_t f2_pack(float a, float b) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void f2_unpack(uint64_t v, float& a, float& b) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ uint64_t f2_mul(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t f2_add(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t f2_splat(float c) { return f2_pack(c, c); }

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// Whole-warp: allocate `ncols` (power of two >= 32) TMEM columns; base address lands in *smem_slot.
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// D[tmem] (+)= A[smem] * B[smem]; one thread issues for the CTA. kind::f16 (fp16/bf16 in, fp32 accumulate).
__device__ __forceinline__ void umma_f16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// A operand from TMEM (e.g. softmax probabilities), B from smem.
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed.
// (Implies tcgen05.fence::before_thread_sync.)
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// TMEM -> registers. 32x32b: thread t of the warp reads lane (base_lane + t), N consecutive 32-bit columns.
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Orders later uses of v[] after a preceding tcgen05.wait::ld when loads are software-pipelined (the compiler
// sees no data dependence between the wait and the registers an earlier tcgen05.ld filled).
template <int N>
__device__ __forceinline__ void tmem_pin(uint32_t (&v)[N]) {
#pragma unroll
  for (int e = 0; e < N; ++e) asm volatile("" : "+r"(v[e]));
}

// registers -> TMEM (32x32b, 16 columns): thread t writes lane (base_lane + t).
__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      :
      : "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_x8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               :
               : "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- UMMA descriptors
// Shared-memory matrix descriptor (sm_100 "version 1"), see DESIGN.md §kernels:
//   [0,14)  start address >> 4      [16,30) leading byte offset >> 4
//   [32,46) stride byte offset >> 4 [46,48) version = 1
//   [61,64) layout: 0 none, 2 SWIZZLE_128B, 4 SWIZZLE_64B, 6 SWIZZLE_32B
enum : uint32_t { kSwzNone = 0, kSwz128 = 2, kSwz64 = 4, kSwz32 = 6 };

__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                                   uint32_t layout) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(layout & 7) << 61;
  return d;
}

// Instruction descriptor for kind::f16: fp16 (0) or bf16 (1) operands, fp32 accumulate.
//   [4,6) D fmt (1 = f32)  [7,10) A fmt  [10,13) B fmt  [15] A major (0 = K)  [16] B major (0 = K)
//   [17,23) N >> 3         [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc_f16(uint32_t M, uint32_t N, uint32_t a_mn_major = 0,
                                                      uint32_t b_mn_major = 0, uint32_t fmt = 0) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | (a_mn_major << 15) | (b_mn_major << 16) | ((N >> 3) << 17) |
         ((M >> 4) << 24);
}

}  // namespace thmr

// ================================================================================================
// CTA-pair (cta_group::2) variants: two CTAs of a cluster issue one UMMA of M = 256 together.
// ================================================================================================
namespace thmr {

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release;\n\tbarrier.cluster.wait.acquire;" ::: "memory");
}
// Shared-window addresses of the two CTAs of a pair differ in bit 24; clearing it addresses CTA 0 (the MMA leader).
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;

// TMA load issued by either CTA of the pair into ITS OWN smem; the transaction bytes are credited to the
// leader CTA's mbarrier (same offset, peer bit cleared).
__device__ __forceinline__ void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int32_t c0,
                                                int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0),
        "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t* smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2sm() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_f16_ss_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive (once the issued MMAs retire) on the barrier at this offset in every CTA of `cta_mask`.
__device__ __forceinline__ void umma_commit_2sm_mcast(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}
// Arrive on the barrier at the same offset in CTA `cta` of the cluster.
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t cta) {
  asm volatile(
      "{\n\t"
      ".reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(cta)
      : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ bool mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
#pragma unroll 1
  for (uint32_t it = 0; it < kSpinLimit; ++it) {
    if (mbar_try_wait_cluster(bar, parity)) return true;
  }
  atomicExch(&g_pipeline_timeout, 1u);
  return false;
}

}  // namespace thmr
