// Shared pieces of the fused ViT attention (reference: Attention.forward, vit.py:116-122): problem geometry, kernel
// parameters, the 3-D TMA view of the QKV GEMM's [B*192, 3*H*80] fp16 output (16 dims x 192 tokens x 5 chunks, 32B
// swizzle) and the launch plan.  The kernel itself is attention3_tcgen05.cuh (two tile chains per CTA, S / P / O in TMEM);
// the first two generations (P through shared memory; single chain with P in TMEM) were removed in round 2 after losing
// their A/B (round-1 numbers: DESIGN.md section 9).
#pragma once
#include "common.cuh"
#include "ptx.cuh"

namespace thmr {

constexpr int kAttTokens = 192;
constexpr int kAttHeadDim = 80;
constexpr int kAttChunks = kAttHeadDim / 16;                     // 16-element (32 B) K-chunks
constexpr uint32_t kAttChunkBytes = kAttTokens * 32;             // 6144
constexpr uint32_t kAttMatBytes = kAttChunks * kAttChunkBytes;   // 30720 (one of Q / K / V)
constexpr uint32_t kAttWideBytes = kAttTokens * 128;             // 24576: the [192 x 64] SWIZZLE_128B block of Q / K

struct AttnParams {
  int num_problems;  // B * H
  int heads;
  float scale_log2e; // head_dim^-0.5 * log2(e)
  __half* out;       // [B*192, ldo], head h at columns [80 h, 80 h + 80)
  int ldo;
  float* dbg_s;      // optional [B*H, 192, 192] raw scores (tests only)
  unsigned long long* stamp;   // in-graph start stamp (nullable)
};

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// 3-D view of the QKV activation [rows, 3*H*80] fp16 as (16 elements, rows, chunks of 16 columns).
inline int make_tmap_qkv(CUtensorMap* out, const void* qkv, uint64_t rows, uint64_t ld) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return fail(THMR_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
  THMR_CHECK((reinterpret_cast<uintptr_t>(qkv) & 15) == 0 && ld % 16 == 0, "attention: qkv pointer/pitch alignment");
  cuuint64_t gdim[3] = {16, rows, ld / 16};
  cuuint64_t gstr[2] = {ld * 2, 32};
  cuuint32_t box[3] = {16, static_cast<cuuint32_t>(kAttTokens), static_cast<cuuint32_t>(kAttChunks)};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(qkv), gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(THMR_ERR_CUDA, "cuTensorMapEncodeTiled(qkv) failed (%d)", (int)r);
  return THMR_OK;
}

struct AttnPlan {
  CUtensorMap tm_qk64;  // Q / K: [192 rows x 64 columns] boxes, 128-byte rows, SWIZZLE_128B (dims 0..63 of a head)
  CUtensorMap tm_qk16;  // Q / K: [192 rows x 16 columns] boxes, SWIZZLE_32B (dims 64..79)
  CUtensorMap tm;       // V: the 3-D five-chunk view (make_tmap_qkv)
  CUtensorMap tm_out;   // [B*192, H*80] fp16 output, 32-row x 80-column boxes (third-generation kernel)
  AttnParams p;
  int grid;
};

inline int attention_make_plan(const __half* qkv, int ld_qkv, int B, int heads, __half* out, int ldo, float* dbg_s,
                               AttnPlan* plan) {
  THMR_CHECK(B > 0 && heads > 0, "attention: bad shape");
  THMR_CHECK(ld_qkv >= 3 * heads * kAttHeadDim, "attention: qkv pitch %d < %d", ld_qkv, 3 * heads * kAttHeadDim);
  THMR_CHECK(ldo % 8 == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0, "attention: output alignment");
  THMR_TRY(make_tmap_qkv(&plan->tm, qkv, static_cast<uint64_t>(B) * kAttTokens, ld_qkv));
  THMR_TRY(make_tmap_2d_f16(&plan->tm_qk64, qkv, static_cast<uint64_t>(B) * kAttTokens, static_cast<uint64_t>(ld_qkv), ld_qkv,
                            kAttTokens, 64, CU_TENSOR_MAP_SWIZZLE_128B));
  THMR_TRY(make_tmap_2d_f16(&plan->tm_qk16, qkv, static_cast<uint64_t>(B) * kAttTokens, static_cast<uint64_t>(ld_qkv), ld_qkv,
                            kAttTokens, 16, CU_TENSOR_MAP_SWIZZLE_32B));
  THMR_TRY(make_tmap_2d_f16(&plan->tm_out, out, static_cast<uint64_t>(B) * kAttTokens,
                            static_cast<uint64_t>(heads) * kAttHeadDim, ldo, 32, kAttHeadDim, CU_TENSOR_MAP_SWIZZLE_NONE));
  plan->p.num_problems = B * heads;
  plan->p.heads = heads;
  plan->p.scale_log2e = 1.4426950408889634f / sqrtf(static_cast<float>(kAttHeadDim));
  plan->p.out = out;
  plan->p.ldo = ldo;
  plan->p.dbg_s = dbg_s;
  plan->p.stamp = nullptr;
  plan->grid = plan->p.num_problems < num_sms() ? plan->p.num_problems : num_sms();
  return THMR_OK;
}


}  // namespace thmr
