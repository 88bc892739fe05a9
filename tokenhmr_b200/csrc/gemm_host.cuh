// Host side of the tcgen05 GEMM: plan construction (TMA descriptors, tile choice) and launch.
#pragma once
#include "common.cuh"

#include "gemm2_tcgen05.cuh"
#include "gemm_tcgen05.cuh"

namespace thmr {

struct GemmPlan {
  CUtensorMap tmA, tmB, tmC;
  GemmParams p;
  int bn;
  int epi;
  int grid;
  int two_cta;  // CTA-pair kernel (256 x 256 tiles)
};

struct GemmDesc {
  const __half* A; int lda; long long a_rows;  // a_rows: rows addressable through the A descriptor
  const __half* B; int ldb;
  int M, N, K;
  const float* bias = nullptr;
  const float* resid = nullptr; int ldr = 0; int resid_mod = 0;
  int act = kActNone; int act32 = 0;
  float* out32 = nullptr; int ld32 = 0;
  __half* out16 = nullptr; int ld16 = 0;
  // implicit conv1d (taps > 1): K = taps * cin, tap t reads A rows (m + tap_row0 + t*tap_stride), cols [0,cin)
  int taps = 1; int cin = 0; int tap_row0 = 0; int tap_stride = 0;
  int seq_pitch = 0, seq_lo = 0, seq_hi = 0;
  float alpha = 1.0f;
  long long* argmin_out = nullptr; const float* row_sq = nullptr; const float* col_sq = nullptr;
  // screened arg-min (GemmParams): pass 1 queues uncertain rows, the exact pass takes its row count from the device
  int* screen_rows = nullptr; int* screen_count = nullptr; const float* screen_cmax2 = nullptr;
  float screen_rel = 0.f, screen_abs = 0.f; int screen_row0 = 0;
  const int* row_map = nullptr; const int* m_dev = nullptr; int m_dev_off = 0;
  int force_bn = 0;      // 512: the CTA-pair kernel whatever the shape (needs a TMA epilogue)
  bool no_2cta = false;  // never use the CTA-pair kernel
  unsigned int* sk_flags = nullptr;  // >= gemm_sk_flag_count(M, N) zeroed uints: enables stream-K for reduce-add GEMMs
  unsigned long long* stamp = nullptr;   // in-graph start stamp slot (nullable)
};

// Flags a stream-K GEMM of this shape needs (4 per 256 x 256 tile); the buffer must be zero before the first launch and
// is left zero by every launch, so consecutive GEMMs of one stream can share it.
inline size_t gemm_sk_flag_count(long long M, long long N) {
  return static_cast<size_t>((M + 255) / 256) * ((N + kG2BN - 1) / kG2BN) * 4;
}

// Ordering flags for stream-K GEMMs launched through the stand-alone C entry points (the engine carves its own out of
// the caller's workspace): one lazily grown, zero-initialised buffer per device.  Launches that use it must be
// stream-ordered with respect to each other (single-stream use of thmr_gemm_f16, as in the tests).
inline unsigned int* default_sk_flags(size_t count) {
  static unsigned int* buf[16] = {nullptr};
  static size_t cap[16] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) return nullptr;
  if (count > cap[dev]) {
    unsigned int* nb = nullptr;
    const size_t n = count < 4096 ? 4096 : count;
    if (cudaMalloc(&nb, n * sizeof(unsigned int)) != cudaSuccess || cudaMemset(nb, 0, n * sizeof(unsigned int)) != cudaSuccess) {
      cudaGetLastError();
      return nullptr;      // (e.g. called under stream capture): the GEMM falls back to whole tiles
    }
    buf[dev] = nb;         // the old buffer may still be referenced by earlier plans: intentionally not freed
    cap[dev] = n;
  }
  return buf[dev];
}

// Which epilogue can serve this GEMM (see gemm_tcgen05.cuh).
inline int pick_epi(const GemmDesc& d) {
  const bool plain = !d.argmin_out && d.seq_pitch == 0 && d.resid_mod == 0 && !d.act32 && d.N % 4 == 0 &&
                     d.M >= kGemmBM && (!d.bias || (reinterpret_cast<uintptr_t>(d.bias) & 15) == 0);
  if (!plain) return kEpiGeneric;
  if (d.out16 && !d.out32 && !d.resid && d.ld16 % 8 == 0 && d.N % 8 == 0 && d.alpha == 1.0f) return kEpiStore16;
  if (d.out32 && !d.out16 && d.resid == d.out32 && d.ldr == d.ld32 && d.act == kActNone && d.ld32 % 4 == 0)
    return kEpiAdd32;      // alpha * acc + bias reduce-added into the output
  if (d.out32 && !d.out16 && !d.resid && d.act == kActNone && d.ld32 % 4 == 0) return kEpiStore32;
  return kEpiGeneric;
}

// Tile width: the main loop is L2-feed bound (every k-block moves (128 + BN) * 128 bytes for 128 * BN * 64 MACs),
// so wide tiles win unless they leave SMs idle.  Cost model per k-block in cycles: max(MMA, L2 feed at ~40 B/clk/SM).
inline int pick_bn(int M, int N, int force, int epi) {
  if (force) return force;
  const int sms = num_sms();
  const int tm = (M + kGemmBM - 1) / kGemmBM;
  int best = 256;
  double best_cost = -1;
  const int cands[4] = {256, 128, 64, 32};
  for (int i = 0; i < 4; ++i) {
    const int bn = cands[i];
    if (epi != kEpiGeneric && bn < 128) continue;
    const long tiles = static_cast<long>(tm) * ((N + bn - 1) / bn);
    const long waves = (tiles + sms - 1) / sms;
    const double mma = 2.0 * bn;
    const double feed = (128.0 + bn) * 128.0 / 40.0;
    const double cost = waves * ((mma > feed ? mma : feed) + 40.0);
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = bn; }
  }
  return best;
}

inline int gemm_make_plan(const GemmDesc& d, GemmPlan* plan) {
  THMR_CHECK(d.M > 0 && d.N > 0 && d.K > 0, "gemm: bad shape %dx%dx%d", d.M, d.N, d.K);
  THMR_CHECK(d.out32 || d.out16 || d.argmin_out, "gemm: no output");
  int epi = pick_epi(d);
  if (d.force_bn && d.force_bn < 128) epi = kEpiGeneric;
  THMR_CHECK(d.force_bn != 512 || epi != kEpiGeneric, "gemm: block_n 512 (CTA pair) needs a TMA-epilogue eligible call");
  const int bn = pick_bn(d.M, d.N, d.force_bn == 512 ? 0 : d.force_bn, epi);
  THMR_CHECK(bn == 32 || bn == 64 || bn == 128 || bn == 256, "gemm: bad block_n %d", bn);
  GemmParams& p = plan->p;
  memset(&p, 0, sizeof(p));
  p.M = d.M; p.N = d.N; p.K = d.K;
  p.out32 = d.out32; p.ld32 = d.ld32; p.out16 = d.out16; p.ld16 = d.ld16;
  p.bias = d.bias; p.resid = d.resid; p.ldr = d.ldr; p.resid_mod = d.resid_mod; p.act = d.act; p.act32 = d.act32;
  p.seq_pitch = d.seq_pitch; p.seq_lo = d.seq_lo; p.seq_hi = d.seq_hi;
  p.alpha = d.alpha; p.argmin_out = d.argmin_out; p.row_sq = d.row_sq; p.col_sq = d.col_sq;
  THMR_CHECK(!d.screen_rows || (d.argmin_out && d.screen_count && d.screen_cmax2 && d.N % 32 == 0),
             "gemm: screened arg-min needs its queue and N %% 32 == 0");
  THMR_CHECK((!d.m_dev && !d.row_map) || d.argmin_out, "gemm: device row count / row map are arg-min options");
  p.screen_rows = d.screen_rows; p.screen_count = d.screen_count; p.screen_cmax2 = d.screen_cmax2;
  p.screen_rel = d.screen_rel; p.screen_abs = d.screen_abs; p.screen_row0 = d.screen_row0;
  p.row_map = d.row_map; p.m_dev = d.m_dev; p.m_dev_off = d.m_dev_off;
  p.stamp = d.stamp;
  const int num_kb = (d.K + kGemmBK - 1) / kGemmBK;
  uint64_t a_cols = d.K;
  if (d.taps > 1) {
    THMR_CHECK(d.cin % kGemmBK == 0 && d.K == d.taps * d.cin, "gemm conv: cin %d taps %d K %d", d.cin, d.taps, d.K);
    p.kblocks_per_tap = d.cin / kGemmBK;
    p.tap_row0 = d.tap_row0; p.tap_stride = d.tap_stride;
    a_cols = d.cin;
  } else {
    p.kblocks_per_tap = num_kb;
  }
  // CTA-pair kernel for the large TMA-epilogue GEMMs (the ViT projections)
  const bool two = epi != kEpiGeneric && d.taps == 1 && !d.no_2cta &&
                   (d.force_bn == 512 || (d.M >= 256 && d.N >= 256 && !d.force_bn));
  plan->two_cta = two ? 1 : 0;
  THMR_TRY(make_tmap_2d_f16(&plan->tmA, d.A, d.a_rows, a_cols, d.lda, kGemmBM, kGemmBK, CU_TENSOR_MAP_SWIZZLE_128B));
  const int b_box_rows = two ? kG2BN / 2 : bn;
  THMR_TRY(make_tmap_2d_f16(&plan->tmB, d.B, d.N, d.K, d.ldb, b_box_rows, kGemmBK, CU_TENSOR_MAP_SWIZZLE_128B));
  plan->bn = two ? kG2BN : bn;
  plan->epi = epi;
  // output boxes: 32 rows per epilogue warp, or (CTA-pair kernel) one 128-row slab per column half
  const uint32_t c_rows = two ? 128 : 32;
  if (epi == kEpiStore16)
    THMR_TRY(make_tmap_2d(&plan->tmC, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, d.out16, d.M, d.N, d.ld16, c_rows, 64,
                          CU_TENSOR_MAP_SWIZZLE_128B));
  else if (epi == kEpiAdd32 || epi == kEpiStore32)
    THMR_TRY(make_tmap_2d(&plan->tmC, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, d.out32, d.M, d.N, d.ld32, c_rows, 32,
                          CU_TENSOR_MAP_SWIZZLE_128B));
  else
    plan->tmC = plan->tmA;
  if (two) {
    const int clusters = num_sms() / 2;
    const long tiles = static_cast<long>((d.M + 255) / 256) * ((d.N + kG2BN - 1) / kG2BN);
    plan->grid = 2 * static_cast<int>(tiles < clusters ? tiles : clusters);
    // Stream-K (gemm2_tcgen05.cuh) when whole tiles quantise badly over the clusters: needs the reduce-add epilogue,
    // caller-provided ordering flags and at least two tiles of work per cluster (a tile is then shared by at most two
    // clusters).
    p.sk_flags = nullptr;
    p.sk_tiles = 0;
    // Short tiles do not pay: every partial tile costs a full 128 x 256 fp32 epilogue, which a 10-k-block main loop no
    // longer hides (proj, 20 k-blocks per tile: 45.3 us with stream-K vs 42.5 us without; fc2, 80: 126.7 vs 138.8 us).
    if (epi == kEpiAdd32 && d.sk_flags && tiles >= 2L * clusters && tiles % clusters != 0 && num_kb >= 40) {
      const double eff = static_cast<double>(tiles) / (((tiles + clusters - 1) / clusters) * clusters);
      const long sk_tiles = tiles % clusters + clusters;      // the last partial round plus one full round
      if (eff < 0.97 && static_cast<double>(sk_tiles) * num_kb * clusters < 2.0e9) {
        p.sk_flags = d.sk_flags;
        p.sk_tiles = static_cast<int>(sk_tiles);
        plan->grid = 2 * clusters;
      }
    }
    return THMR_OK;
  }
  const long tiles_m = (d.M + kGemmBM - 1) / kGemmBM;
  const long tiles = d.argmin_out ? tiles_m : tiles_m * ((d.N + bn - 1) / bn);
  // the CTAs of a wave should share tiles of the larger operand (TileIter)
  p.m_fast = (!d.argmin_out && tiles_m > 1 && d.M < d.N) ? 1 : 0;
  plan->grid = static_cast<int>(tiles < num_sms() ? tiles : num_sms());
  return THMR_OK;
}

template <int BN, int STAGES, int EPI>
inline int gemm_launch_t(const GemmPlan& plan, cudaStream_t stream) {
  using S = GemmSmem<BN, STAGES, EPI>;
  static bool configured = false;
  if (!configured) {
    THMR_CUDA(cudaFuncSetAttribute(gemm_f16_tn_kernel<BN, STAGES, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   S::kTotal));
    configured = true;
  }
  gemm_f16_tn_kernel<BN, STAGES, EPI><<<plan.grid, kGemmThreads, S::kTotal, stream>>>(plan.tmA, plan.tmB, plan.tmC,
                                                                                      plan.p);
  THMR_CUDA(cudaGetLastError());
  return THMR_OK;
}

template <int EPI>
inline int gemm2_launch_t(const GemmPlan& plan, cudaStream_t stream) {
  static bool configured = false;
  if (!configured) {
    THMR_CUDA(cudaFuncSetAttribute(gemm_f16_tn_2cta_kernel<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   kG2SmemTotal));
    configured = true;
  }
  gemm_f16_tn_2cta_kernel<EPI><<<plan.grid, kGemmThreads, kG2SmemTotal, stream>>>(plan.tmA, plan.tmB, plan.tmC, plan.p);
  THMR_CUDA(cudaGetLastError());
  return THMR_OK;
}

inline int gemm_launch(const GemmPlan& plan, cudaStream_t stream) {
  if (plan.two_cta) {
    if (plan.epi == kEpiStore16) return gemm2_launch_t<kEpiStore16>(plan, stream);
    if (plan.epi == kEpiAdd32) return gemm2_launch_t<kEpiAdd32>(plan, stream);
    if (plan.epi == kEpiStore32) return gemm2_launch_t<kEpiStore32>(plan, stream);
    return fail(THMR_ERR_INVALID, "gemm: CTA-pair kernel needs a TMA epilogue");
  }
  if (plan.epi == kEpiStore16) {
    if (plan.bn == 256) return gemm_launch_t<256, 4, kEpiStore16>(plan, stream);
    if (plan.bn == 128) return gemm_launch_t<128, 6, kEpiStore16>(plan, stream);
  } else if (plan.epi == kEpiAdd32) {
    if (plan.bn == 256) return gemm_launch_t<256, 4, kEpiAdd32>(plan, stream);
    if (plan.bn == 128) return gemm_launch_t<128, 6, kEpiAdd32>(plan, stream);
  } else if (plan.epi == kEpiStore32) {
    if (plan.bn == 256) return gemm_launch_t<256, 4, kEpiStore32>(plan, stream);
    if (plan.bn == 128) return gemm_launch_t<128, 6, kEpiStore32>(plan, stream);
  } else {
    switch (plan.bn) {
      case 256: return gemm_launch_t<256, 4, kEpiGeneric>(plan, stream);
      case 128: return gemm_launch_t<128, 6, kEpiGeneric>(plan, stream);
      case 64: return gemm_launch_t<64, 8, kEpiGeneric>(plan, stream);
      case 32: return gemm_launch_t<32, 8, kEpiGeneric>(plan, stream);
    }
  }
  return fail(THMR_ERR_INVALID, "gemm: unsupported block_n %d / epilogue %d", plan.bn, plan.epi);
}

}  // namespace thmr
