// Persistent warp-specialised tcgen05 GEMM:  C[M,N] = epilogue(alpha * A[M,K] * B[N,K]^T)
//   A (activations) and B (nn.Linear / conv weight, stored [out, in]) are both K-major fp16,
//   accumulation is fp32 in TMEM.
//
//   warps 0-7  : epilogue (two warps per TMEM lane quarter, each owning half of the tile's columns)
//   warp 8     : TMA producer (one thread)       global -> 128B-swizzled smem ring
//   warp 9     : MMA issuer   (one thread)       tcgen05.mma.cta_group::1.kind::f16, M=128, N=BN, K=16
//   warp 10    : TMEM allocator / deallocator
//
// Two TMEM accumulator buffers let the epilogue of tile i overlap the MMAs of tile i+1.
//
// Epilogue flavours (template EPI):
//   kEpiGeneric : tcgen05.ld -> bias / residual / activation -> direct global stores; handles every option
//                 (two outputs, residual tables, padded-sequence masking, row-argmin).  Used by the small-M tail.
//   kEpiStore16 : act(acc + bias) -> fp16 -> 128B-swizzled smem -> TMA store            (QKV, fc1+GELU, to_kv)
//   kEpiStore32 : alpha * acc + bias, fp32 -> swizzled smem -> TMA store                 (SMPL pose-blend offsets)
//   kEpiAdd32   : (acc + bias) fp32 -> swizzled smem -> TMA reduce-add into the output   (proj / fc2: x += ...)
//                 the residual add happens in the L2 reduction unit, the residual is never read by the SM.
//
// The same kernel runs the implicit-GEMM Conv1d (k=3, dilated) of the pose-token decoder: k-blocks are
// grouped in "taps", each tap reads the A rows shifted by a row offset (TMA zero-fills out-of-range rows).
#pragma once
#include "ptx.cuh"

namespace thmr {

enum : int { kActNone = 0, kActGelu = 1, kActRelu = 2 };
enum : int { kEpiGeneric = 0, kEpiStore16 = 1, kEpiAdd32 = 2, kEpiStore32 = 3 };

struct GemmParams {
  int M, N, K;
  float* out32;   // acc + bias + resid, fp32 (nullable)
  int ld32;
  __half* out16;  // act(acc + bias + resid) rounded to fp16 (nullable)
  int ld16;
  const float* bias;   // [N] (nullable)
  const float* resid;  // fp32 [*, N] (nullable); may alias out32 (same element, same thread)
  int ldr;
  int resid_mod;  // > 0: residual row = row % resid_mod (position-embedding table)
  int act;
  int act32;  // apply the activation to the fp32 output as well (conv + ReLU feeding a residual)
  // implicit conv: tap t = kb / kblocks_per_tap reads A rows (m + tap_row0 + t * tap_stride)
  int kblocks_per_tap;
  int tap_row0, tap_stride;
  // padded sequences: rows with (row % seq_pitch) outside [seq_lo, seq_hi) are stored as zero
  int seq_pitch, seq_lo, seq_hi;
  float alpha;  // accumulator scale (split-precision operands are pre-scaled by powers of two)
  // row-argmin mode (VQ nearest code, quantize_cnn.py:80-86): the CTA walks all column tiles of one row
  // block and keeps a running first-minimum of  d = (row_sq[row] - 2*alpha*acc) + col_sq[col]
  long long* argmin_out;   // [M] int64 (nullable = normal GEMM)
  const float* row_sq;     // [M]
  const float* col_sq;     // [N]
  // screened row-argmin (vq.cuh, two-pass hard quantise).  Pass 1 (screen_rows != nullptr) runs single-product fp16
  // operands, keeps the best AND the second-best of  e = col_sq - 2*alpha*acc  per row, always stores the best index
  // and appends the row to screen_rows when (second - best) does not exceed the rigorous error margin
  //   tau = screen_rel * sqrt(row_sq * cmax2) + screen_abs * (row_sq + cmax2) + 1e-12   (cmax2 = max col_sq);
  // such rows are re-done by the exact split-precision pass.  The exact pass reads its row count from device memory
  // (m_dev, minus m_dev_off, clamped to [0, M]) and scatters through row_map.
  int* screen_rows;            // [>= M rows of capacity overall] global row ids of the rows to re-do (nullable)
  int* screen_count;           // device counter (appended with one atomicAdd per warp)
  const float* screen_cmax2;   // device scalar: max over col_sq
  float screen_rel, screen_abs;
  int screen_row0;             // global id of row 0 of this launch (pass 1 runs in L2-sized chunks)
  const int* row_map;          // exact pass: argmin_out[row_map[row]] (nullable = identity)
  const int* m_dev;            // device row count (nullable = M)
  int m_dev_off;
  // stream-K (CTA-pair kernel, reduce-add epilogue): non-null = the k-blocks of all tiles are cut into one contiguous
  // range per cluster; a tile shared by two clusters is reduce-added in a FIXED order through these flags
  // ([tile][cta rank][column half], zero between launches)
  unsigned int* sk_flags;
  int sk_tiles;   // trailing tiles scheduled stream-K (gemm2_tcgen05.cuh G2Work)
  unsigned long long* stamp;   // in-graph start stamp (common.cuh stamp_start), nullable
  int m_fast;     // 1-CTA kernel: row tile fastest in the tile order (see TileIter)
};

// Tile order shared by the three warp roles.  Normal mode: tiles round-robin over CTAs, column tile
// fastest -- or row tile fastest (GemmParams::m_fast, chosen by the host when M < N): the CTAs of a wave then share the
// tiles of the LARGER operand, which is streamed from HBM once instead of once per wave (SMPL blend GEMM: 512 poses x
// 20672 basis rows).  Row-argmin mode: row blocks round-robin over CTAs, all column tiles of a row block in sequence.
struct TileIter {
  int tiles_m, tiles_n, m_blk, n_blk, tile, num_tiles;
  bool m_stationary, m_fast;
  __device__ TileIter(int tm, int tn, bool ms, bool mf = false) : tiles_m(tm), tiles_n(tn), m_stationary(ms), m_fast(mf) {
    num_tiles = tm * tn;
    tile = blockIdx.x;
    m_blk = blockIdx.x;
    n_blk = 0;
  }
  __device__ bool valid() const { return m_stationary ? (m_blk < tiles_m) : (tile < num_tiles); }
  __device__ int m0(int bm) const { return (m_stationary ? m_blk : (m_fast ? tile % tiles_m : tile / tiles_n)) * bm; }
  __device__ int n0(int bn) const { return (m_stationary ? n_blk : (m_fast ? tile / tiles_m : tile % tiles_n)) * bn; }
  __device__ bool last_n() const { return n_blk == tiles_n - 1; }
  __device__ void next() {
    if (m_stationary) {
      if (++n_blk == tiles_n) { n_blk = 0; m_blk += gridDim.x; }
    } else {
      tile += gridDim.x;
    }
  }
};

constexpr int kGemmBM = 128;
constexpr int kGemmBK = 64;
constexpr int kGemmEpiWarps = 8;
constexpr int kGemmThreads = 128 + 32 * kGemmEpiWarps;  // 8 epilogue warps + 4 control warps
// The SMSP arbiter favours the highest warp id: the latency-critical single-thread roles get the top ids so that
// bursts of epilogue ALU work (bias, GELU, packing) never delay a TMA issue or a tcgen05.mma issue.
constexpr int kWarpTma = kGemmEpiWarps;        // 8
constexpr int kWarpMma = kGemmEpiWarps + 1;    // 9
constexpr int kWarpAlloc = kGemmEpiWarps + 2;  // 10

template <int BN, int STAGES, int EPI>
struct GemmSmem {
  static constexpr uint32_t kABytes = kGemmBM * kGemmBK * 2;
  static constexpr uint32_t kBBytes = BN * kGemmBK * 2;
  static constexpr uint32_t kStageBytes = kABytes + kBBytes;
  static constexpr uint32_t kStagingOffset = STAGES * kStageBytes;              // 1024-aligned
  static constexpr uint32_t kStagingBytes = (EPI == kEpiGeneric) ? 0 : kGemmEpiWarps * 4096;
  static constexpr uint32_t kBarOffset = kStagingOffset + kStagingBytes;
  static constexpr uint32_t kTotal = kBarOffset + 1792 + 1024;  // barriers + argmin exchange, alignment slack
};

// Exact-erf GELU (nn.GELU default, vit.py:73).  The epilogue evaluates 63 M of these per MLP layer, so erf uses
// Abramowitz-Stegun 7.1.28  erf(a) = 1 - (1 + c1 a + ... + c6 a^6)^-16  (|err| < 2e-6 in fp32, i.e. GELU within
// 9e-7 absolute of the libm path; the result is rounded to fp16 afterwards): 7 FMA + 4 MUL + 1 MUFU.RCP, no branches.
__device__ __forceinline__ float gelu_erf(float x) {
  const float a = fabsf(x) * 0.70710678118654752f;
  float p = fmaf(0.0000430638f, a, 0.0002765672f);
  p = fmaf(p, a, 0.0001520143f);
  p = fmaf(p, a, 0.0092705272f);
  p = fmaf(p, a, 0.0422820123f);
  p = fmaf(p, a, 0.0705230784f);
  p = fmaf(p, a, 1.0f);
  p *= p; p *= p; p *= p; p *= p;
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(p));   // 1 ulp-class MUFU reciprocal (p >= 1; p = inf -> 0)
  const float e = 1.0f - r;                       // erf(|x| / sqrt(2))
  return 0.5f * x + 0.5f * fabsf(x) * e;          // 0.5 x (1 + sign(x) e)
}

// Two GELUs per instruction stream on the packed fp32 pipe (FFMA2: fma.rn.f32x2, IEEE per lane).  Same polynomial as
// gelu_erf, rearranged so that everything but |x|, max and the reciprocal is packed:
//   t = -0.5|x|,  a = |x|/sqrt(2) = t * (-sqrt(2)),  r = 1 / (1 + c1 a + ... + c6 a^6)^16,  gelu = max(x, 0) + t * r
// 18 issue slots per PAIR instead of ~17 per element: the fc1 epilogue (63 M GELUs per layer) is issue-bound.
// x = (x0, x1) packed -> (gelu(x0), gelu(x1)) packed
__device__ __forceinline__ uint64_t gelu_erf2(uint64_t x) {
  float x0, x1;
  f2_unpack(x, x0, x1);
  const uint64_t t = f2_pack(fabsf(x0) * -0.5f, fabsf(x1) * -0.5f);
  const uint64_t a = f2_mul(t, f2_splat(-1.41421356237309505f));
  uint64_t p = f2_fma(f2_splat(0.0000430638f), a, f2_splat(0.0002765672f));
  p = f2_fma(p, a, f2_splat(0.0001520143f));
  p = f2_fma(p, a, f2_splat(0.0092705272f));
  p = f2_fma(p, a, f2_splat(0.0422820123f));
  p = f2_fma(p, a, f2_splat(0.0705230784f));
  p = f2_fma(p, a, f2_splat(1.0f));
  p = f2_mul(p, p); p = f2_mul(p, p); p = f2_mul(p, p); p = f2_mul(p, p);
  float p0, p1, r0, r1;
  f2_unpack(p, p0, p1);
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r0) : "f"(p0));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r1) : "f"(p1));
  return f2_fma(t, f2_pack(r0, r1), f2_pack(fmaxf(x0, 0.f), fmaxf(x1, 0.f)));
}

__device__ __forceinline__ void named_bar_sync_64(int id) {
  asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory");
}
__device__ __forceinline__ void named_bar_sync_128(int id) {
  asm volatile("bar.sync %0, 128;" ::"r"(id) : "memory");
}
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* m, const void* smem_src, int32_t c0, int32_t c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.bulk_group [%0, {%2, %3}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}

template <int BN, int STAGES, int EPI>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_f16_tn_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                   const __grid_constant__ CUtensorMap tmC, const GemmParams p) {
  using S = GemmSmem<BN, STAGES, EPI>;
  constexpr uint32_t kTmemCols = (2 * BN < 32) ? 32 : 2 * BN;
  static_assert(BN == 32 || BN == 64 || BN == 128 || BN == 256, "BN must be a power of two in [32,256]");
  static_assert(EPI == kEpiGeneric || BN >= 128, "TMA epilogues need BN >= 128 (two column halves of >= 64)");

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + S::kBarOffset);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tfull_bar = empty_bar + STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  float* xch_val = reinterpret_cast<float*>(smem + S::kBarOffset + 256);   // [128] argmin exchange
  int* xch_idx = reinterpret_cast<int*>(xch_val + 128);                     // [128]
  float* xch_sec = reinterpret_cast<float*>(xch_idx + 128);                 // [128] second-best (screened arg-min)

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // rows of this launch: p.M, or (exact pass of the screened arg-min) a count a previous kernel left in device memory.
  // Every thread reads the same word, so the three warp roles walk identical tile sequences.
  int M_eff = p.M;
  if (p.m_dev != nullptr) {
    const int m = __ldg(p.m_dev) - p.m_dev_off;
    M_eff = m < 0 ? 0 : (m < p.M ? m : p.M);
  }
  const int tiles_m = (M_eff + kGemmBM - 1) / kGemmBM;
  const int tiles_n = (p.N + BN - 1) / BN;
  const int num_kb = (p.K + kGemmBK - 1) / kGemmBK;

  stamp_start(p.stamp);
  if (warp == kWarpTma && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (EPI != kEpiGeneric) tma_prefetch_desc(&tmC);
  }
  if (warp == kWarpMma && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], kGemmEpiWarps);  // one arrive per epilogue warp
    }
    fence_mbar_init();
  }
  if (warp == kWarpAlloc) {
    tmem_alloc(tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kWarpTma) {
    if (lane == 0) {
      // ------------------------------------------------------------ TMA producer
      int stage = 0;
      uint32_t phase = 0;
      for (TileIter it(tiles_m, tiles_n, p.argmin_out != nullptr, p.m_fast != 0); it.valid(); it.next()) {
        const int m0 = it.m0(kGemmBM);
        const int n0 = it.n0(BN);
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * S::kStageBytes;
          uint8_t* sb = sa + S::kABytes;
          const int tap = kb / p.kblocks_per_tap;
          const int kk = kb - tap * p.kblocks_per_tap;
          mbar_arrive_expect_tx(&full_bar[stage], S::kStageBytes);
          tma_load_2d(sa, &tmA, &full_bar[stage], kk * kGemmBK, m0 + p.tap_row0 + tap * p.tap_stride);
          tma_load_2d(sb, &tmB, &full_bar[stage], kb * kGemmBK, n0);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == kWarpMma) {
    {
      // ------------------------------------------------------------ MMA issuer (warp-converged, one elected lane issues)
      // All 32 lanes walk the pipeline: uniform control flow lets ptxas keep the descriptors in uniform registers and
      // issue the four UTCHMMA of a k-block back to back (see gemm2_tcgen05.cuh for the measurement behind this).
      constexpr uint32_t idesc = make_idesc_f16(kGemmBM, BN);
      const uint32_t smem_base = smem_u32(smem);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      // The readiness of the NEXT smem stage is probed right after the MMA issues of the current one, so the latency of
      // mbarrier.try_wait (~100-200 cycles even when the phase is complete) overlaps with tensor work.
      bool ready = false;
      for (TileIter it(tiles_m, tiles_n, p.argmin_out != nullptr, p.m_fast != 0); it.valid(); it.next()) {
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_u + acc * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          if (!ready) mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_base + stage * S::kStageBytes;
          const uint32_t sb = sa + S::kABytes;
          const int nstage = (stage + 1 == STAGES) ? 0 : stage + 1;
          const uint32_t nphase = (stage + 1 == STAGES) ? (phase ^ 1) : phase;
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < kGemmBK / 16; ++k) {
              const uint64_t da = make_smem_desc(sa + k * 32, 16, 1024, kSwz128);
              const uint64_t db = make_smem_desc(sb + k * 32, 16, 1024, kSwz128);
              umma_f16_ss(d_tmem, da, db, idesc, (kb | k) != 0 ? 1u : 0u);
            }
            umma_commit(&empty_bar[stage]);  // smem slot free once these MMAs retire
            if (kb == num_kb - 1) umma_commit(&tfull_bar[acc]);
          }
          __syncwarp();
          ready = __all_sync(0xffffffffu, mbar_try_wait(&full_bar[nstage], nphase));   // peek (result is only a hint)
          stage = nstage;
          phase = nphase;
        }
        if ((acc ^= 1) == 0) acc_phase ^= 1;
      }
    }
  } else if (warp < kGemmEpiWarps) {
    // -------------------------------------------------------------- epilogue
    const int q = warp & 3;            // TMEM lane quarter this warp may access
    const int half = warp >> 2;  // which half of the tile's columns
    const uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
    int acc = 0;
    uint32_t acc_phase = 0;

    if constexpr (EPI == kEpiGeneric) {
      constexpr int kChunks = BN / 32;
      constexpr int kChunksPerHalf = (kChunks + 1) / 2;
      const bool vec16 = p.out16 && (p.ld16 % 8 == 0);
      const bool vec32 = (!p.out32 || p.ld32 % 4 == 0) && (!p.resid || p.ldr % 4 == 0);
      float best = INFINITY;
      int best_idx = 0;
      float second = INFINITY;                 // screened arg-min: second-smallest value of the row
      const bool screen = p.argmin_out != nullptr && p.screen_rows != nullptr;
      const float m2a = -2.0f * p.alpha;
      for (TileIter it(tiles_m, tiles_n, p.argmin_out != nullptr, p.m_fast != 0); it.valid(); it.next()) {
        const int m0 = it.m0(kGemmBM);
        const int n0 = it.n0(BN);
        const int row = m0 + q * 32 + lane;
        const bool row_ok = row < M_eff;
        bool row_zero = false;
        if (p.seq_pitch > 0) {
          const int r = row % p.seq_pitch;
          row_zero = (r < p.seq_lo) || (r >= p.seq_hi);
        }
        const float* rrow = nullptr;
        if (p.resid) rrow = p.resid + static_cast<size_t>(p.resid_mod > 0 ? row % p.resid_mod : row) * p.ldr;

        // row-argmin: this warp's column norms (lane l: 4 columns of its column half) and the row norm are
        // fetched while the MMAs run; the inner loop then only shuffles
        float4 cq = make_float4(0.f, 0.f, 0.f, 0.f);
        float x2 = 0.f;
        if (p.argmin_out) {
          const int bc = n0 + half * kChunksPerHalf * 32 + lane * 4;
          if (lane * 4 < kChunksPerHalf * 32 && bc + 3 < p.N) cq = __ldg(reinterpret_cast<const float4*>(p.col_sq + bc));
          if (row_ok) x2 = __ldg(p.row_sq + row);
        }
        if (lane == 0) mbar_wait(&tfull_bar[acc], acc_phase);   // one polling lane per warp
        __syncwarp();
        tc_fence_after();
#pragma unroll 1
        for (int cc = 0; cc < kChunksPerHalf; ++cc) {
          const int c = half * kChunksPerHalf + cc;
          if (c >= kChunks) break;
          uint32_t v[32];
          tmem_ld_x32(tmem_base + lane_addr + acc * BN + c * 32, v);
          tmem_ld_wait();
          const int col0 = n0 + c * 32;
          if (screen) {
            // pass 1 of the screened arg-min: e = col_sq - 2 alpha acc (the row norm is common to every column), running
            // best / second best; ties and near-ties are settled by the exact pass, so only the margin matters here
            // The epilogue is ALU-pipe bound (min / compare / select are half rate), so the column index rides in the value: the
            // low byte of e's mantissa is replaced by the column's position in its 32-column chunk (one byte permute), which
            // perturbs e by < 2^-15 relative (covered by screen_abs), and the chunk itself is noted once per chunk.  Three
            // min / max and a permute per column instead of three min / max, a compare, a select and the index arithmetic.
            if (col0 < p.N) {   // (warp-uniform: shuffles below need every lane; N % 32 == 0 is checked by the host)
              const float best_before = best;
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                const int bl = (cc * 32 + j) >> 2;
                float c2[4];
                c2[0] = __shfl_sync(0xffffffffu, cq.x, bl); c2[1] = __shfl_sync(0xffffffffu, cq.y, bl);
                c2[2] = __shfl_sync(0xffffffffu, cq.z, bl); c2[3] = __shfl_sync(0xffffffffu, cq.w, bl);
                // (a group-minimum pre-test that skips columns above the current second best was tried: the divergent branch
                //  cost more than the skipped min / compare / select chain saved, 2.17 vs 1.95 ms per 1 M queries)
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const float d = fmaf(m2a, __uint_as_float(v[j + e]), c2[e]);
                  // low byte of the value := position in the chunk (one PRMT; the byte constants live in 8 registers)
                  const float k = __uint_as_float(__byte_perm(__float_as_uint(d), 0x03020100u + 0x04040404u * ((j + e) >> 2),
                                                              0x3214u + ((j + e) & 3)));
                  second = fminf(second, fmaxf(k, best));
                  best = fminf(best, k);
                }
              }
              if (best < best_before) best_idx = col0;   // chunk of the running best; the column is in the key's low bits
            }
          } else if (p.argmin_out) {
            if (col0 < p.N) {   // (warp-uniform: shuffles below need every lane)
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                const int bl = (cc * 32 + j) >> 2;
                float c2[4];
                c2[0] = __shfl_sync(0xffffffffu, cq.x, bl); c2[1] = __shfl_sync(0xffffffffu, cq.y, bl);
                c2[2] = __shfl_sync(0xffffffffu, cq.z, bl); c2[3] = __shfl_sync(0xffffffffu, cq.w, bl);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  // same expression order as the reference: (sum x^2 - 2 x.c) + sum c^2
                  const float d = (x2 - 2.0f * (p.alpha * __uint_as_float(v[j + e]))) + c2[e];
                  if (col0 + j + e < p.N && d < best) { best = d; best_idx = col0 + j + e; }
                }
              }
            }
          } else if (row_ok && col0 < p.N) {
            const bool full = (col0 + 32 <= p.N);
            float f[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) f[j] = p.alpha * __uint_as_float(v[j]);
            if (p.bias) {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (full || col0 + j < p.N) f[j] += __ldg(p.bias + col0 + j);
            }
            if (rrow) {
              if (full && vec32) {
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                  const float4 r4 = *reinterpret_cast<const float4*>(rrow + col0 + j);
                  f[j] += r4.x; f[j + 1] += r4.y; f[j + 2] += r4.z; f[j + 3] += r4.w;
                }
              } else {
#pragma unroll
                for (int j = 0; j < 32; ++j)
                  if (col0 + j < p.N) f[j] += rrow[col0 + j];
              }
            }
            if (row_zero) {
#pragma unroll
              for (int j = 0; j < 32; ++j) f[j] = 0.f;
            }
            if (p.act32) {
              if (p.act == kActGelu) {
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = gelu_erf(f[j]);
              } else if (p.act == kActRelu) {
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
              }
            }
            if (p.out32) {
              float* o = p.out32 + static_cast<size_t>(row) * p.ld32 + col0;
              if (full && vec32) {
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                  *reinterpret_cast<float4*>(o + j) = make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]);
              } else {
#pragma unroll
                for (int j = 0; j < 32; ++j)
                  if (col0 + j < p.N) o[j] = f[j];
              }
            }
            if (p.out16) {
              if (p.act32) {
              } else if (p.act == kActGelu) {
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = gelu_erf(f[j]);
              } else if (p.act == kActRelu) {
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
              }
              __half* o = p.out16 + static_cast<size_t>(row) * p.ld16 + col0;
              if (full && vec16) {
#pragma unroll
                for (int j = 0; j < 32; j += 8) {
                  uint4 pk;
                  __half2 h0 = __floats2half2_rn(f[j], f[j + 1]);
                  __half2 h1 = __floats2half2_rn(f[j + 2], f[j + 3]);
                  __half2 h2 = __floats2half2_rn(f[j + 4], f[j + 5]);
                  __half2 h3 = __floats2half2_rn(f[j + 6], f[j + 7]);
                  pk.x = *reinterpret_cast<uint32_t*>(&h0);
                  pk.y = *reinterpret_cast<uint32_t*>(&h1);
                  pk.z = *reinterpret_cast<uint32_t*>(&h2);
                  pk.w = *reinterpret_cast<uint32_t*>(&h3);
                  *reinterpret_cast<uint4*>(o + j) = pk;
                }
              } else {
#pragma unroll
                for (int j = 0; j < 32; ++j)
                  if (col0 + j < p.N) o[j] = __float2half_rn(f[j]);
              }
            }
          }
        }
        if (p.argmin_out && it.last_n()) {
          // merge the two column halves: smaller distance wins, equal distances -> smaller index
          // (== first minimum over the whole row, as torch.min returns)
          if (screen) best_idx += static_cast<int>(__float_as_uint(best) & 255u);   // unpack the column (pass-1 keys)
          if (half == 1) {
            xch_val[q * 32 + lane] = best; xch_idx[q * 32 + lane] = best_idx; xch_sec[q * 32 + lane] = second;
          }
          named_bar_sync_64(1 + q);
          if (half == 0) {
            const float ob = xch_val[q * 32 + lane];
            const int oi = xch_idx[q * 32 + lane];
            // second best of the whole row: the smaller of the two seconds and the larger of the two bests
            const float sec = fminf(fminf(second, xch_sec[q * 32 + lane]), fmaxf(best, ob));
            if (ob < best || (ob == best && oi < best_idx)) { best = ob; best_idx = oi; }
            if (row_ok) p.argmin_out[p.row_map ? __ldg(p.row_map + row) : row] = best_idx;
            if (screen) {
              // rows whose margin does not clear the error bound of the single-product pass are queued for the exact pass
              // (NaNs fail the comparison and are queued too); one atomicAdd per warp
              const float cm2 = __ldg(p.screen_cmax2);
              const float tau = p.screen_rel * sqrtf(x2 * cm2) + p.screen_abs * (x2 + cm2) + 1e-12f;
              const bool redo = row_ok && !(sec - best > tau);
              const unsigned mask = __ballot_sync(0xffffffffu, redo);
              if (mask != 0u) {
                const int leader = __ffs(mask) - 1;
                int base = 0;
                if (lane == leader) base = atomicAdd(p.screen_count, __popc(mask));
                base = __shfl_sync(0xffffffffu, base, leader);
                if (redo) p.screen_rows[base + __popc(mask & ((1u << lane) - 1u))] = p.screen_row0 + row;
              }
            }
          }
          named_bar_sync_64(1 + q);
          best = INFINITY;
          best_idx = 0;
          second = INFINITY;
        }
        // all TMEM reads of this warp are complete (wait::ld above): hand the buffer back
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty_bar[acc]);
        if ((acc ^= 1) == 0) acc_phase ^= 1;
      }
    } else {
      // ---------------------------------------------------------- TMA-store epilogues
      // chunk = 128 bytes of output per row: 64 fp16 columns (Store16) or 32 fp32 columns (Add32).
      constexpr int kChunkCols = (EPI == kEpiStore16) ? 64 : 32;
      constexpr int kChunks = BN / kChunkCols;
      constexpr int kChunksPerHalf = kChunks / 2;
      uint8_t* stage_buf = smem + S::kStagingOffset + warp * 4096;   // [32 rows][128 B], 128B-swizzled
      const uint32_t srow = smem_u32(stage_buf) + lane * 128;
      const int sw = lane & 7;
      for (TileIter it(tiles_m, tiles_n, false, p.m_fast != 0); it.valid(); it.next()) {
        const int m0 = it.m0(kGemmBM);
        const int n0 = it.n0(BN);
        // this warp's BN/2 bias values (lane l: columns 4l..4l+3 of its column half), fetched while the MMAs run
        float4 bq = make_float4(0.f, 0.f, 0.f, 0.f);
        {
          const int bc = n0 + half * (BN / 2) + lane * 4;
          if (p.bias && lane * 4 < BN / 2 && bc < p.N) bq = __ldg(reinterpret_cast<const float4*>(p.bias + bc));
        }
        if (lane == 0) mbar_wait(&tfull_bar[acc], acc_phase);   // one polling lane per warp
        __syncwarp();
        tc_fence_after();
#pragma unroll 1
        for (int cc = 0; cc < kChunksPerHalf; ++cc) {
          const int c = half * kChunksPerHalf + cc;
          const int col0 = n0 + c * kChunkCols;
          uint32_t pk[32];
          if constexpr (EPI == kEpiStore16) {
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              uint32_t v[32];
              tmem_ld_x32(tmem_base + lane_addr + acc * BN + c * 64 + hh * 32, v);
              tmem_ld_wait();
              float f[32];
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                const int bl = (cc * 64 + hh * 32 + j) >> 2;   // lane holding these 4 columns' bias
                float4 b4;
                b4.x = __shfl_sync(0xffffffffu, bq.x, bl); b4.y = __shfl_sync(0xffffffffu, bq.y, bl);
                b4.z = __shfl_sync(0xffffffffu, bq.z, bl); b4.w = __shfl_sync(0xffffffffu, bq.w, bl);
                f[j] = __uint_as_float(v[j]) + b4.x; f[j + 1] = __uint_as_float(v[j + 1]) + b4.y;
                f[j + 2] = __uint_as_float(v[j + 2]) + b4.z; f[j + 3] = __uint_as_float(v[j + 3]) + b4.w;
              }
              // warp-uniform branch OUTSIDE the element loop (otherwise the compiler if-converts it and every element
              // pays for GELU and ReLU even when no activation is requested)
              if (p.act == kActGelu) {
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = gelu_erf(f[j]);
              } else if (p.act == kActRelu) {
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
              }
#pragma unroll
              for (int j = 0; j < 32; j += 2) {
                __half2 h2 = __floats2half2_rn(f[j], f[j + 1]);
                pk[hh * 16 + (j >> 1)] = *reinterpret_cast<uint32_t*>(&h2);
              }
            }
          } else {
            uint32_t v[32];
            tmem_ld_x32(tmem_base + lane_addr + acc * BN + c * 32, v);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const int bl = (cc * 32 + j) >> 2;
              float4 b4;
              b4.x = __shfl_sync(0xffffffffu, bq.x, bl); b4.y = __shfl_sync(0xffffffffu, bq.y, bl);
              b4.z = __shfl_sync(0xffffffffu, bq.z, bl); b4.w = __shfl_sync(0xffffffffu, bq.w, bl);
              pk[j] = __float_as_uint(fmaf(p.alpha, __uint_as_float(v[j]), b4.x));
              pk[j + 1] = __float_as_uint(fmaf(p.alpha, __uint_as_float(v[j + 1]), b4.y));
              pk[j + 2] = __float_as_uint(fmaf(p.alpha, __uint_as_float(v[j + 2]), b4.z));
              pk[j + 3] = __float_as_uint(fmaf(p.alpha, __uint_as_float(v[j + 3]), b4.w));
            }
          }
          // the previous TMA store of this warp must have finished reading the staging tile
          if (lane == 0) tma_store_wait_read<0>();
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(srow + ((j ^ sw) << 4)), "r"(pk[4 * j]),
                         "r"(pk[4 * j + 1]), "r"(pk[4 * j + 2]), "r"(pk[4 * j + 3])
                         : "memory");
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0 && col0 < p.N && m0 + q * 32 < M_eff) {
            if constexpr (EPI == kEpiStore16) tma_store_2d(&tmC, stage_buf, col0, m0 + q * 32);
            else if constexpr (EPI == kEpiStore32) tma_store_2d(&tmC, stage_buf, col0, m0 + q * 32);
            else tma_reduce_add_2d(&tmC, stage_buf, col0, m0 + q * 32);
            tma_store_commit();
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty_bar[acc]);
        if ((acc ^= 1) == 0) acc_phase ^= 1;
      }
      if (lane == 0) tma_store_wait<0>();   // all bulk stores complete before the CTA exits
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kWarpAlloc) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

}  // namespace thmr
