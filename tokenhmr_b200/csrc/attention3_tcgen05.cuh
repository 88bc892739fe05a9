// Fused ViT attention (reference: Attention.forward, vit.py:116-122): two independent tile chains per CTA.
//
// The first two generations of this kernel (removed) ran S-MMA -> softmax -> PV-MMA -> epilogue as one serial chain per
// 128-row tile, with the same eight warps doing every softmax and every epilogue (counters: each role idle ~60 %, ~12 k
// cycles per head while the tensor pipe needs ~1.9 k and the exp unit ~2.3 k).  Here the CTA holds TWO tile buffers in TMEM, each owned by
// its own group of four softmax warps and its own MMA-issuing thread, so that one group's exponentials overlap the
// other group's MMAs, TMEM traffic and epilogue.  (One issuer polling both chains was tried first: a non-blocking
// mbarrier probe costs 130-260 cycles, so every hand-over was detected ~500 cycles late.)
//
//   head i (per CTA), 192 query rows = tile 0 (rows 0..127) + tile 1 (64 useful rows + 64 wasted MMA rows):
//     tile 0 -> chain (i & 1), tile 1 -> chain (i & 1) ^ 1      (the 128-row and the 64-row tiles alternate, so both
//                                                                  groups carry 192 rows per two heads)
//     tile 1 = rows 64..191 (useful TMEM lanes 64..127) for heads with (i >> 1) even, rows 128..255 (useful lanes
//     0..63, rows >= 192 read whatever follows Q in shared memory) otherwise, so that the four SM sub-partitions,
//     each with its own exp unit, see the same number of rows
//   chain g owns TMEM columns [192 g, 192 g + 192):
//     S = Q_t K^T          tcgen05.mma SS (fp32, 192 columns)
//     softmax              thread = one query row: pass 1 row max, pass 2 exp2 / row sum, both streamed from TMEM
//                          in 32-column loads that are one load ahead of the arithmetic; P (fp16 pairs) is written
//                          IN PLACE over consumed S columns [0, 96)
//     O = P V              tcgen05.mma TS (A = P from TMEM, V N-major from smem) into columns [96, 176)
//     epilogue             O / rowsum -> fp16 -> global (row sum stays in the thread's register)
//   Q, K, V of a head are double-buffered in shared memory (2 x 90 KB), so the next head streams in from HBM/L2 while
//   this one is computed; both chains release a stage (two commits per barrier).
//
//   warps 0..3 : softmax group 0 (TMEM lane quarter = warp id)      warp 8     : TMA producer
//   warps 4..7 : softmax group 1                                     warps 9,10 : MMA issuers of chains 0,1 (9 owns TMEM)
#pragma once
#include "attention_common.cuh"

namespace thmr {

constexpr uint32_t kAtt3StageBytes = 3 * kAttMatBytes;            // Q | K | V of one head
constexpr uint32_t kAtt3OffOut = 2 * kAtt3StageBytes;              // 8 warps x [32 rows][80] fp16 TMA-store staging
constexpr uint32_t kAtt3OutWarpBytes = 32 * kAttHeadDim * 2;
constexpr uint32_t kAtt3OffBars = kAtt3OffOut + 8 * kAtt3OutWarpBytes;
constexpr uint32_t kAtt3SmemBytes = kAtt3OffBars + 34 * 8 + 1024;
constexpr int kAtt3Threads = 352;
constexpr uint32_t kAtt3BufCols = 192;                            // TMEM columns per chain
constexpr uint32_t kAtt3ColO = 96;

// 32 keys of softmax pass 2: exp2(s * scale - mo), accumulated into four partial row sums and written to TMEM as 16
// fp16 pairs.
__device__ __forceinline__ void att3_exp_chunk(const uint32_t (&cur)[32], uint32_t taddr, float sc, float mo,
                                               float& s0, float& s1, float& s2, float& s3) {
  uint32_t w16[16];
#pragma unroll
  for (int e = 0; e < 32; e += 4) {
    const float x0 = fmaf(__uint_as_float(cur[e]), sc, -mo);
    const float x1 = fmaf(__uint_as_float(cur[e + 1]), sc, -mo);
    const float x2 = fmaf(__uint_as_float(cur[e + 2]), sc, -mo);
    const float x3 = fmaf(__uint_as_float(cur[e + 3]), sc, -mo);
    const float e0 = fast_exp2(x0);
    const float e1 = fast_exp2(x1);
    const float e2 = fast_exp2(x2);
    const float e3 = fast_exp2(x3);
    s0 += e0; s1 += e1; s2 += e2; s3 += e3;
    __half2 h01 = __floats2half2_rn(e0, e1);
    __half2 h23 = __floats2half2_rn(e2, e3);
    w16[e >> 1] = *reinterpret_cast<uint32_t*>(&h01);
    w16[(e >> 1) + 1] = *reinterpret_cast<uint32_t*>(&h23);
  }
  tmem_st_x16(taddr, w16);
}

// Softmax pass 2 of one row: exp2(s * scale - mo) over 192 keys streamed from TMEM (one 32-column load ahead),
// P as fp16 pairs written in place over consumed columns (keys [32 j, 32 j + 32) -> columns [16 j, 16 j + 16), always
// behind the columns already read); returns the fp32 row sum.
// The loops are deliberately NOT fully unrolled: the straight-line version of this kernel was ~100 KB of SASS and the
// softmax warps spent 40-50 % of their samples in stall_no_inst (instruction fetch).
__device__ __forceinline__ float att3_pass2(uint32_t tb, float sc, float mo) {
  uint32_t va[32], vb[32];
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  tmem_ld_x32(tb, va);
#pragma unroll 1
  for (int jj = 0; jj < 3; ++jj) {
    tmem_ld_x32(tb + (2 * jj + 1) * 32, vb);
    tmem_ld_wait();
    att3_exp_chunk(va, tb + (2 * jj) * 16, sc, mo, s0, s1, s2, s3);
    if (jj < 2) tmem_ld_x32(tb + (2 * jj + 2) * 32, va);
    tmem_ld_wait();
    att3_exp_chunk(vb, tb + (2 * jj + 1) * 16, sc, mo, s0, s1, s2, s3);
  }
  tmem_st_wait();
  return (s0 + s1) + (s2 + s3);
}

__device__ __forceinline__ void att3_max_chunk(const uint32_t (&cur)[32], float& m0, float& m1, float& m2, float& m3) {
#pragma unroll
  for (int e = 0; e < 32; e += 4) {
    m0 = fmaxf(m0, __uint_as_float(cur[e]));
    m1 = fmaxf(m1, __uint_as_float(cur[e + 1]));
    m2 = fmaxf(m2, __uint_as_float(cur[e + 2]));
    m3 = fmaxf(m3, __uint_as_float(cur[e + 3]));
  }
}

// Softmax pass 1 of one row: maximum of the 192 raw scores (4 chains); DBG also dumps them (tests).
template <bool DBG>
__device__ __forceinline__ float att3_pass1(uint32_t tb, float* dbg_row) {
  uint32_t va[32], vb[32];
  float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
  tmem_ld_x32(tb, va);
#pragma unroll 1
  for (int jj = 0; jj < 3; ++jj) {
    tmem_ld_x32(tb + (2 * jj + 1) * 32, vb);
    tmem_ld_wait();
    att3_max_chunk(va, m0, m1, m2, m3);
    if (DBG) {
#pragma unroll
      for (int e = 0; e < 32; ++e) dbg_row[(2 * jj) * 32 + e] = __uint_as_float(va[e]);
#pragma unroll
      for (int e = 0; e < 32; ++e) dbg_row[(2 * jj + 1) * 32 + e] = __uint_as_float(vb[e]);
    }
    if (jj < 2) tmem_ld_x32(tb + (2 * jj + 2) * 32, va);
    tmem_ld_wait();
    att3_max_chunk(vb, m0, m1, m2, m3);
  }
  return fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
}

template <bool DBG>
__global__ void __launch_bounds__(kAtt3Threads, 1)
vit_attention3_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmQK64,
                      const __grid_constant__ CUtensorMap tmQK16, const __grid_constant__ CUtensorMap tmO,
                      const AttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kAtt3OffBars);
  uint64_t* qk_full = bars + 0;     // [stage]
  uint64_t* qk_empty = bars + 2;    // [stage]  2 arrivals (one commit per chain)
  uint64_t* v_full = bars + 4;      // [stage]
  uint64_t* v_empty = bars + 6;     // [stage]  2 arrivals
  uint64_t* s_full = bars + 8;      // [chain]
  uint64_t* p_full = bars + 10;     // [chain]  4 arrivals (warps of the group)
  uint64_t* o_full = bars + 12;     // [chain]
  uint64_t* o_empty = bars + 14;    // [chain]  4 arrivals
  uint64_t* turn = bars + 16;       // [chain][lane quarter]  exp-phase token between the two warps of a sub-partition
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 26);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // Q and K arrive as one [192 x 64] SWIZZLE_128B box (dims 0..63: four of the five 16-wide UMMA k-chunks) plus one
  // [192 x 16] SWIZZLE_32B box: 384 TMA row requests per matrix instead of the 960 32-byte requests of five chunk boxes
  // (the MMA issuers spent 15 % of the kernel waiting for the next head's Q, K).  V keeps the five-chunk 3-D view.
  const int nheads = (p.num_problems - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) /
                     static_cast<int>(gridDim.x);

  stamp_start(p.stamp);
  if (warp == 8 && lane == 0) {
    tma_prefetch_desc(&tmQKV);
    tma_prefetch_desc(&tmQK64);
    tma_prefetch_desc(&tmQK16);
    tma_prefetch_desc(&tmO);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&qk_full[i], 1);
      mbar_init(&qk_empty[i], 2);
      mbar_init(&v_full[i], 1);
      mbar_init(&v_empty[i], 2);
      mbar_init(&s_full[i], 1);
      mbar_init(&p_full[i], 4);
      mbar_init(&o_full[i], 1);
      mbar_init(&o_empty[i], 4);
    }
    for (int i = 0; i < 8; ++i) mbar_init(&turn[i], 1);
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

  if (warp == 8) {
    // ---------------------------------------------------------------- TMA producers: lane 0 streams Q,K, lane 1 streams V
    // (two threads so that a V stage still held by the PV MMAs never delays the next Q,K load)
    if (lane < 2) {
      for (int i = 0; i < nheads; ++i) {
        const int prob = blockIdx.x + i * gridDim.x;
        const int b = prob / p.heads, h = prob % p.heads;
        const int st = i & 1;
        const uint32_t ph = (i >> 1) & 1;
        uint8_t* sQ = smem + st * kAtt3StageBytes;
        if (lane == 0) {
          mbar_wait(&qk_empty[st], ph ^ 1);
          mbar_arrive_expect_tx(&qk_full[st], 2 * kAttMatBytes);
          const int cq = h * kAttHeadDim, ck = (p.heads + h) * kAttHeadDim;
          tma_load_2d(sQ, &tmQK64, &qk_full[st], cq, b * kAttTokens);
          tma_load_2d(sQ + kAttWideBytes, &tmQK16, &qk_full[st], cq + 64, b * kAttTokens);
          tma_load_2d(sQ + kAttMatBytes, &tmQK64, &qk_full[st], ck, b * kAttTokens);
          tma_load_2d(sQ + kAttMatBytes + kAttWideBytes, &tmQK16, &qk_full[st], ck + 64, b * kAttTokens);
        } else {
          mbar_wait(&v_empty[st], ph ^ 1);
          mbar_arrive_expect_tx(&v_full[st], kAttMatBytes);
          tma_load_3d(sQ + 2 * kAttMatBytes, &tmQKV, &v_full[st], 0, b * kAttTokens, (2 * p.heads + h) * kAttChunks);
        }
      }
    }
  } else if (warp >= 9) {
    {
      // ---------------------------------------------------------------- MMA issuer of chain g
      // All 32 lanes walk the chain (uniform control flow: ptxas keeps the descriptors in uniform registers and the 5 / 12
      // UTCHMMA of a step issue back to back); one elected lane issues.  With a single active lane every descriptor
      // went through an ELECT / R2UR waterfall loop of ~25 dependent instructions per MMA.
      const int g = warp - 9;
      constexpr uint32_t idesc_s = make_idesc_f16(128, kAttTokens);            // Q K^T : both K-major
      constexpr uint32_t idesc_o = make_idesc_f16(128, kAttHeadDim, 0, 1);     // P V   : V is N-major
      const uint32_t smem_a = smem_u32(smem);
      const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0) + g * kAtt3BufCols;
      for (int i = 0; i < nheads; ++i) {
        const int st = i & 1;
        const uint32_t ph = (i >> 1) & 1;
        const uint32_t sQ = smem_a + st * kAtt3StageBytes;
        const int t = ((i & 1) == g) ? 0 : 1;
        const int row0 = t ? (((i >> 1) & 1) ? 128 : 64) : 0;
        mbar_wait(&o_empty[g], (i & 1) ^ 1);     // the chain's previous tile has drained
        mbar_wait(&qk_full[st], ph);
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int kc = 0; kc < kAttChunks; ++kc) {
            uint64_t da, db;
            if (kc < 4) {           // k-chunk kc = bytes [32 kc, 32 kc + 32) of the 128-byte rows
              da = make_smem_desc(sQ + row0 * 128 + kc * 32, 16, 1024, kSwz128);
              db = make_smem_desc(sQ + kAttMatBytes + kc * 32, 16, 1024, kSwz128);
            } else {
              da = make_smem_desc(sQ + kAttWideBytes + row0 * 32, 16, 256, kSwz32);
              db = make_smem_desc(sQ + kAttMatBytes + kAttWideBytes, 16, 256, kSwz32);
            }
            umma_f16_ss(tb, da, db, idesc_s, kc != 0);
          }
          umma_commit(&s_full[g]);
          umma_commit(&qk_empty[st]);
        }
        __syncwarp();
        mbar_wait(&p_full[g], i & 1);
        mbar_wait(&v_full[st], ph);
        tc_fence_after();
        const uint32_t sV = sQ + 2 * kAttMatBytes;
        // (splitting these into two halves that start under the second half of the exponentials is not possible: O
        // aliases S columns 96..175, which pass 2 is still reading, and the 128 spare TMEM columns cannot hold two Os)
        if (elect_one()) {
#pragma unroll
          for (int ks = 0; ks < kAttTokens / 16; ++ks) {
            const uint64_t db = make_smem_desc(sV + ks * 512, kAttChunkBytes, 256, kSwz32);
            umma_f16_ts(tb + kAtt3ColO, tb + ks * 8, db, idesc_o, ks != 0);
          }
          umma_commit(&o_full[g]);
          umma_commit(&v_empty[st]);
        }
        __syncwarp();
      }
    }
  } else {
    // ------------------------------------------------------------------ softmax + epilogue groups
    const int g = warp >> 2;
    const int q = warp & 3;                  // TMEM lane quarter
    const int trow = q * 32 + lane;          // row inside the 128-row tile == TMEM lane
    const uint32_t tb = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + g * kAtt3BufCols;
    uint8_t* stage_out = smem + kAtt3OffOut + warp * kAtt3OutWarpBytes;
    for (int i = 0; i < nheads; ++i) {
      const int prob = blockIdx.x + i * gridDim.x;
      const int b = prob / p.heads, h = prob % p.heads;
      const int t = ((i & 1) == g) ? 0 : 1;
      const bool low = (i >> 1) & 1;            // tile 1 = rows 128..255, useful lanes 0..63
      const bool active = (t == 0) || (low ? q < 2 : q >= 2);
      const int row0 = t ? (low ? 128 : 64) : 0;
      if (lane == 0) mbar_wait(&s_full[g], i & 1);
      __syncwarp();
      tc_fence_after();
      float sum = 0.f;
      float mo = 0.f;
      if (active) {
        // ---- pass 1: row maximum
        float* dbg_row = DBG ? p.dbg_s + (static_cast<size_t>(prob) * kAttTokens + row0 + trow) * kAttTokens : nullptr;
        mo = att3_pass1<DBG>(tb, dbg_row) * p.scale_log2e;
      }
      // the exp unit belongs to one warp of the sub-partition at a time: two chains left alone run in lock-step
      // (both exponentiate, then both queue for the tensor pipe), which serialises everything again
      if (lane == 0) mbar_wait(&turn[g * 4 + q], g ? (i & 1) : ((i & 1) ^ 1));
      __syncwarp();
      if (active) {
        // ---- pass 2: exponentials, row sum, P (fp16) in place over the consumed S columns
        sum = att3_pass2(tb, p.scale_log2e, mo);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&turn[(g ^ 1) * 4 + q]);
        mbar_arrive(&p_full[g]);
      }
      // ---- epilogue of this tile
      if (lane == 0) mbar_wait(&o_full[g], i & 1);
      __syncwarp();
      tc_fence_after();
      if (active) {
        uint32_t o0[32], o1[32], o2[16];
        tmem_ld_x32(tb + kAtt3ColO, o0);
        tmem_ld_x32(tb + kAtt3ColO + 32, o1);
        tmem_ld_x16(tb + kAtt3ColO + 64, o2);
        tmem_ld_wait();
        tmem_pin(o0);
        tmem_pin(o1);
        tmem_pin(o2);
        // O is in registers: hand the tile buffer back NOW, so that the next tile's S = Q K^T is issued while this warp
        // still converts, stages and stores its rows (the arrive used to sit at the end of the epilogue, ~600 cycles later)
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&o_empty[g]);
        const float inv = 1.0f / sum;
        auto pack8 = [&](const uint32_t* v) {
          uint4 w;
          __half2 a = __floats2half2_rn(__uint_as_float(v[0]) * inv, __uint_as_float(v[1]) * inv);
          __half2 bb = __floats2half2_rn(__uint_as_float(v[2]) * inv, __uint_as_float(v[3]) * inv);
          __half2 c = __floats2half2_rn(__uint_as_float(v[4]) * inv, __uint_as_float(v[5]) * inv);
          __half2 d = __floats2half2_rn(__uint_as_float(v[6]) * inv, __uint_as_float(v[7]) * inv);
          w.x = *reinterpret_cast<uint32_t*>(&a); w.y = *reinterpret_cast<uint32_t*>(&bb);
          w.z = *reinterpret_cast<uint32_t*>(&c); w.w = *reinterpret_cast<uint32_t*>(&d);
          return w;
        };
        // rows of this warp -> dense [32][80] fp16 staging -> one TMA store (a direct store would be 32 scattered
        // 16-byte sectors per instruction and saturates the LSU)
        if (lane == 0) tma_store_wait_read<0>();   // the previous tile's store has finished reading the staging
        __syncwarp();
        uint4* o = reinterpret_cast<uint4*>(stage_out) + lane * (kAttHeadDim / 8);
#pragma unroll
        for (int c = 0; c < 4; ++c) o[c] = pack8(o0 + 8 * c);
#pragma unroll
        for (int c = 0; c < 4; ++c) o[4 + c] = pack8(o1 + 8 * c);
#pragma unroll
        for (int c = 0; c < 2; ++c) o[8 + c] = pack8(o2 + 8 * c);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(&tmO, stage_out, h * kAttHeadDim, b * kAttTokens + row0 + q * 32);
          tma_store_commit();
        }
      } else {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&o_empty[g]);
      }
    }
    if (lane == 0) tma_store_wait_read<0>();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <bool DBG>
inline int attention3_launch_t(const AttnPlan& plan, cudaStream_t st) {
  static bool configured = false;
  if (!configured) {
    THMR_CUDA(cudaFuncSetAttribute(vit_attention3_kernel<DBG>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   kAtt3SmemBytes));
    configured = true;
  }
  vit_attention3_kernel<DBG><<<plan.grid, kAtt3Threads, kAtt3SmemBytes, st>>>(plan.tm, plan.tm_qk64, plan.tm_qk16,
                                                                              plan.tm_out, plan.p);
  THMR_CUDA(cudaGetLastError());
  return THMR_OK;
}

inline int attention3_launch(const AttnPlan& plan, cudaStream_t st) {
  return plan.p.dbg_s ? attention3_launch_t<true>(plan, st) : attention3_launch_t<false>(plan, st);
}

inline int attention_dispatch(const AttnPlan& plan, cudaStream_t st) { return attention3_launch(plan, st); }

}  // namespace thmr
