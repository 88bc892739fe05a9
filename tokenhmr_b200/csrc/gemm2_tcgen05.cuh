// CTA-pair tcgen05 GEMM (cta_group::2): two CTAs of a cluster compute one 256 x 256 output tile.
//
// Why: with one CTA per 128 x 256 tile every k-block moves 48 KB of operands through L2 -> SM for 128*256*64
// MACs; the profile (profiles/r1_gemm_ncu.md) shows the tensor pipe waiting on that feed.  In a pair each CTA
// stages its own 128 rows of A plus only HALF of the B tile (128 of the 256 weight rows) and the UMMA reads the
// other half from the peer's shared memory: 32 KB per k-block per SM for the same MACs, 1.5x less L2 traffic.
//
//   both CTAs : warp 0 TMA producer (own A rows, own half of B; bytes credited to the LEADER's full barrier)
//               warps 4-11 epilogue of the CTA's own 128 accumulator rows (own TMEM)
//   leader    : warp 9 (all lanes walk the pipeline, one elected lane issues) tcgen05.mma.cta_group::2 (M = 256, N = 256) and multicasts the completion to the
//               "smem slot free" and "accumulator ready" barriers of both CTAs
//   peer      : its epilogue warps release the accumulator buffer by arriving on the leader's barrier
//
// Only the TMA epilogues are supported here (fp16 store, fp32 store, fp32 reduce-add); everything else runs on the
// single-CTA kernel.  The reduce-add flavour supports stream-K (partial tiles add into the output in L2, in a fixed
// order).
#pragma once
#include "gemm_tcgen05.cuh"

namespace thmr {

constexpr int kG2BN = 256;
constexpr int kG2Stages = 6;
constexpr uint32_t kG2ABytes = kGemmBM * kGemmBK * 2;        // 16 KB: this CTA's 128 rows of A
constexpr uint32_t kG2BBytes = (kG2BN / 2) * kGemmBK * 2;    // 16 KB: this CTA's half of the B tile
constexpr uint32_t kG2StageBytes = kG2ABytes + kG2BBytes;
constexpr uint32_t kG2StagingOffset = kG2Stages * kG2StageBytes;
constexpr uint32_t kG2BarOffset = kG2StagingOffset + kGemmEpiWarps * 4096;
constexpr uint32_t kG2BiasOffset = kG2BarOffset + 256;       // [2 column halves][128] fp32 bias of the current tile
constexpr uint32_t kG2SmemTotal = kG2BiasOffset + 1024 + 1024;
static_assert(kG2SmemTotal <= 232448, "CTA-pair GEMM shared memory exceeds 227 KB");

// Work decomposition shared by the three warp roles of a cluster (all of them walk the same item sequence).
//   classic : whole tiles round-robin over the clusters, column tile fastest (clusters running side by side share
//             A row blocks and weight column blocks in L2).
//   stream-K: whole tiles quantise badly when tiles / clusters is small -- proj / fc2 have 240 tiles on 74 clusters, i.e.
//             3.24 waves rounded up to 4.  Hybrid schedule: the first floor(tiles / clusters) - 1 rounds run classic
//             (148 tiles); the k-blocks of the remaining tiles (92 tiles = 1.24 per cluster) are cut into one contiguous
//             range per cluster, so every cluster does the same amount of tensor work.  A range boundary inside a tile
//             splits it between cluster c (head k-blocks, at the END of its range) and cluster c+1 (tail k-blocks, at the
//             START of its range); both partial sums go into the output through the reduce-add epilogue, the head part
//             strictly after the tail part (GemmParams::sk_flags), so the result does not depend on timing.  Ranges
//             are at least one tile long, hence at most two clusters per tile.
//             (Cutting ALL k-blocks into per-cluster ranges was measured first: the clusters then walk 74 different A row
//             blocks at any time, A is re-read from HBM once per column tile, fc2 159 us vs 139 us classic.)
struct G2Work {
  int tiles_m, tiles_n, num_kb;
  int tile, dp_tiles, stride;                    // classic phase: tile index, < dp_tiles
  int u, u_end;                                  // stream-K phase: units (k-blocks) of tiles [dp_tiles, tiles) of this cluster
  int cur_tile, cur_m, cur_n, cur_kb0, cur_kb1;  // the current item
  __device__ void load() {
    if (tile < dp_tiles) {
      cur_tile = tile;
      cur_kb0 = 0;
      cur_kb1 = num_kb;
    } else {
      const int t = u / num_kb;
      cur_tile = dp_tiles + t;
      cur_kb0 = u - t * num_kb;
      const int rest = u_end - t * num_kb;
      cur_kb1 = rest < num_kb ? rest : num_kb;
    }
    cur_m = cur_tile / tiles_n;
    cur_n = cur_tile - cur_m * tiles_n;
  }
  // sk_tiles = number of trailing tiles scheduled stream-K (0 = all classic); the host guarantees sk_tiles >= nclusters
  // and sk_tiles * num_kb * nclusters < 2^31
  __device__ G2Work(int sk_tiles, int tm, int tn, int nkb, int cluster, int nclusters)
      : tiles_m(tm), tiles_n(tn), num_kb(nkb), tile(cluster), dp_tiles(tm * tn - sk_tiles), stride(nclusters), u(0),
        u_end(0) {
    if (sk_tiles > 0) {
      const long long total = static_cast<long long>(sk_tiles) * nkb;
      u = static_cast<int>(total * cluster / nclusters);
      u_end = static_cast<int>(total * (cluster + 1) / nclusters);
    }
    load();
  }
  __device__ bool valid() const { return tile < dp_tiles || u < u_end; }
  __device__ void next() {
    if (tile < dp_tiles) tile += stride;
    else u = (cur_tile - dp_tiles) * num_kb + cur_kb1;
    load();
  }
  __device__ bool in_streamk() const { return tile >= dp_tiles; }
  __device__ int tile_index() const { return cur_tile; }
  __device__ int m_blk() const { return cur_m; }
  __device__ int n_blk() const { return cur_n; }
  __device__ int kb0() const { return cur_kb0; }
  __device__ int kb1() const { return cur_kb1; }
};

template <int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGemmThreads, 1)
gemm_f16_tn_2cta_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                        const __grid_constant__ CUtensorMap tmC, const GemmParams p) {
  static_assert(EPI == kEpiStore16 || EPI == kEpiAdd32 || EPI == kEpiStore32, "CTA-pair GEMM supports the TMA epilogues only");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kG2BarOffset);   // used in the leader only
  uint64_t* empty_bar = full_bar + kG2Stages;
  uint64_t* tfull_bar = empty_bar + kG2Stages;
  uint64_t* tempty_bar = tfull_bar + 2;                                     // used in the leader only
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int cluster_id = blockIdx.x >> 1;
  const int num_clusters = gridDim.x >> 1;

  const int tiles_m = (p.M + 2 * kGemmBM - 1) / (2 * kGemmBM);
  const int tiles_n = (p.N + kG2BN - 1) / kG2BN;
  const int num_kb = (p.K + kGemmBK - 1) / kGemmBK;
  const int sk_tiles = (EPI == kEpiAdd32 && p.sk_flags != nullptr) ? p.sk_tiles : 0;

  stamp_start(p.stamp);
  if (warp == kWarpTma && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmC);
  }
  if (warp == kWarpMma && lane == 0) {
    for (int s = 0; s < kG2Stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], 2 * kGemmEpiWarps);   // epilogue warps of both CTAs
    }
    fence_mbar_init();
  }
  if (warp == kWarpAlloc) {
    tmem_alloc_2sm(tmem_slot, 512);
    tmem_relinquish_2sm();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();     // peer barriers initialised, both TMEM allocations done
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kWarpTma) {
    if (lane == 0) {
      // ------------------------------------------------------------ TMA producer (both CTAs)
      int stage = 0;
      uint32_t phase = 0;
      for (G2Work w(sk_tiles, tiles_m, tiles_n, num_kb, cluster_id, num_clusters); w.valid(); w.next()) {
        const int m0 = w.m_blk() * 2 * kGemmBM + static_cast<int>(rank) * kGemmBM;
        const int n0 = w.n_blk() * kG2BN + static_cast<int>(rank) * (kG2BN / 2);
        const int kb0 = w.kb0();
        const int kb1 = w.kb1();
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * kG2StageBytes;
          uint8_t* sb = sa + kG2ABytes;
          if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * kG2StageBytes);
          tma_load_2d_2sm(sa, &tmA, &full_bar[stage], kb * kGemmBK, m0);
          tma_load_2d_2sm(sb, &tmB, &full_bar[stage], kb * kGemmBK, n0);
          if (++stage == kG2Stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == kWarpMma) {
    if (rank == 0) {
      // ---------------------------------------------------------- MMA issuer (leader CTA), warp-converged
      // The whole warp walks the pipeline, so control flow is uniform and ptxas keeps the shared-memory and instruction
      // descriptors in uniform registers: four UTCHMMA issue back to back.  (With a single active lane every descriptor
      // went through an ELECT / R2UR waterfall loop, ~85 dependent instructions per k-block: the issuing thread itself
      // was the critical path -- its counters showed < 3 % of its time waiting for operands or accumulators.)
      // One elected lane issues the tcgen05 instructions.  The barriers waited on here are signalled by TMA
      // complete_tx, tcgen05.commit and remote arrives that guard TMEM, never generic-proxy data, so the waits use the
      // default .cta scope (an .acquire.cluster probe makes ptxas invalidate L1 after every success).
      constexpr uint32_t idesc = make_idesc_f16(2 * kGemmBM, kG2BN);
      const uint32_t smem_base = smem_u32(smem);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      bool ready = false;
      for (G2Work w(sk_tiles, tiles_m, tiles_n, num_kb, cluster_id, num_clusters); w.valid(); w.next()) {
        const int kb0 = w.kb0();
        const int kb1 = w.kb1();
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_u + acc * kG2BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          if (!ready) mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_base + stage * kG2StageBytes;
          const uint32_t sb = sa + kG2ABytes;
          const int nstage = (stage + 1 == kG2Stages) ? 0 : stage + 1;
          const uint32_t nphase = (stage + 1 == kG2Stages) ? (phase ^ 1) : phase;
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < kGemmBK / 16; ++k) {
              const uint64_t da = make_smem_desc(sa + k * 32, 16, 1024, kSwz128);
              const uint64_t db = make_smem_desc(sb + k * 32, 16, 1024, kSwz128);
              umma_f16_ss_2sm(d_tmem, da, db, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
            }
            umma_commit_2sm_mcast(&empty_bar[stage], 3);
            if (kb == kb1 - 1) umma_commit_2sm_mcast(&tfull_bar[acc], 3);
          }
          __syncwarp();
          ready = __all_sync(0xffffffffu, mbar_try_wait(&full_bar[nstage], nphase));   // peek the next stage (a hint)
          stage = nstage;
          phase = nphase;
        }
        if ((acc ^= 1) == 0) acc_phase ^= 1;
      }
    }
  } else if (warp < kGemmEpiWarps) {
    // -------------------------------------------------------------- epilogue (both CTAs, own 128 rows)
    const int q = warp & 3;
    const int half = warp >> 2;
    const uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
    constexpr int kChunkCols = (EPI == kEpiStore16) ? 64 : 32;
    constexpr int kChunksPerHalf = kG2BN / kChunkCols / 2;
    uint8_t* stage_buf = smem + kG2StagingOffset + warp * 4096;
    // Slab stores: the four row-quarter warps of a column half stage their 32 rows side by side (their 4 KB buffers are
    // contiguous and share the 128B-swizzle phase), meet at a named barrier and ONE thread issues a 128-row TMA store:
    // 4 (fp16) / 8 (fp32) TMA operations per tile and CTA instead of 16 / 32.
    uint8_t* slab_buf = smem + kG2StagingOffset + half * 4 * 4096;
    // Bias of the tile's column half in shared memory (fp16 epilogue): each of the half's four warps writes the same 128
    // values and reads them back as broadcast 16-byte loads -- one LDS per 4 columns instead of 4 shuffles.  The named
    // barriers of the slab stores keep the four warps inside the same tile, so one buffer per half is enough: nobody
    // reads the previous tile's bias after the last chunk's barrier.
    float* sbias = reinterpret_cast<float*>(smem + kG2BiasOffset) + half * 128;
    const uint32_t srow = smem_u32(stage_buf) + lane * 128;
    const int sw = lane & 7;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (G2Work w(sk_tiles, tiles_m, tiles_n, num_kb, cluster_id, num_clusters); w.valid(); w.next()) {
      const int m0 = w.m_blk() * 2 * kGemmBM + static_cast<int>(rank) * kGemmBM;
      const int n0 = w.n_blk() * kG2BN;
      const bool add_bias = p.bias && w.kb0() == 0;
      // stream-K ordering of a tile shared by two clusters: the tail part (kb0 > 0) lands first and raises the flag,
      // the head part (kb1 < num_kb) waits for it, then clears it for the next launch.  One flag per store-issuing
      // thread (cta rank x column half): each covers exactly the output block that thread reduce-adds.
      const bool sk_item = w.in_streamk();
      const bool sk_head = sk_item && w.kb1() < num_kb;
      const bool sk_tail = sk_item && w.kb0() > 0;
      unsigned int* sk_flag = sk_item ? p.sk_flags + (static_cast<size_t>(w.tile_index()) * 2 + rank) * 2 + half : nullptr;
      bool sk_waited = false;
      // this warp's 128 bias values (lane l: columns 4l..4l+3 of its column half), fetched while the MMAs run
      float4 bq = make_float4(0.f, 0.f, 0.f, 0.f);
      {
        const int bc = n0 + half * (kG2BN / 2) + lane * 4;
        if (add_bias && lane * 4 < kG2BN / 2 && bc < p.N) bq = __ldg(reinterpret_cast<const float4*>(p.bias + bc));
      }
      if constexpr (EPI == kEpiStore16) {
        *reinterpret_cast<float4*>(sbias + lane * 4) = bq;
        __syncwarp();
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
          // packed fp32 path: bias add, GELU and the fp16 conversion two columns at a time
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            uint32_t v[32];
            tmem_ld_x32(tmem_base + lane_addr + acc * kG2BN + c * 64 + hh * 32, v);
            tmem_ld_wait();
            uint64_t f2[16];
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 b4 = *reinterpret_cast<const float4*>(sbias + cc * 64 + hh * 32 + j);   // broadcast
              f2[j >> 1] = f2_add(f2_pack(__uint_as_float(v[j]), __uint_as_float(v[j + 1])), f2_pack(b4.x, b4.y));
              f2[(j >> 1) + 1] = f2_add(f2_pack(__uint_as_float(v[j + 2]), __uint_as_float(v[j + 3])), f2_pack(b4.z, b4.w));
            }
            if (p.act == kActGelu) {
#pragma unroll
              for (int j = 0; j < 16; ++j) f2[j] = gelu_erf2(f2[j]);
            } else if (p.act == kActRelu) {
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                float a, b;
                f2_unpack(f2[j], a, b);
                f2[j] = f2_pack(fmaxf(a, 0.f), fmaxf(b, 0.f));
              }
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              float a, b;
              f2_unpack(f2[j], a, b);
              __half2 h2 = __floats2half2_rn(a, b);
              pk[hh * 16 + j] = *reinterpret_cast<uint32_t*>(&h2);
            }
          }
        } else {
          uint32_t v[32];
          tmem_ld_x32(tmem_base + lane_addr + acc * kG2BN + c * 32, v);
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
        if (q == 0 && lane == 0) tma_store_wait_read<0>();     // the previous slab has been read out of smem
        named_bar_sync_128(1 + half);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(srow + ((j ^ sw) << 4)), "r"(pk[4 * j]),
                       "r"(pk[4 * j + 1]), "r"(pk[4 * j + 2]), "r"(pk[4 * j + 3])
                       : "memory");
        }
        fence_proxy_async_smem();
        named_bar_sync_128(1 + half);
        if (q == 0 && lane == 0 && col0 < p.N && m0 < p.M) {
          if constexpr (EPI == kEpiStore16) tma_store_2d(&tmC, slab_buf, col0, m0);
          else if constexpr (EPI == kEpiStore32) tma_store_2d(&tmC, slab_buf, col0, m0);
          else {
            if (sk_head && !sk_waited) {
              uint32_t it = 0;
              while (ld_acquire_gpu(sk_flag) == 0u && ++it < kSpinLimit) {}
              if (it >= kSpinLimit) atomicExch(&g_pipeline_timeout, 1u);
              *sk_flag = 0u;                      // consumed: ready for the next launch
              fence_proxy_async_all();
              sk_waited = true;
            }
            tma_reduce_add_2d(&tmC, slab_buf, col0, m0);
          }
          tma_store_commit();
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(&tempty_bar[acc], 0);   // accumulator buffer free (leader's barrier)
      if ((acc ^= 1) == 0) acc_phase ^= 1;
      if (sk_tail && q == 0 && lane == 0) {
        // every reduce-add of this partial tile has been performed in L2: let the head part go
        tma_store_wait<0>();
        fence_proxy_async_all();
        __threadfence();
        st_release_gpu(sk_flag, 1u);
      }
    }
    if (lane == 0) tma_store_wait<0>();
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();     // neither CTA may exit (or free TMEM) while the peer can still reach it
  if (warp == kWarpAlloc) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, 512);
  }
}

}  // namespace thmr
