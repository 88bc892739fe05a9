// HBM-bound row kernels: patch im2col, LayerNorm, softmax, gathers.  Warp-shuffle reductions, fp32 math,
// vectorised coalesced loads; outputs are written in the operand format of the consuming tcgen05 GEMM (fp16).
#pragma once
#include "common.cuh"
#include "ptx.cuh"

namespace thmr {

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

// ------------------------------------------------------------------------------------------------
// Patch im2col (vit.py:341-343 crop + PatchEmbed conv as a GEMM, vit.py:168-175)
//   img  (B,3,S,S) fp32 NCHW, cropped to columns [x0, x0+Wc)
//   out  (B*gh*gw, 3*P*P) fp16, k = c*P*P + dy*P + dx, zero outside the cropped image (padding `pad`).
// One thread per (row, c, dy): writes P consecutive fp16 (32 B for P=16).
// ------------------------------------------------------------------------------------------------
__global__ void im2col_patch_kernel(const float* __restrict__ img, __half* __restrict__ out, int B, int S, int x0,
                                    int Wc, int P, int pad, int gh, int gw, unsigned long long* stamp) {
  stamp_start(stamp);
  const long total = static_cast<long>(B) * gh * gw * 3 * P;
  const long t = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  if (t >= total) return;
  const int dy = t % P;
  const int c = (t / P) % 3;
  const long row = t / (3 * P);
  const int j = row % gw;
  const int i = (row / gw) % gh;
  const int b = row / (static_cast<long>(gw) * gh);
  const int y = i * P - pad + dy;
  __half* o = out + row * (3 * P * P) + c * P * P + dy * P;
  const float* src = img + ((static_cast<long>(b) * 3 + c) * S + y) * S + x0;
  for (int dx = 0; dx < P; ++dx) {
    const int x = j * P - pad + dx;
    float v = 0.f;
    if (y >= 0 && y < S && x >= 0 && x < Wc) v = src[x];
    o[dx] = __float2half_rn(v);
  }
}

// ------------------------------------------------------------------------------------------------
// LayerNorm over the last dimension (nn.LayerNorm: biased variance, eps inside the sqrt).
//   x (R,C) fp32 -> y16 (fp16, nullable) and/or y32 (fp32, nullable); optional ReLU (FCBlock, modules.py:15-19).
//   One warp per row; the row lives in registers (C <= 32*4*VEC4 elements), two-pass statistics.
//   out_t > 0: outputs (fp16 and fp32) written transposed inside groups of out_t rows:
//       y16[(r / T) * C * T + c * T + (r % T)]   (MixerLayer token mixing, modules.py:56-59)
//   Row pitch of the fp16 output is ld16 (elements) when not transposed.
// ------------------------------------------------------------------------------------------------
// PLAIN16: the ViT's case (fp16 output only, no ReLU, not transposed, C == 128 * VEC4 exactly), compiled without the other
// output modes' branches and without the per-chunk column guards.
template <int VEC4, bool PLAIN16 = false>  // float4 loads per lane
__global__ void __launch_bounds__(256, VEC4 > 10 ? 2 : 4)
layernorm_reg_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                     __half* __restrict__ y16, int ld16, float* __restrict__ y32_, int R, int C_, float eps, int relu_,
                     int out_t_, unsigned long long* stamp) {
  const int C = PLAIN16 ? VEC4 * 128 : C_;
  float* const y32 = PLAIN16 ? nullptr : y32_;
  const int relu = PLAIN16 ? 0 : relu_;
  const int out_t = PLAIN16 ? 0 : out_t_;
  stamp_start(stamp);
  // gamma/beta staged in shared memory once per (persistent) block: read from global inside the output loop they
  // were the largest stall of the kernel (an L2-latency load per 4 outputs, after the reductions)
  extern __shared__ float4 s_gb[];   // [2][C/4]
  float4* sg = s_gb;
  float4* sb = s_gb + C / 4;
  for (int c = threadIdx.x; c < C / 4; c += blockDim.x) {
    sg[c] = reinterpret_cast<const float4*>(gamma)[c];
    sb[c] = reinterpret_cast<const float4*>(beta)[c];
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int warps_total = (gridDim.x * blockDim.x) >> 5;
  auto load_row = [&](float4 (&v)[VEC4], int row) {
    const float* xr = x + static_cast<size_t>(row) * C;
#pragma unroll
    for (int i = 0; i < VEC4; ++i) {
      const int c = (i * 32 + lane) * 4;
      v[i] = (PLAIN16 || c < C) ? *reinterpret_cast<const float4*>(xr + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  // persistent warps: the grid is sized to the resident capacity and every warp walks rows with a grid stride
  for (int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; warp < R; warp += warps_total) {
    float4 v[VEC4];
    load_row(v, warp);
    // Packed fp32 (FFMA2: two IEEE lanes per instruction) for the three arithmetic passes: the kernel issues ~320
    // instructions per lane and row and sits at 60 % issue utilisation next to its HBM stalls (ncu); packing takes it to ~200.
    // Rows shorter than the register tile hold zeros beyond C (they add 0 to the sum; the variance pass masks them).
    uint64_t s2 = f2_pack(0.f, 0.f);
#pragma unroll
    for (int i = 0; i < VEC4; ++i) {
      s2 = f2_add(s2, f2_pack(v[i].x, v[i].y));
      s2 = f2_add(s2, f2_pack(v[i].z, v[i].w));
    }
    float s_lo, s_hi;
    f2_unpack(s2, s_lo, s_hi);
    const float mean = warp_sum(s_lo + s_hi) / C;
    const uint64_t nmean2 = f2_pack(-mean, -mean);
    uint64_t q2 = f2_pack(0.f, 0.f);
#pragma unroll
    for (int i = 0; i < VEC4; ++i) {
      const int c = (i * 32 + lane) * 4;
      if (PLAIN16 || c < C) {
        const uint64_t d0 = f2_add(f2_pack(v[i].x, v[i].y), nmean2);
        const uint64_t d1 = f2_add(f2_pack(v[i].z, v[i].w), nmean2);
        q2 = f2_fma(d0, d0, q2);
        q2 = f2_fma(d1, d1, q2);
      }
    }
    float q_lo, q_hi;
    f2_unpack(q2, q_lo, q_hi);
    const float rstd = rsqrtf(warp_sum(q_lo + q_hi) / C + eps);
    const uint64_t rstd2 = f2_pack(rstd, rstd);
#pragma unroll
    for (int i = 0; i < VEC4; ++i) {
      const int c = (i * 32 + lane) * 4;
      if (PLAIN16 || c < C) {
        const float4 g = sg[c >> 2];
        const float4 bb = sb[c >> 2];
        // ((x - mean) * rstd) * g + b, the reference's order of operations
        const uint64_t t0 = f2_mul(f2_add(f2_pack(v[i].x, v[i].y), nmean2), rstd2);
        const uint64_t t1 = f2_mul(f2_add(f2_pack(v[i].z, v[i].w), nmean2), rstd2);
        const uint64_t o0 = f2_fma(t0, f2_pack(g.x, g.y), f2_pack(bb.x, bb.y));
        const uint64_t o1 = f2_fma(t1, f2_pack(g.z, g.w), f2_pack(bb.z, bb.w));
        float4 o;
        f2_unpack(o0, o.x, o.y);
        f2_unpack(o1, o.z, o.w);
        if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
        if (y32) {
          if (out_t > 0) {   // transposed inside groups of out_t rows, like the fp16 output (strict mode operand)
            float* base = y32 + static_cast<size_t>(warp / out_t) * C * out_t + (warp % out_t);
            base[static_cast<size_t>(c) * out_t] = o.x;
            base[static_cast<size_t>(c + 1) * out_t] = o.y;
            base[static_cast<size_t>(c + 2) * out_t] = o.z;
            base[static_cast<size_t>(c + 3) * out_t] = o.w;
          } else {
            *reinterpret_cast<float4*>(y32 + static_cast<size_t>(warp) * C + c) = o;
          }
        }
        if (y16) {
          if (out_t > 0) {
            __half* base = y16 + static_cast<size_t>(warp / out_t) * C * out_t + (warp % out_t);
            base[static_cast<size_t>(c) * out_t] = __float2half_rn(o.x);
            base[static_cast<size_t>(c + 1) * out_t] = __float2half_rn(o.y);
            base[static_cast<size_t>(c + 2) * out_t] = __float2half_rn(o.z);
            base[static_cast<size_t>(c + 3) * out_t] = __float2half_rn(o.w);
          } else {
            __half2 h0 = __floats2half2_rn(o.x, o.y), h1 = __floats2half2_rn(o.z, o.w);
            uint2 pk;
            pk.x = *reinterpret_cast<uint32_t*>(&h0);
            pk.y = *reinterpret_cast<uint32_t*>(&h1);
            *reinterpret_cast<uint2*>(y16 + static_cast<size_t>(warp) * ld16 + c) = pk;
          }
        }
      }
    }
  }
}

// Wide rows (C up to 64K, e.g. the 10240-wide FCBlock norm): one block per row, three passes over L1/L2.
__global__ void __launch_bounds__(256)
layernorm_wide_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                      __half* __restrict__ y16, int ld16, float* __restrict__ y32, int R, int C, float eps, int relu,
                      unsigned long long* stamp) {
  stamp_start(stamp);
  __shared__ float red[8];
  __shared__ float bcast;
  const int row = blockIdx.x;
  const float* xr = x + static_cast<size_t>(row) * C;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  auto block_sum = [&](float v) -> float {
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) red[w] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
      for (int i = 0; i < 8; ++i) t += red[i];
      bcast = t;
    }
    __syncthreads();
    return bcast;
  };
  float s = 0.f;
  for (int c = threadIdx.x; c < C; c += 256) s += xr[c];
  const float mean = block_sum(s) / C;
  float q = 0.f;
  for (int c = threadIdx.x; c < C; c += 256) { const float d = xr[c] - mean; q += d * d; }
  const float rstd = rsqrtf(block_sum(q) / C + eps);
  for (int c = threadIdx.x; c < C; c += 256) {
    float o = (xr[c] - mean) * rstd * gamma[c] + beta[c];
    if (relu) o = fmaxf(o, 0.f);
    if (y32) y32[static_cast<size_t>(row) * C + c] = o;
    if (y16) y16[static_cast<size_t>(row) * ld16 + c] = __float2half_rn(o);
  }
}

inline int layernorm_launch(const float* x, const float* gamma, const float* beta, __half* y16, int ld16, float* y32,
                            int R, int C, float eps, int relu, int out_t, cudaStream_t st,
                            unsigned long long* stamp = nullptr) {
  THMR_CHECK(C % 4 == 0, "layernorm: C=%d not a multiple of 4", C);
  if (ld16 == 0) ld16 = C;
  if (C <= 2048) {
    // Persistent warps walk the rows with a grid stride over 4 resident blocks of 256 threads per SM.  (Launch shapes that
    // divide the rows more evenly were measured and are not faster: the kernel is not tail-bound.)
    constexpr int threads = 256;
    const int rows_per_block = threads / 32;
    int grid = (R + rows_per_block - 1) / rows_per_block;
    const int resident = num_sms() * 4;
    if (grid > resident) grid = resident;
    const size_t smem = 2 * static_cast<size_t>(C) * sizeof(float);
    const int vec4 = (C / 4 + 31) / 32;
    // register tile of 1, 8, 10 or 16 float4 per lane; [1] = the PLAIN16 form, for rows that fill the tile exactly
    using LnKernel = void (*)(const float*, const float*, const float*, __half*, int, float*, int, int, float, int, int,
                              unsigned long long*);
    const int tile[4] = {1, 8, 10, 16};
    const LnKernel kernels[4][2] = {{layernorm_reg_kernel<1>, layernorm_reg_kernel<1, true>},
                                    {layernorm_reg_kernel<8>, layernorm_reg_kernel<8, true>},
                                    {layernorm_reg_kernel<10>, layernorm_reg_kernel<10, true>},
                                    {layernorm_reg_kernel<16>, layernorm_reg_kernel<16, true>}};
    const int ti = vec4 <= 1 ? 0 : vec4 <= 8 ? 1 : vec4 <= 10 ? 2 : 3;
    const bool plain16 = y16 && !y32 && !relu && out_t == 0 && C == 128 * vec4 && vec4 == tile[ti];
    kernels[ti][plain16 ? 1 : 0]<<<grid, threads, smem, st>>>(x, gamma, beta, y16, ld16, y32, R, C, eps, relu, out_t,
                                                               stamp);
  } else {
    THMR_CHECK(out_t == 0, "layernorm: transposed output needs C <= 2048");
    layernorm_wide_kernel<<<R, 256, 0, st>>>(x, gamma, beta, y16, ld16, y32, R, C, eps, relu, stamp);
  }
  THMR_CUDA(cudaGetLastError());
  return THMR_OK;
}

// ------------------------------------------------------------------------------------------------
// Row softmax over C = 32*4*VEC4 classes (token_classifier.py:104): logits fp32 -> probs fp32 (the
// cls_logits_softmax output) + an fp16 copy laid out for the soft-codebook GEMM (quantize_cnn.py:92-93),
// whose rows live in zero-padded sequences: row r = b*T + t  ->  p16 row b*pitch + lo + t.
// ------------------------------------------------------------------------------------------------
template <int VEC4>
__global__ void __launch_bounds__(256)
softmax_rows_kernel(const float* __restrict__ logits, float* __restrict__ p32, __half* __restrict__ p16, int R, int C,
                    int T, int pitch, int lo) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= R) return;
  const float* xr = logits + static_cast<size_t>(warp) * C;
  float4 v[VEC4];
  float m = -INFINITY;
#pragma unroll
  for (int i = 0; i < VEC4; ++i) {
    const int c = (i * 32 + lane) * 4;
    v[i] = (c < C) ? *reinterpret_cast<const float4*>(xr + c) : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    m = fmaxf(m, fmaxf(fmaxf(v[i].x, v[i].y), fmaxf(v[i].z, v[i].w)));
  }
  m = warp_max(m);
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < VEC4; ++i) {
    v[i].x = expf(v[i].x - m); v[i].y = expf(v[i].y - m); v[i].z = expf(v[i].z - m); v[i].w = expf(v[i].w - m);
    s += v[i].x + v[i].y + v[i].z + v[i].w;
  }
  const float inv = 1.0f / warp_sum(s);
  const size_t prow = (T > 0) ? (static_cast<size_t>(warp / T) * pitch + lo + warp % T) : warp;
#pragma unroll
  for (int i = 0; i < VEC4; ++i) {
    const int c = (i * 32 + lane) * 4;
    if (c < C) {
      float4 o = make_float4(v[i].x * inv, v[i].y * inv, v[i].z * inv, v[i].w * inv);
      if (p32) *reinterpret_cast<float4*>(p32 + static_cast<size_t>(warp) * C + c) = o;
      if (p16) {
        __half2 h0 = __floats2half2_rn(o.x, o.y), h1 = __floats2half2_rn(o.z, o.w);
        uint2 pk;
        pk.x = *reinterpret_cast<uint32_t*>(&h0);
        pk.y = *reinterpret_cast<uint32_t*>(&h1);
        *reinterpret_cast<uint2*>(p16 + prow * C + c) = pk;
      }
    }
  }
}

inline int softmax_rows_launch(const float* logits, float* p32, __half* p16, int R, int C, int T, int pitch, int lo,
                               cudaStream_t st) {
  THMR_CHECK(C % 4 == 0 && C <= 2048, "softmax: C=%d unsupported", C);
  const int grid = (R + 7) / 8;
  softmax_rows_kernel<16><<<grid, 256, 0, st>>>(logits, p32, p16, R, C, T, pitch, lo);
  THMR_CUDA(cudaGetLastError());
  return THMR_OK;
}

// ------------------------------------------------------------------------------------------------
// nn.Upsample(size) nearest on zero-padded channels-last sequences (vanilla_pose_vqvae.py:139-141):
//   dst (B, Lout + 2*pad, C) <- src (B, Lin + 2*pad, C),   dst[b, pad + j] = src[b, pad + idx[j]]
// idx[j] = floor(j * (Lin/Lout)) computed in fp32 like ATen's legacy 'nearest'.  Pad rows are zeroed.
// ------------------------------------------------------------------------------------------------
__global__ void upsample_rows_kernel(const __half* __restrict__ src, __half* __restrict__ dst, int B, int Lin, int Lout,
                                     int pad, int C8 /* C/8 */) {
  const long total = static_cast<long>(B) * (Lout + 2 * pad) * C8;
  const long t = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  if (t >= total) return;
  const int c8 = t % C8;
  const long row = t / C8;
  const int r = row % (Lout + 2 * pad);
  const int b = row / (Lout + 2 * pad);
  uint4 v = make_uint4(0, 0, 0, 0);
  if (r >= pad && r < pad + Lout) {
    const float scale = static_cast<float>(Lin) / static_cast<float>(Lout);
    int si = static_cast<int>(floorf(static_cast<float>(r - pad) * scale));
    si = si < Lin - 1 ? si : Lin - 1;
    v = reinterpret_cast<const uint4*>(src)[(static_cast<long>(b) * (Lin + 2 * pad) + pad + si) * C8 + c8];
  }
  reinterpret_cast<uint4*>(dst)[row * C8 + c8] = v;
}

// Mixer glue (modules.py:55-63):  out = x + y^T (+ z), where yT (B, H, T) fp32 is the token-mix MLP output
// in its transposed layout and z (B*T, H) fp32 the channel-mix output.  x, out: (B*T, H).
__global__ void mixer_add_kernel(const float* __restrict__ x, const float* __restrict__ yT, const float* __restrict__ z,
                                 float* __restrict__ out, int B, int T, int H) {
  const long total = static_cast<long>(B) * T * H;
  const long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  if (i >= total) return;
  const int h = i % H;
  const int t = (i / H) % T;
  const int b = i / (static_cast<long>(H) * T);
  float v = x[i] + yT[(static_cast<long>(b) * H + h) * T + t];
  if (z) v += z[i];
  out[i] = v;
}

// fp32 -> fp16 cast (GEMM operand format), 4 elements per thread.
__global__ void cast_f16_kernel(const float* __restrict__ in, __half* __restrict__ out, long n4) {
  const long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  if (i >= n4) return;
  const float4 v = reinterpret_cast<const float4*>(in)[i];
  __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
  uint2 pk;
  pk.x = *reinterpret_cast<uint32_t*>(&h0);
  pk.y = *reinterpret_cast<uint32_t*>(&h1);
  reinterpret_cast<uint2*>(out)[i] = pk;
}

// Broadcast one fp32 row to R rows (the constant decoder query token, pose_transformer.py:350,354).
__global__ void broadcast_row_kernel(const float* __restrict__ row, float* __restrict__ out, int R, int C) {
  const long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  if (i < static_cast<long>(R) * C) out[i] = row[i % C];
}

}  // namespace thmr
