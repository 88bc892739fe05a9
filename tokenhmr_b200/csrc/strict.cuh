// Strict mode: every contraction of the path at fp32-grade accuracy on the tensor cores.
//
// The reference runs the forward in fp32 (demo.py:35-37,77-78: no autocast).  The default engine rounds both operands
// of every product to fp16 (DESIGN.md §2), which shows as ~2e-4 on the vertices after 32 blocks.  Strict mode keeps
// every activation in fp32 and feeds the SAME tcgen05 GEMM kernels split operands:
//      a * 2^4 = a_hi + a_lo,   w * 2^8 = w_hi + w_lo      (hi = fp16(x), lo = fp16(x - hi): 22 significand bits)
//      a . w  ~=  2^-12 * ( a_hi.w_hi + a_lo.w_hi + a_hi.w_lo )         (the lo.lo term is 2^-22 relative)
// as ONE GEMM with K' = 3K over A' = [a_hi | a_lo | a_hi] and W' = [w_hi | w_hi | w_lo], fp32 accumulation in TMEM.
// The fixed power-of-two scales keep the lo parts out of the fp16 subnormal range for |a| > 2^-6, |w| > 2^-10 (below
// that the absolute error floor is 2^-29 resp. 2^-33) and bound the representable range to |a| < 4094, |w| < 255;
// the weight side is checked at pack time (weights.py), the activation side raises a device flag here.
//
// Kernels in this file: the fp32 -> split-fp16 operand builder (with the consumer's activation fused: exact erf GELU /
// ReLU, so GEMM epilogues stay linear), an fp32 CUDA-core attention (QK^T, softmax and PV never leave fp32), and fp32
// variants of the patch im2col and the decoder's one-query cross-attention.
#pragma once
#include "common.cuh"
#include "elementwise.cuh"
#include "gemm_host.cuh"

namespace thmr {

constexpr float kStrictActScale = 16.0f;    // A side (activations)
constexpr float kStrictWScale = 256.0f;     // B side (weights; packed on the host)
constexpr float kStrictAlpha = 1.0f / (kStrictActScale * kStrictWScale);

__device__ unsigned int g_strict_overflow = 0;

enum : int { kSplitActNone = 0, kSplitActGelu = 1, kSplitActRelu = 2 };

// nn.GELU() (approximate='none'): 0.5 x (1 + erf(x / sqrt(2))), erff = CUDA libm (<= 2 ulp)
__device__ __forceinline__ float gelu_exact(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }

// src fp32 [R, C] (row pitch lds) -> dst fp16 [*, 3C] = [hi | lo | hi] of act(x) * 2^4.
// Optional row remap into zero-padded sequences: source row r = b*T + t  ->  dst row b*pitch + lo + t  (T == 0: identity).
__global__ void __launch_bounds__(256)
split_rows_kernel(const float* __restrict__ src, long lds, __half* __restrict__ dst, long R, int C, int act, int T,
                  int pitch, int lo) {
  const int c4 = C >> 2;
  const long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  if (i >= R * c4) return;
  const long r = i / c4;
  const int c = static_cast<int>(i - r * c4) << 2;
  float4 v = *reinterpret_cast<const float4*>(src + r * lds + c);
  if (act == kSplitActGelu) { v.x = gelu_exact(v.x); v.y = gelu_exact(v.y); v.z = gelu_exact(v.z); v.w = gelu_exact(v.w); }
  else if (act == kSplitActRelu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
  const float f[4] = {v.x * kStrictActScale, v.y * kStrictActScale, v.z * kStrictActScale, v.w * kStrictActScale};
  __half hi[4], lw[4];
  bool over = false;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    over |= !(fabsf(f[e]) <= 65504.0f);       // also catches NaN
    hi[e] = __float2half_rn(f[e]);
    lw[e] = __float2half_rn(f[e] - __half2float(hi[e]));
  }
  if (over) atomicExch(&g_strict_overflow, 1u);
  uint2 phi, plo;
  phi.x = (static_cast<uint32_t>(__half_as_ushort(hi[1])) << 16) | __half_as_ushort(hi[0]);
  phi.y = (static_cast<uint32_t>(__half_as_ushort(hi[3])) << 16) | __half_as_ushort(hi[2]);
  plo.x = (static_cast<uint32_t>(__half_as_ushort(lw[1])) << 16) | __half_as_ushort(lw[0]);
  plo.y = (static_cast<uint32_t>(__half_as_ushort(lw[3])) << 16) | __half_as_ushort(lw[2]);
  const long dr = (T > 0) ? ((r / T) * pitch + lo + r % T) : r;
  __half* o = dst + dr * (3L * C) + c;
  *reinterpret_cast<uint2*>(o) = phi;
  *reinterpret_cast<uint2*>(o + C) = plo;
  *reinterpret_cast<uint2*>(o + 2 * C) = phi;
}

inline int split_rows_launch(const float* src, long lds, __half* dst, long R, int C, int act, int T, int pitch, int lo,
                             cudaStream_t st) {
  THMR_CHECK(C % 4 == 0 && lds % 4 == 0, "split_rows: C=%d lds=%ld must be multiples of 4", C, lds);
  const long n = R * (C / 4);
  split_rows_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(src, lds, dst, R, C, act, T, pitch, lo);
  THMR_CUDA(cudaGetLastError());
  return THMR_OK;
}

// The GEMM over a split operand: sA = split_rows of `rows` rows of K channels, times the split weight f16 [N, taps * 3K]
// (per tap [hi | hi | lo] of w * 2^8, packed on the host); out32 = 2^-12 * acc + bias (+ resid), both with row pitch
// ld32.  taps > 1: implicit conv1d, tap t reads row m + (t - 1) * dil.  seq_len > 0: the rows are sequences of seq_len
// rows with seq_pad zero rows on either side, and the pad rows of the output are written as zero.
inline GemmDesc split_gemm_desc(const __half* sA, long rows, int K, int taps, int dil, const void* Wt, int N,
                                const float* bias, const float* resid, float* o32, int ld32, int seq_len = 0,
                                int seq_pad = 0) {
  const int ks = 3 * K;   // one split row: [hi | lo | hi]
  GemmDesc d;
  d.A = sA; d.lda = ks; d.a_rows = rows;
  d.B = static_cast<const __half*>(Wt); d.ldb = taps * ks;
  d.M = static_cast<int>(rows); d.N = N; d.K = taps * ks;
  d.bias = bias; d.resid = resid; d.ldr = ld32;
  d.out32 = o32; d.ld32 = ld32;
  d.alpha = kStrictAlpha;
  if (taps > 1) { d.taps = taps; d.cin = ks; d.tap_row0 = -dil; d.tap_stride = dil; }
  if (seq_len > 0) { d.seq_pitch = seq_len + 2 * seq_pad; d.seq_lo = seq_pad; d.seq_hi = seq_pad + seq_len; }
  return d;
}

__global__ void relu_inplace_kernel(float* __restrict__ x, long n4) {
  const long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  if (i >= n4) return;
  float4 v = reinterpret_cast<float4*>(x)[i];
  v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
  reinterpret_cast<float4*>(x)[i] = v;
}

// Patch im2col in fp32 (see im2col_patch_kernel): out (B*gh*gw, 3*P*P) fp32.
__global__ void im2col_patch_f32_kernel(const float* __restrict__ img, float* __restrict__ out, int B, int S, int x0,
                                        int Wc, int P, int pad, int gh, int gw) {
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
  float* o = out + row * (3 * P * P) + c * P * P + dy * P;
  const float* src = img + ((static_cast<long>(b) * 3 + c) * S + y) * S + x0;
  for (int dx = 0; dx < P; ++dx) {
    const int x = j * P - pad + dx;
    o[dx] = (y >= 0 && y < S && x >= 0 && x < Wc) ? src[x] : 0.f;
  }
}

// ViT attention core in fp32 (vit.py:116-122): q *= scale; softmax(q k^T) v, per (image, head).
//   qkv fp32 [B*T, ld]: q heads | k heads | v heads, head h at columns h*HD (+ H*HD, + 2*H*HD);  out fp32 [B*T, ldo].
// One block per (image, head), thread = query row; K and V of the head live in shared memory (every thread reads the
// same key row: broadcast), the query row and the output accumulator in registers.  Two passes over the keys (row
// maximum, then exp / sum / PV) so that the softmax is the reference's max-subtracted form.
template <int T, int HD>
__global__ void __launch_bounds__(T, 1)
attention_f32_kernel(const float* __restrict__ qkv, int ld, float* __restrict__ out, int ldo, int H, float scale) {
  extern __shared__ float4 s_kv[];                    // K [T][HD] then V [T][HD]
  float* sK = reinterpret_cast<float*>(s_kv);
  float* sV = sK + T * HD;
  const int b = blockIdx.x / H, h = blockIdx.x % H;
  const float* base = qkv + static_cast<size_t>(b) * T * ld + h * HD;
  constexpr int V4 = HD / 4;
  for (int i = threadIdx.x; i < T * V4; i += T) {
    const int r = i / V4, c = (i % V4) * 4;
    *reinterpret_cast<float4*>(sK + r * HD + c) = *reinterpret_cast<const float4*>(base + static_cast<size_t>(r) * ld + H * HD + c);
    *reinterpret_cast<float4*>(sV + r * HD + c) = *reinterpret_cast<const float4*>(base + static_cast<size_t>(r) * ld + 2 * H * HD + c);
  }
  float q[HD];
  {
    const float* qr = base + static_cast<size_t>(threadIdx.x) * ld;
#pragma unroll
    for (int c = 0; c < HD; c += 4) {
      const float4 v = *reinterpret_cast<const float4*>(qr + c);
      q[c] = v.x * scale; q[c + 1] = v.y * scale; q[c + 2] = v.z * scale; q[c + 3] = v.w * scale;
    }
  }
  __syncthreads();
  auto score = [&](int j) -> float {
    const float4* kr = reinterpret_cast<const float4*>(sK + j * HD);
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
    for (int c = 0; c < V4; ++c) {
      const float4 k = kr[c];
      s0 = fmaf(q[4 * c], k.x, s0); s1 = fmaf(q[4 * c + 1], k.y, s1);
      s2 = fmaf(q[4 * c + 2], k.z, s2); s3 = fmaf(q[4 * c + 3], k.w, s3);
    }
    return (s0 + s1) + (s2 + s3);
  };
  float m = -INFINITY;
#pragma unroll 1
  for (int j = 0; j < T; ++j) m = fmaxf(m, score(j));
  float o[HD];
#pragma unroll
  for (int c = 0; c < HD; ++c) o[c] = 0.f;
  float l = 0.f;
#pragma unroll 1
  for (int j = 0; j < T; ++j) {
    const float p = expf(score(j) - m);
    l += p;
    const float4* vr = reinterpret_cast<const float4*>(sV + j * HD);
#pragma unroll
    for (int c = 0; c < V4; ++c) {
      const float4 v = vr[c];
      o[4 * c] = fmaf(p, v.x, o[4 * c]); o[4 * c + 1] = fmaf(p, v.y, o[4 * c + 1]);
      o[4 * c + 2] = fmaf(p, v.z, o[4 * c + 2]); o[4 * c + 3] = fmaf(p, v.w, o[4 * c + 3]);
    }
  }
  const float inv = 1.0f / l;
  float* orow = out + (static_cast<size_t>(b) * T + threadIdx.x) * ldo + h * HD;
#pragma unroll
  for (int c = 0; c < HD; c += 4)
    *reinterpret_cast<float4*>(orow + c) = make_float4(o[c] * inv, o[c + 1] * inv, o[c + 2] * inv, o[c + 3] * inv);
}

inline int attention_f32_launch(const float* qkv, int ld, int B, int H, float* out, int ldo, float scale, cudaStream_t st) {
  constexpr int T = 192, HD = 80;
  constexpr size_t smem = 2 * T * HD * sizeof(float);
  static bool configured = false;
  if (!configured) {
    THMR_CUDA(cudaFuncSetAttribute(attention_f32_kernel<T, HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = true;
  }
  attention_f32_kernel<T, HD><<<B * H, T, smem, st>>>(qkv, ld, out, ldo, H, scale);
  THMR_CUDA(cudaGetLastError());
  return THMR_OK;
}

// One-query cross-attention of the decoder in fp32 (see dec_cross_attn_kernel): kv fp32, out fp32.
template <int T>
__global__ void __launch_bounds__(T)
dec_cross_attn_f32_kernel(const float* __restrict__ q, const float* __restrict__ kv, int ld, int koff, int voff,
                          float scale, float* __restrict__ out, int heads) {
  __shared__ float sq[64];
  __shared__ float sp[T];
  __shared__ float red[T / 32];
  __shared__ float so[T / 64][64];
  const int b = blockIdx.x / heads;
  const int h = blockIdx.x % heads;
  const int j = threadIdx.x;
  const int lane = j & 31, w = j >> 5;
  const int inner = heads * 64;
  if (j < 64) sq[j] = q[static_cast<size_t>(b) * inner + h * 64 + j];
  __syncthreads();
  const float* kr = kv + (static_cast<size_t>(b) * T + j) * ld + koff + h * 64;
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < 64; c += 4) {
    const float4 k = *reinterpret_cast<const float4*>(kr + c);
    s += sq[c] * k.x + sq[c + 1] * k.y + sq[c + 2] * k.z + sq[c + 3] * k.w;
  }
  s *= scale;
  float m = warp_max(s);
  if (lane == 0) red[w] = m;
  __syncthreads();
  m = red[0];
#pragma unroll
  for (int i = 1; i < T / 32; ++i) m = fmaxf(m, red[i]);
  const float e = expf(s - m);
  float sum = warp_sum(e);
  __syncthreads();
  if (lane == 0) red[w] = sum;
  __syncthreads();
  sum = 0.f;
#pragma unroll
  for (int i = 0; i < T / 32; ++i) sum += red[i];
  sp[j] = e / sum;
  __syncthreads();
  const int d = j & 63, g = j >> 6;
  const float* vb = kv + static_cast<size_t>(b) * T * ld + voff + h * 64 + d;
  float o = 0.f;
  for (int k = g; k < T; k += T / 64) o += sp[k] * vb[static_cast<size_t>(k) * ld];
  so[g][d] = o;
  __syncthreads();
  if (j < 64) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < T / 64; ++i) t += so[i][j];
    out[static_cast<size_t>(b) * inner + h * 64 + j] = t;
  }
}

}  // namespace thmr
