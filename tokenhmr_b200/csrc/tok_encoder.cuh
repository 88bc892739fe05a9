// Tokenizer encoder + hard quantisation (SURVEY §8 row f4): EncodeTokens.forward
// (tokenization/models/vanilla_pose_vqvae.py:304-346) = PoseSPEncoderV1.encoder (:42-111) followed by
// QuantizeEMAReset.preprocess / quantize (tokenization/models/quantize_cnn.py:74-86).
//
//   pose6d (B,21,6) -> Conv1d(6,W,3)+ReLU -> Upsample(40) Conv+ReLU -> [Upsample(x2) Conv+ReLU] x (mul-1)
//   -> Conv1d(W,W,4,stride 2,pad 1) -> Resnet1D(depth, dilation rate^d, reversed) -> Conv1d(W,code_dim,3)
//   -> (B*T, code_dim) -> argmin_k |x - c_k|^2 -> code_idx (B*T,) int64        (T = 20 * 2^mul / 2 = 160)
//
// The output is an INDEX: it has to equal the fp32 reference's, so the whole operator runs in split precision
// (strict.cuh): activations stay fp32, every convolution is the tcgen05 implicit GEMM over split-fp16 operands
// (3 products, ~2^-21 relative), the quantiser is the split-fp16 distance GEMM with the running arg-min in its epilogue.
// (Round 1 ran the convolutions with plain fp16 operands: latents within 3e-3, but 3 % of the indices moved.)
// Sequences are channels-last and zero-padded, [B, L + 2*kEncPad, C].  Two layers need a gather first:
//   * the 6 input channels are zero-padded to 64 (one 128-byte TMA row per tap);
//   * the stride-2, 4-tap down-sampling conv reads rows 2j-1 .. 2j+2: those four rows are gathered side by side
//     into one [B*(Lout+2 pad), 4W] operand (tap-major, like the repacked weight) and the conv becomes a plain GEMM.
// Activations (ReLU) are applied by the consumer's operand split, so buffers hold pre-activation values.
// Batches are processed in chunks of kEncChunk poses to bound the workspace.
#pragma once
#include "common.cuh"
#include "elementwise.cuh"
#include "gemm_host.cuh"
#include "strict.cuh"

struct thmr_tok_encoder {
  thmr_tok_encoder_desc d;
};

namespace thmr {

constexpr int kEncPad = 3;      // zero rows either side of every sequence (max dilation of the release tokenizer)
constexpr int kEncCin0 = 64;    // the 6 input channels padded to one 64-wide k-block
constexpr int kEncChunk = 256;  // poses per pass

// pose6d fp32 [B, J, in_dim] -> fp32 [B, J + 2 pad, 64], channels >= in_dim and pad rows zero.
__global__ void enc_input_kernel(const float* __restrict__ pose, float* __restrict__ dst, int B, int J, int in_dim,
                                 int pad) {
  const long t = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  const long total = static_cast<long>(B) * (J + 2 * pad) * kEncCin0;
  if (t >= total) return;
  const int c = t % kEncCin0;
  const long row = t / kEncCin0;
  const int r = row % (J + 2 * pad);
  const int b = row / (J + 2 * pad);
  float v = 0.f;
  if (r >= pad && r < pad + J && c < in_dim) v = pose[(static_cast<long>(b) * J + (r - pad)) * in_dim + c];
  dst[t] = v;
}

// Operand of Conv1d(C, C, 4, stride 2, padding 1): dst[b, pad + j, tap*C + c] = src[b, pad + 2j - 1 + tap, c]
// (rows -1 and Lin are pad rows of src, i.e. zero).  Pad rows of dst are zeroed.  C4 = C / 4 (16-byte units of fp32).
__global__ void enc_gather_s2_kernel(const float* __restrict__ src, float* __restrict__ dst, int B, int Lin, int Lout,
                                     int pad, int C4) {
  const long total = static_cast<long>(B) * (Lout + 2 * pad) * 4 * C4;
  const long t = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x;
  if (t >= total) return;
  const int c4 = t % C4;
  const int tap = (t / C4) % 4;
  const long row = t / (4L * C4);
  const int r = row % (Lout + 2 * pad);
  const int b = row / (Lout + 2 * pad);
  uint4 v = make_uint4(0, 0, 0, 0);
  if (r >= pad && r < pad + Lout) {
    const int sr = pad + 2 * (r - pad) - 1 + tap;          // in [pad - 1, pad + Lin]: always inside the padded row range
    v = reinterpret_cast<const uint4*>(src)[(static_cast<long>(b) * (Lin + 2 * pad) + sr) * C4 + c4];
  }
  reinterpret_cast<uint4*>(dst)[t] = v;
}

struct EncWs {
  __half* sA;
  float *in0, *bufA, *bufB, *gat, *x32, *lat_pad, *lat;
  void* vq;
  size_t total;
};
inline int enc_seq_lens(const thmr_tok_encoder_desc& d, int* L_up_max, int* T) {
  int L = ((d.joints * 2) / 10) * 10;                       // vanilla_pose_vqvae.py:69
  for (int i = 1; i < d.size_mul; ++i) L *= 2;
  *L_up_max = L;
  *T = (L + 2 - 4) / 2 + 1;                                 // Conv1d(k=4, s=2, p=1)
  return THMR_OK;
}
inline void enc_carve(const thmr_tok_encoder_desc& d, void* base, int B, EncWs* ws) {
  Bump bp(base);
  int Lmax, T;
  enc_seq_lens(d, &Lmax, &T);
  const int Bc = B < kEncChunk ? B : kEncChunk;
  const size_t rows_max = static_cast<size_t>(Bc) * (Lmax + 2 * kEncPad);
  const size_t rows_T = static_cast<size_t>(Bc) * (T + 2 * kEncPad);
  size_t sa = rows_T * 3 * 4 * d.width;                     // the gathered down-sampling operand is the widest A'
  if (rows_max * 3 * d.width > sa) sa = rows_max * 3 * d.width;
  ws->sA = bp.take<__half>(sa);
  ws->in0 = bp.take<float>(static_cast<size_t>(Bc) * (d.joints + 2 * kEncPad) * kEncCin0);
  ws->bufA = bp.take<float>(rows_max * d.width);
  ws->bufB = bp.take<float>(rows_max * d.width);
  ws->gat = bp.take<float>(rows_T * 4 * d.width);
  ws->x32 = bp.take<float>(rows_T * d.width);
  ws->lat_pad = bp.take<float>(rows_T * d.code_dim);
  ws->lat = bp.take<float>(static_cast<size_t>(B) * T * d.code_dim);
  const size_t vq = thmr_vq_workspace_bytes(static_cast<int64_t>(B) * T, d.nb_code, d.code_dim);
  ws->vq = bp.take<uint8_t>(vq);
  ws->total = (bp.off + 1023) & ~size_t(1023);
}

// One convolution in split precision: split(act_in(in32)) into sA, then out32 = conv(., weight) + bias (+ resid) with
// the pad rows of the output zero (split_gemm_desc; the weights are packed by tokenizer.py).
inline int enc_conv(const float* in, int B, int Lcur, int cin, int taps, int dil, int act_in, const thmr_tok_conv& cw,
                    int cout, float* o32, const float* resid, __half* sA, cudaStream_t st) {
  const long rows = static_cast<long>(B) * (Lcur + 2 * kEncPad);
  THMR_TRY(split_rows_launch(in, cin, sA, rows, cin, act_in, 0, 0, 0, st));
  GemmPlan plan;
  THMR_TRY(gemm_make_plan(split_gemm_desc(sA, rows, cin, taps, dil, cw.w, cout, cw.b, resid, o32, cout, Lcur, kEncPad),
                          &plan));
  return gemm_launch(plan, st);
}

inline int enc_run(const thmr_tok_encoder* e, const float* pose6d, int B, int64_t* code_idx, float* latent, void* workspace,
                   cudaStream_t st) {
  const thmr_tok_encoder_desc& d = e->d;
  EncWs ws;
  enc_carve(d, workspace, B, &ws);
  const int W = d.width, PAD = kEncPad;
  auto blocks = [](long n) { return static_cast<unsigned>((n + 255) / 256); };
  int Lmax, T;
  enc_seq_lens(d, &Lmax, &T);
  float* lat = latent ? latent : ws.lat;
  for (int b0 = 0; b0 < B; b0 += kEncChunk) {
    const int Bc = (B - b0) < kEncChunk ? (B - b0) : kEncChunk;
    int L = d.joints;
    enc_input_kernel<<<blocks(static_cast<long>(Bc) * (L + 2 * PAD) * kEncCin0), 256, 0, st>>>(
        pose6d + static_cast<size_t>(b0) * d.joints * d.in_dim, ws.in0, Bc, L, d.in_dim, PAD);
    THMR_CUDA(cudaGetLastError());
    THMR_TRY(enc_conv(ws.in0, Bc, L, kEncCin0, 3, 1, kSplitActNone, d.conv_in, W, ws.bufA, nullptr, ws.sA, st));
    int Lout = ((d.joints * 2) / 10) * 10;
    for (int u = 0; u < d.size_mul; ++u) {                  // Upsample -> Conv1d(W,W,3) -> ReLU (ReLU of the previous
      upsample_rows_kernel<<<blocks(static_cast<long>(Bc) * (Lout + 2 * PAD) * (W / 4)), 256, 0, st>>>(   // conv: in the split)
          reinterpret_cast<const __half*>(ws.bufA), reinterpret_cast<__half*>(ws.bufB), Bc, L, Lout, PAD, W / 4);
      THMR_CUDA(cudaGetLastError());
      L = Lout;
      THMR_TRY(enc_conv(ws.bufB, Bc, L, W, 3, 1, kSplitActRelu, d.conv_up[u], W, ws.bufA, nullptr, ws.sA, st));
      Lout = 2 * L;
    }
    // down-sampling conv: gather the four taps (pre-ReLU values), then one GEMM over relu(.); its output is the residual
    // stream of the Resnet1D (ResConv1DBlock applies its activation first, resnet.py:51-60)
    enc_gather_s2_kernel<<<blocks(static_cast<long>(Bc) * (T + 2 * PAD) * 4 * (W / 4)), 256, 0, st>>>(ws.bufA, ws.gat, Bc, L,
                                                                                                     T, PAD, W / 4);
    THMR_CUDA(cudaGetLastError());
    THMR_TRY(enc_conv(ws.gat, Bc, T, 4 * W, 1, 1, kSplitActRelu, d.conv_down, W, ws.x32, nullptr, ws.sA, st));
    for (int dd = 0; dd < d.depth; ++dd) {                  // stored order = dilation descending (reverse_dilation)
      int dil = 1;
      for (int k = 0; k < d.depth - 1 - dd; ++k) dil *= d.dilation_rate;
      THMR_CHECK(dil <= PAD, "tok_encoder: dilation %d exceeds the sequence padding %d", dil, PAD);
      THMR_TRY(enc_conv(ws.x32, Bc, T, W, 3, dil, kSplitActRelu, d.res_conv1[dd], W, ws.bufB, nullptr, ws.sA, st));
      THMR_TRY(enc_conv(ws.bufB, Bc, T, W, 1, 1, kSplitActRelu, d.res_conv2[dd], W, ws.x32, ws.x32, ws.sA, st));
    }
    THMR_TRY(enc_conv(ws.x32, Bc, T, W, 3, 1, kSplitActNone, d.conv_out, d.code_dim, ws.lat_pad, nullptr, ws.sA, st));
    // QuantizeEMAReset.preprocess: (B, C, T) -> (B*T, C): drop the pad rows
    const size_t row_bytes = sizeof(float) * d.code_dim;
    THMR_CUDA(cudaMemcpy2DAsync(lat + static_cast<size_t>(b0) * T * d.code_dim, row_bytes * T,
                                ws.lat_pad + static_cast<size_t>(PAD) * d.code_dim, row_bytes * (T + 2 * PAD), row_bytes * T,
                                Bc, cudaMemcpyDeviceToDevice, st));
  }
  return thmr_vq_argmin(lat, static_cast<int64_t>(B) * T, d.codebook, d.nb_code, d.code_dim, code_idx, ws.vq, st);
}

}  // namespace thmr
