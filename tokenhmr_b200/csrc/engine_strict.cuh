// Strict-mode forward (thmr_config::strict = 1): the same launch list as engine_build() with every activation kept
// in fp32 and every contraction run as a split-fp16 GEMM (strict.cuh): fp32-grade results on the tensor cores.
// Weight pointers of thmr_weights then address split matrices  f16 [out, 3*in] = [hi | hi | lo] of w * 2^8
// (conv weights: per tap [hi | hi | lo]; packed by weights.py with strict=True).
//
// Every GEMM is preceded by split_rows (fp32 -> [hi | lo | hi] * 2^4, with the consumer-side activation fused: exact
// erf GELU / ReLU), so all epilogues are linear: alpha * acc + bias (+ residual), fp32 out.
#pragma once
#include "engine.cuh"
#include "strict.cuh"

namespace thmr {

inline size_t engine_build_strict(thmr_engine* e, void* workspace, int B, bool build, int* status, cudaStream_t stream) {
  const thmr_config& c = e->cfg;
  const thmr_weights& w = e->w;
  *status = THMR_OK;
  Bump bp(workspace);
  const int T = 192, D = c.vit_dim, M = B * T, H = c.vit_heads;
  const int E = c.dec_dim, inner = c.dec_heads * c.dec_dim_head, L = c.dec_depth;
  const int TN = c.token_num, CH = c.cls_hidden, NC = c.token_class_num, W = c.tok_width;
  const int gh = (c.image_size + 2 * c.patch_pad - c.patch) / c.patch + 1;
  const int gw = (c.crop_w + 2 * c.patch_pad - c.patch) / c.patch + 1;
  const int KP = 3 * c.patch * c.patch;
  const int PAD = kTokPad;
  const int HID = c.vit_mlp_ratio * D;
  const int Lp0 = TN + 2 * PAD;
  const int Lj = c.tok_joints, Lpj = Lj + 2 * PAD;

  // ---------------------------------------------------------------- workspace (all activations fp32)
  // split-operand scratch: the widest A' of the forward
  size_t sa_elems = static_cast<size_t>(M) * 3 * HID;
  {
    const size_t cand[] = {static_cast<size_t>(M) * 3 * KP, static_cast<size_t>(B) * Lp0 * 3 * NC,
                           static_cast<size_t>(B) * Lp0 * 3 * W, static_cast<size_t>(B) * 3 * E * 2,
                           static_cast<size_t>(B) * TN * 3 * c.cls_hidden_inter, static_cast<size_t>(B) * CH * 3 * TN};
    for (size_t v : cand) sa_elems = v > sa_elems ? v : sa_elems;
  }
  __half* sA = bp.take<__half>(sa_elems);
  const size_t n_skf = gemm_sk_flag_count(M, HID);
  unsigned* skf = bp.take<unsigned>(n_skf);        // stream-K ordering flags (zero between launches)
  float* a0 = bp.take<float>(static_cast<size_t>(M) * KP);
  float* x = bp.take<float>(static_cast<size_t>(M) * D);
  float* xn = bp.take<float>(static_cast<size_t>(M) * D);
  float* qkv = bp.take<float>(static_cast<size_t>(M) * 3 * D);
  float* ao = bp.take<float>(static_cast<size_t>(M) * D);
  float* hbuf = bp.take<float>(static_cast<size_t>(M) * HID);
  float* feat = bp.take<float>(static_cast<size_t>(M) * D);
  float* kv = bp.take<float>(static_cast<size_t>(M) * L * 2 * inner);
  float* tok = bp.take<float>(static_cast<size_t>(B) * E);
  float* y32 = bp.take<float>(static_cast<size_t>(B) * E);
  float* v32 = bp.take<float>(static_cast<size_t>(B) * inner);
  float* q32 = bp.take<float>(static_cast<size_t>(B) * inner);
  float* att32 = bp.take<float>(static_cast<size_t>(B) * inner);
  float* hid32 = bp.take<float>(static_cast<size_t>(B) * c.dec_mlp_dim);
  float* readout = bp.take<float>(static_cast<size_t>(B) * 32);
  float* mt32 = bp.take<float>(static_cast<size_t>(B) * TN * CH);
  float* cx = bp.take<float>(static_cast<size_t>(B) * TN * CH);
  float* yT = bp.take<float>(static_cast<size_t>(B) * CH * TN);
  float* t1 = bp.take<float>(static_cast<size_t>(B) * CH * c.cls_token_inter);
  float* yT2 = bp.take<float>(static_cast<size_t>(B) * CH * TN);
  float* xy = bp.take<float>(static_cast<size_t>(B) * TN * CH);
  float* z32 = bp.take<float>(static_cast<size_t>(B) * TN * CH);
  float* c1 = bp.take<float>(static_cast<size_t>(B) * TN * c.cls_hidden_inter);
  float* mn32 = bp.take<float>(static_cast<size_t>(B) * TN * CH);
  float* mnn = bp.take<float>(static_cast<size_t>(B) * TN * CH);
  float* logits = bp.take<float>(static_cast<size_t>(B) * TN * NC);
  float* probs_fallback = bp.take<float>(static_cast<size_t>(B) * TN * NC);
  float* d32 = bp.take<float>(static_cast<size_t>(B) * Lp0 * c.code_dim);
  float* bufA = bp.take<float>(static_cast<size_t>(B) * Lp0 * W);
  float* bufB = bp.take<float>(static_cast<size_t>(B) * Lp0 * W);
  float* out6 = bp.take<float>(static_cast<size_t>(B) * Lpj * 8);
  TailWs tail;
  tail_carve(bp, e->smpl->m, B, &tail);
  const size_t total = (bp.off + 1023) & ~size_t(1023);
  if (!build) return total;

  // ---------------------------------------------------------------- steps
  e->steps.clear();
  e->stamps = nullptr;       // (in-graph stamps are a default-mode instrument)
  StepList S{e->steps};
  int err = THMR_OK;

  // One step of two kernels: split_rows(act_in(A)) of `srows` rows of K channels into sA, then the GEMM d over sA
  // (split_gemm_desc).  (sT, spitch, slo): optional remap of the split rows into padded sequences (split_rows_kernel).
  auto slinear = [&](GemmDesc d, const float* A, long lda, long srows, int K, int act_in, int sT = 0, int spitch = 0,
                     int slo = 0) {
    if (!c.concurrent && gemm_sk_flag_count(d.M, d.N) <= n_skf) d.sk_flags = skf;
    GemmPlan plan;
    const int s = gemm_make_plan(d, &plan);
    if (s != THMR_OK) { err = s; return; }
    S.flops = 2.0 * d.M * d.N * d.taps * K;     // algorithmic (one product), the kernel does three
    S.bytes = 0;
    __half* dst = sA;
    S.push_back([=](const RunCtx&, cudaStream_t st) -> int {
      THMR_TRY(split_rows_launch(A, lda, dst, srows, K, act_in, sT, spitch, slo, st));
      return gemm_launch(plan, st);
    }, 2);
  };
  auto lin = [&](const float* A, int K, long rows, int act_in, const void* Wt, int N, const float* bias, float* o32,
                 const float* resid = nullptr) {
    slinear(split_gemm_desc(sA, rows, K, 1, 1, Wt, N, bias, resid, o32, N), A, K, rows, K, act_in);
  };
  auto ln = [&](const float* in, const float* g, const float* b, float* o32, int R, int C, float eps, int relu, int out_t) {
    S.flops = 0;
    S.bytes = static_cast<double>(R) * C * 8;
    S.push_back([=](const RunCtx&, cudaStream_t st) -> int {
      return layernorm_launch(in, g, b, nullptr, 0, o32, R, C, eps, relu, out_t, st);
    });
  };

  // ---- ViT backbone (vit.py:320-343)
  {
    const int S_ = c.image_size, x0 = (c.image_size - c.crop_w) / 2, Wc = c.crop_w, P = c.patch, pad = c.patch_pad;
    S.tag("vit.patch_im2col", 0, static_cast<double>(B) * 3 * c.image_size * c.crop_w * 4 + static_cast<double>(M) * KP * 4);
    S.push_back([=](const RunCtx& r, cudaStream_t st) -> int {
      const long total_t = static_cast<long>(B) * gh * gw * 3 * P;
      im2col_patch_f32_kernel<<<static_cast<unsigned>((total_t + 255) / 256), 256, 0, st>>>(r.img, a0, B, S_, x0, Wc, P,
                                                                                           pad, gh, gw);
      THMR_CUDA(cudaGetLastError());
      return THMR_OK;
    });
    S.tag("vit.patch_embed_gemm");
    GemmDesc d = split_gemm_desc(sA, M, KP, 1, 1, w.patch_w, D, w.patch_b, w.pos, x, D);
    d.resid_mod = T;
    slinear(d, a0, KP, M, KP, kSplitActNone);
  }
  const float att_scale = 1.0f / sqrtf(static_cast<float>(D / H));
  for (int i = 0; i < c.vit_depth; ++i) {
    const thmr_vit_block& bw = e->blocks[i];
    S.tag("vit.layernorm");
    ln(x, bw.ln1_g, bw.ln1_b, xn, M, D, c.vit_ln_eps, 0, 0);
    S.tag("vit.qkv_gemm");
    lin(xn, D, M, kSplitActNone, bw.qkv_w, 3 * D, bw.qkv_b, qkv);
    S.tag("vit.attention", 4.0 * B * H * 192.0 * 192.0 * 80.0, 4.0 * M * D * 4);
    S.push_back([=](const RunCtx&, cudaStream_t st) -> int {
      return attention_f32_launch(qkv, 3 * D, B, H, ao, D, att_scale, st);
    });
    S.tag("vit.proj_gemm");
    lin(ao, D, M, kSplitActNone, bw.proj_w, D, bw.proj_b, x, x);
    S.tag("vit.layernorm");
    ln(x, bw.ln2_g, bw.ln2_b, xn, M, D, c.vit_ln_eps, 0, 0);
    S.tag("vit.fc1_gelu_gemm");
    lin(xn, D, M, kSplitActNone, bw.fc1_w, HID, bw.fc1_b, hbuf);             // pre-GELU; GELU is applied by fc2's split
    S.tag("vit.fc2_gemm");
    lin(hbuf, HID, M, kSplitActGelu, bw.fc2_w, D, bw.fc2_b, x, x);
  }
  {
    S.tag("vit.layernorm", 0, static_cast<double>(M) * D * 8);
    const float* g = w.last_g; const float* b = w.last_b;
    const float eps = c.vit_ln_eps;
    S.push_back([=](const RunCtx& r, cudaStream_t st) -> int {
      THMR_TRY(layernorm_launch(x, g, b, nullptr, 0, feat, M, D, eps, 0, 0, st));
      float* t32 = r.vit_tokens_only ? r.vit_tokens_only : r.out.vit_tokens;
      if (t32) THMR_CUDA(cudaMemcpyAsync(t32, feat, sizeof(float) * M * D, cudaMemcpyDeviceToDevice, st));
      return THMR_OK;
    });
  }
  e->vit_steps = S.size();

  // ---- decoder (pose_transformer.py:191-201,349-357)
  S.tag("dec.to_kv_gemm");
  lin(feat, D, M, kSplitActNone, w.kv_w, L * 2 * inner, nullptr, kv);
  S.tag("dec.token_ops");
  {
    const float* t0 = w.token0;
    S.push_back([=](const RunCtx&, cudaStream_t st) -> int {
      broadcast_row_kernel<<<(B * E + 255) / 256, 256, 0, st>>>(t0, tok, B, E);
      THMR_CUDA(cudaGetLastError());
      return THMR_OK;
    });
  }
  for (int l = 0; l < L; ++l) {
    const thmr_dec_layer& dw = e->dec[l];
    ln(tok, dw.ln0_g, dw.ln0_b, y32, B, E, c.ln_eps, 0, 0);
    lin(y32, E, B, kSplitActNone, dw.sa_v_w, inner, nullptr, v32);
    lin(v32, inner, B, kSplitActNone, dw.sa_out_w, E, dw.sa_out_b, tok, tok);
    ln(tok, dw.ln1_g, dw.ln1_b, y32, B, E, c.ln_eps, 0, 0);
    lin(y32, E, B, kSplitActNone, dw.ca_q_w, inner, nullptr, q32);
    {
      const int ld = L * 2 * inner, koff = l * 2 * inner, voff = koff + inner, heads = c.dec_heads;
      const float scale = 1.0f / sqrtf(static_cast<float>(c.dec_dim_head));
      S.push_back([=](const RunCtx&, cudaStream_t st) -> int {
        dec_cross_attn_f32_kernel<192><<<B * heads, 192, 0, st>>>(q32, kv, ld, koff, voff, scale, att32, heads);
        THMR_CUDA(cudaGetLastError());
        return THMR_OK;
      });
    }
    lin(att32, inner, B, kSplitActNone, dw.ca_out_w, E, dw.ca_out_b, tok, tok);
    ln(tok, dw.ln2_g, dw.ln2_b, y32, B, E, c.ln_eps, 0, 0);
    lin(y32, E, B, kSplitActNone, dw.ff1_w, c.dec_mlp_dim, dw.ff1_b, hid32);
    lin(hid32, c.dec_mlp_dim, B, kSplitActGelu, dw.ff2_w, E, dw.ff2_b, tok, tok);
  }
  S.push_back([=](const RunCtx& r, cudaStream_t st) -> int {
    if (r.out.token_out)
      THMR_CUDA(cudaMemcpyAsync(r.out.token_out, tok, sizeof(float) * B * E, cudaMemcpyDeviceToDevice, st));
    return THMR_OK;
  }, 0);
  lin(tok, E, B, kSplitActNone, w.readout_w, 32, w.readout_b, readout);

  // ---- token classifier (token_classifier.py:89-104)
  S.tag("cls.mixer_ops");
  lin(tok, E, B, kSplitActNone, w.mt_w, TN * CH, w.mt_b, mt32);
  ln(mt32, w.mt_ln_g, w.mt_ln_b, cx, B, TN * CH, c.ln_eps, 1, 0);
  for (int i = 0; i < c.cls_blocks; ++i) {
    const thmr_mixer_block& mw = e->mixer[i];
    ln(cx, mw.ln1_g, mw.ln1_b, yT, B * TN, CH, c.ln_eps, 0, TN);                      // transposed: (B*H, T)
    lin(yT, TN, static_cast<long>(B) * CH, kSplitActNone, mw.tok1_w, c.cls_token_inter, mw.tok1_b, t1);
    lin(t1, c.cls_token_inter, static_cast<long>(B) * CH, kSplitActGelu, mw.tok2_w, TN, mw.tok2_b, yT2);
    S.push_back([=](const RunCtx&, cudaStream_t st) -> int {
      const long n = static_cast<long>(B) * TN * CH;
      mixer_add_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(cx, yT2, nullptr, xy, B, TN, CH);
      THMR_CUDA(cudaGetLastError());
      return THMR_OK;
    });
    ln(xy, mw.ln2_g, mw.ln2_b, z32, B * TN, CH, c.ln_eps, 0, 0);
    lin(z32, CH, static_cast<long>(B) * TN, kSplitActNone, mw.ch1_w, c.cls_hidden_inter, mw.ch1_b, c1);
    lin(c1, c.cls_hidden_inter, static_cast<long>(B) * TN, kSplitActGelu, mw.ch2_w, CH, mw.ch2_b, cx, xy);
  }
  lin(cx, CH, static_cast<long>(B) * TN, kSplitActNone, w.mn_w, CH, w.mn_b, mn32);
  ln(mn32, w.mn_ln_g, w.mn_ln_b, mnn, B * TN, CH, c.ln_eps, 1, 0);
  lin(mnn, CH, static_cast<long>(B) * TN, kSplitActNone, w.cls_w, NC, w.cls_b, logits);
  // the softmax output p32 is held in a member of the step closure below: the dequant GEMM reads it through the split
  S.push_back([=](const RunCtx& r, cudaStream_t st) -> int {
    float* p32 = r.out.cls_logits_softmax ? r.out.cls_logits_softmax : probs_fallback;
    THMR_TRY(softmax_rows_launch(logits, p32, nullptr, B * TN, NC, TN, Lp0, PAD, st));
    // probabilities must sit in probs_fallback for the (pre-planned) split below
    if (p32 != probs_fallback)
      THMR_CUDA(cudaMemcpyAsync(probs_fallback, p32, sizeof(float) * B * TN * NC, cudaMemcpyDeviceToDevice, st));
    return THMR_OK;
  });

  S.tag("tok.decoder_ops");
  // ---- tokenizer: soft codebook lookup + Conv1d decoder (vanilla_pose_vqvae.py:294-297, 135-154)
  // dequantize_logits on the padded layout: the split scatters the B*TN rows into [B, Lp0] sequences; the pad rows of
  // the scratch hold stale data, so the output rows are masked to zero (real zeros for the conv)
  slinear(split_gemm_desc(sA, static_cast<long>(B) * Lp0, NC, 1, 1, w.codebook_t, c.code_dim, nullptr, nullptr, d32,
                          c.code_dim, TN, PAD),
          probs_fallback, NC, static_cast<long>(B) * TN, NC, kSplitActNone, TN, Lp0, PAD);
  auto conv = [&](const float* in, int Lcur, int cin, int act_in, const thmr_conv& cw, int cout, int dil, int taps,
                  float* o32, int ld32, const float* resid) {
    const long rows = static_cast<long>(B) * (Lcur + 2 * PAD);
    slinear(split_gemm_desc(sA, rows, cin, taps, dil, cw.w, cout, cw.b, resid, o32, ld32, Lcur, PAD), in, cin, rows, cin,
            act_in);
  };
  int Lcur = TN;
  // activations are applied by the consumer's split: bufA holds the PRE-ReLU conv output from here on
  conv(d32, Lcur, c.code_dim, kSplitActNone, w.conv_in, W, 1, 3, bufA, W, nullptr);
  for (int u = 0; u < c.n_upsample; ++u) {
    const int Lout = c.upsample_sizes[u], Lin = Lcur;
    S.push_back([=](const RunCtx&, cudaStream_t st) -> int {   // nearest gather commutes with ReLU: copy the pre-ReLU rows
      const long n = static_cast<long>(B) * (Lout + 2 * PAD) * (W / 4);
      upsample_rows_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(
          reinterpret_cast<const __half*>(bufA), reinterpret_cast<__half*>(bufB), B, Lin, Lout, PAD, W / 4);
      THMR_CUDA(cudaGetLastError());
      return THMR_OK;
    });
    Lcur = Lout;
    conv(bufB, Lcur, W, kSplitActRelu, w.conv_up[u], W, 1, 3, bufA, W, nullptr);
  }
  // Resnet1D (resnet.py:51-82): x = x + conv1x1(relu(conv3_dil(relu(x)))).  The residual stream x is relu(bufA) after
  // the last upsample conv (its ReLU belongs to the Sequential, vanilla_pose_vqvae.py:141): materialise it once.
  float* xres = bufA;
  {
    const long n4 = static_cast<long>(B) * (Lcur + 2 * PAD) * W / 4;
    S.push_back([=](const RunCtx&, cudaStream_t st) -> int {
      relu_inplace_kernel<<<static_cast<unsigned>((n4 + 255) / 256), 256, 0, st>>>(xres, n4);
      THMR_CUDA(cudaGetLastError());
      return THMR_OK;
    });
  }
  for (int dd = 0; dd < c.tok_depth; ++dd) {
    int dil = 1;
    for (int k = 0; k < c.tok_depth - 1 - dd; ++k) dil *= c.tok_dilation_rate;
    conv(xres, Lcur, W, kSplitActRelu, w.res_conv1[dd], W, dil, 3, bufB, W, nullptr);       // relu(x) -> conv3
    conv(bufB, Lcur, W, kSplitActRelu, w.res_conv2[dd], W, 1, 1, xres, W, xres);            // x += conv1(relu(.))
  }
  conv(xres, Lcur, W, kSplitActNone, w.conv_post, W, 1, 3, bufB, W, nullptr);
  conv(bufB, Lcur, W, kSplitActNone, w.conv_out, 6, 1, 3, out6, 8, nullptr);

  const int s = add_tail_step(S, e, B, tail, readout, out6);
  if (s != THMR_OK) err = s;
  *status = err;
  if (err == THMR_OK && cudaMemsetAsync(skf, 0, n_skf * sizeof(unsigned), stream) != cudaSuccess)
    *status = fail(THMR_ERR_CUDA, "cudaMemsetAsync(stream-K flags) failed");
  return total;
}

}  // namespace thmr
