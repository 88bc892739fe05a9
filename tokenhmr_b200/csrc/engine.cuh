// Engine: orchestrates TokenHMR.forward (tokenhmr.py:135-188) as a fixed list of stream-ordered launches
// over a caller-provided workspace.  Plans (TMA descriptors, tile shapes) are built once per
// (workspace, batch) and replayed; nothing here synchronises the host, so the whole forward can be
// captured in a CUDA graph by the caller.
#pragma once
#include <functional>
#include <vector>

#include "attention3_tcgen05.cuh"
#include "common.cuh"
#include "elementwise.cuh"
#include "gemm_host.cuh"
#include "head_kernels.cuh"
#include "smpl_lbs.cuh"
#include "vq.cuh"

struct thmr_smpl {
  thmr::SmplModel m;
  int* parents_dev = nullptr;
};

namespace thmr {

struct RunCtx {
  const float* img;
  thmr_outputs out;
  float* vit_tokens_only;  // thmr_engine_vit_forward target
};

using StepFn = std::function<int(const RunCtx&, cudaStream_t)>;

// One launch group of the forward: a label (kernel family + role) and its algorithmic work, so that a timed
// replay (thmr_engine_profile) can attribute device time and compute roofline fractions live.
struct Step {
  StepFn fn;
  const char* name;
  double flops;   // algorithmic FLOPs (2*MAC) of tensor-core work, 0 for bandwidth-bound kernels
  double bytes;   // algorithmic HBM bytes for bandwidth-bound kernels, 0 otherwise
  int kernels;    // kernels fn launches (copies and memsets not counted): thmr_engine_num_launches
};

// Appends the steps of one build; tag() sets the label and work recorded with the steps pushed after it.
struct StepList {
  std::vector<Step>& v;
  const char* name = "";
  double flops = 0, bytes = 0;
  void tag(const char* n, double f = 0, double b = 0) { name = n; flops = f; bytes = b; }
  void push_back(StepFn fn, int kernels = 1) { v.push_back(Step{std::move(fn), name, flops, bytes, kernels}); }
  size_t size() const { return v.size(); }
};

// ---- SMPL stage (shared by thmr_lbs / thmr_smpl_forward / the engine) -----------------------------------
// The blended vertices v_posed (fp32, 82.7 KB per pose) are produced by a GEMM and consumed by the skinning kernel.
// Poses are processed in chunks of kSmplChunk so that the offsets of a chunk (42 MB) stay L2-resident between the
// two kernels instead of making a round trip through HBM.
constexpr int kSmplChunk = 512;
struct SmplWs {
  float* A;        // [B,24,12]
  float* Jposed;   // [B,24,3]
  __half* pf16;    // [B,624]
  float* offsets;  // [min(B,kSmplChunk), off_pitch]
  long off_pitch;  // 3V rounded up to 4 floats (TMA store needs 16-byte row pitch)
};
inline void smpl_carve(Bump& bp, const SmplModel& m, int B, SmplWs* ws) {
  ws->A = bp.take<float>(static_cast<size_t>(B) * kSmplJ * 12);
  ws->Jposed = bp.take<float>(static_cast<size_t>(B) * kSmplJ * 3);
  ws->pf16 = bp.take<__half>(static_cast<size_t>(B) * 3 * kSmplPFPad);
  ws->off_pitch = (3L * m.V + 3) / 4 * 4;
  ws->offsets = bp.take<float>(static_cast<size_t>(B < kSmplChunk ? B : kSmplChunk) * ws->off_pitch);
}

inline int smpl_blend_plan(const SmplModel& m, const SmplWs& ws, int p0, int n, GemmPlan* plan) {
  GemmDesc d;
  d.A = ws.pf16 + static_cast<size_t>(p0) * 3 * kSmplPFPad; d.lda = 3 * kSmplPFPad; d.a_rows = n;
  d.B = m.posedirsT; d.ldb = 3 * kSmplPFPad;
  d.M = n; d.N = static_cast<int>(ws.off_pitch); d.K = 3 * kSmplPFPad;
  d.out32 = ws.offsets; d.ld32 = static_cast<int>(ws.off_pitch);
  d.alpha = 1.0f / (kSplitScale * kSplitScale);
  d.no_2cta = true;
  return gemm_make_plan(d, plan);
}

// verts: fp32 [B,V,3];  lbs_joints (nullable): [B,24,3];  joints44 (nullable): [B,25+n_extra,3]
// blend_plans (nullable): pre-built plans, one per chunk (engine); otherwise built on the fly.
inline int smpl_run(const thmr_smpl* sm, const float* pose, int pose2rot, const float* betas, int B, float* verts,
                    float* lbs_joints, float* joints44, const float* pred_cam, float focal, float image_size,
                    float* cam_t, float* focal_out, float* kp2d, const SmplWs& ws, const GemmPlan* blend_plans,
                    cudaStream_t st) {
  const SmplModel& m = sm->m;
  // vertices per skinning block (smpl_lbs.cuh); read per call so that a benchmark can compare the shapes in one process
  int skin_threads = kSkinThreadsDefault;
  { const char* e = getenv("THMR_SKIN_THREADS"); if (e && (atoi(e) == 128 || atoi(e) == 256)) skin_threads = atoi(e); }
  smpl_pose_kernel<<<B, 32, 0, st>>>(pose, pose2rot, betas, m.J_template, m.J_shapedirs, m.nb, sm->parents_dev, ws.A,
                                     lbs_joints ? lbs_joints : ws.Jposed, ws.pf16, B);
  THMR_CUDA(cudaGetLastError());
  int ci = 0;
  for (int p0 = 0; p0 < B; p0 += kSmplChunk, ++ci) {
    const int n = (B - p0) < kSmplChunk ? (B - p0) : kSmplChunk;
    GemmPlan local;
    const GemmPlan* plan = blend_plans ? &blend_plans[ci] : &local;
    if (!blend_plans) THMR_TRY(smpl_blend_plan(m, ws, p0, n, &local));
    THMR_TRY(gemm_launch(*plan, st));
    const float* Ac = ws.A + static_cast<size_t>(p0) * kSmplJ * 12;
    float* vc = verts + static_cast<size_t>(p0) * m.V * 3;
    const dim3 grid((m.V + skin_threads - 1) / skin_threads, (n + kSkinPoses - 1) / kSkinPoses);
    const long vp = static_cast<long>(m.V) * 3;
    if (skin_threads == 256 && m.ell <= 4)
      smpl_skin_kernel<256, 4><<<grid, 256, 0, st>>>(m.w_idx, m.w_val, m.ell, Ac, ws.offsets, ws.off_pitch, vc, vp, m.V, n);
    else if (skin_threads == 256)
      smpl_skin_kernel<256, 8><<<grid, 256, 0, st>>>(m.w_idx, m.w_val, m.ell, Ac, ws.offsets, ws.off_pitch, vc, vp, m.V, n);
    else if (m.ell <= 4)
      smpl_skin_kernel<128, 4><<<grid, 128, 0, st>>>(m.w_idx, m.w_val, m.ell, Ac, ws.offsets, ws.off_pitch, vc, vp, m.V, n);
    else
      smpl_skin_kernel<128, 8><<<grid, 128, 0, st>>>(m.w_idx, m.w_val, m.ell, Ac, ws.offsets, ws.off_pitch, vc, vp, m.V, n);
    THMR_CUDA(cudaGetLastError());
  }
  if (joints44) {
    smpl_joints_kernel<<<B, 64, 0, st>>>(lbs_joints ? lbs_joints : ws.Jposed, verts, static_cast<long>(m.V) * 3,
                                         m.joint_map, m.extra_vid, m.jx_ptr, m.jx_idx, m.jx_val, m.n_extra, joints44,
                                         pred_cam, focal, image_size, cam_t, focal_out, kp2d);
    THMR_CUDA(cudaGetLastError());
  }
  return THMR_OK;
}

}  // namespace thmr

struct thmr_engine {
  thmr_config cfg;
  thmr_weights w;
  std::vector<thmr_vit_block> blocks;
  std::vector<thmr_dec_layer> dec;
  std::vector<thmr_mixer_block> mixer;
  const thmr_smpl* smpl = nullptr;
  // plan cache
  void* ws = nullptr;
  int B = 0;
  std::vector<thmr::Step> steps;
  size_t vit_steps = 0;  // steps [0, vit_steps) = backbone
  unsigned long long* stamps = nullptr;   // [kMaxStamps] in the workspace: start stamp of step i, end stamp at [n_steps]
};

constexpr int kMaxStamps = 2048;

namespace thmr {

constexpr int kTokPad = 3;  // zero rows on both ends of every tokenizer-decoder sequence (max dilation)

// Workspace of the forward's tail: where the outputs a caller leaves null (thmr_outputs) are written, and SMPL's.
struct TailWs {
  float *rot, *betas, *cam, *camt, *focal, *kp3, *kp2, *verts;
  SmplWs smpl;
};
inline void tail_carve(Bump& bp, const SmplModel& m, int B, TailWs* t) {
  const int NJ = 25 + m.n_extra;
  t->rot = bp.take<float>(static_cast<size_t>(B) * 24 * 9);
  t->betas = bp.take<float>(static_cast<size_t>(B) * 16);
  t->cam = bp.take<float>(static_cast<size_t>(B) * 4);
  t->camt = bp.take<float>(static_cast<size_t>(B) * 4);
  t->focal = bp.take<float>(static_cast<size_t>(B) * 2);
  t->kp3 = bp.take<float>(static_cast<size_t>(B) * NJ * 3);
  t->kp2 = bp.take<float>(static_cast<size_t>(B) * NJ * 2);
  t->verts = bp.take<float>(static_cast<size_t>(B) * m.V * 3);
  smpl_carve(bp, m, B, &t->smpl);
}

// Read-out assembly, 6D -> rotation (token_head.py:103-128), SMPL + projection (tokenhmr.py:162-187) as one step:
// readout fp32 [B, 32], out6 fp32 [B, tok_joints + 2 * kTokPad, 8].  The blend GEMM plans are built here.
inline int add_tail_step(StepList& S, const thmr_engine* e, int B, const TailWs& t, const float* readout,
                         const float* out6) {
  const thmr_smpl* sm = e->smpl;
  const int chunks = (B + kSmplChunk - 1) / kSmplChunk;
  std::vector<GemmPlan> blend(chunks);
  for (int ci = 0; ci < chunks; ++ci) {
    const int p0 = ci * kSmplChunk;
    THMR_TRY(smpl_blend_plan(sm->m, t.smpl, p0, (B - p0) < kSmplChunk ? (B - p0) : kSmplChunk, &blend[ci]));
  }
  const float* ip = e->w.init_pose; const float* ib = e->w.init_betas; const float* ic = e->w.init_cam;
  const int nb = sm->m.nb, Lpj = e->cfg.tok_joints + 2 * kTokPad, PAD = kTokPad;
  const float focal = e->cfg.focal_length, isz = static_cast<float>(e->cfg.image_size);
  S.tag("smpl.lbs");
  S.push_back([=](const RunCtx& r, cudaStream_t st) -> int {
    float* rot = r.out.rotmats ? r.out.rotmats : t.rot;
    float* bet = r.out.betas ? r.out.betas : t.betas;
    float* cam = r.out.pred_cam ? r.out.pred_cam : t.cam;
    head_assemble_kernel<<<(B * 24 + 127) / 128, 128, 0, st>>>(readout, 32, out6, 8, Lpj, PAD, ip, ib, ic, rot, bet, cam,
                                                              r.out.pose6d, B, nb);
    THMR_CUDA(cudaGetLastError());
    float* verts = r.out.pred_vertices ? r.out.pred_vertices : t.verts;
    float* kp3 = r.out.pred_keypoints_3d ? r.out.pred_keypoints_3d : t.kp3;
    float* kp2 = r.out.pred_keypoints_2d ? r.out.pred_keypoints_2d : t.kp2;
    float* camt = r.out.pred_cam_t ? r.out.pred_cam_t : t.camt;
    float* foc = r.out.focal_length ? r.out.focal_length : t.focal;
    return smpl_run(sm, rot, 0, bet, B, verts, nullptr, kp3, cam, focal, isz, camt, foc, kp2, t.smpl, blend.data(), st);
  }, 3 + 2 * chunks);   // head assemble, pose, per chunk blend GEMM + skin, joints
  return THMR_OK;
}

inline size_t engine_build(thmr_engine* e, void* workspace, int B, bool build, int* status, cudaStream_t stream) {
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

  // ---------------------------------------------------------------- workspace
  __half* a0 = bp.take<__half>(static_cast<size_t>(M) * KP);
  float* x = bp.take<float>(static_cast<size_t>(M) * D);
  __half* xn = bp.take<__half>(static_cast<size_t>(M) * D);
  __half* qkv = bp.take<__half>(static_cast<size_t>(M) * 3 * D);
  __half* ao = bp.take<__half>(static_cast<size_t>(M) * D);
  __half* hbuf = bp.take<__half>(static_cast<size_t>(M) * c.vit_mlp_ratio * D);
  __half* feat = bp.take<__half>(static_cast<size_t>(M) * D);
  __half* kv = bp.take<__half>(static_cast<size_t>(M) * L * 2 * inner);
  float* tok = bp.take<float>(static_cast<size_t>(B) * E);
  __half* y16 = bp.take<__half>(static_cast<size_t>(B) * E);
  __half* v16 = bp.take<__half>(static_cast<size_t>(B) * inner);
  float* q32 = bp.take<float>(static_cast<size_t>(B) * inner);
  __half* att16 = bp.take<__half>(static_cast<size_t>(B) * inner);
  __half* hid16 = bp.take<__half>(static_cast<size_t>(B) * c.dec_mlp_dim);
  const size_t n_skf = gemm_sk_flag_count(M, static_cast<long long>(c.vit_mlp_ratio) * D);
  unsigned* skf = bp.take<unsigned>(n_skf);        // stream-K ordering flags (zero between launches)
  unsigned long long* stamps = bp.take<unsigned long long>(kMaxStamps);   // in-graph start stamps, one slot per step
  float* readout = bp.take<float>(static_cast<size_t>(B) * 32);
  float* mt32 = bp.take<float>(static_cast<size_t>(B) * TN * CH);
  float* cx = bp.take<float>(static_cast<size_t>(B) * TN * CH);
  __half* cx16 = bp.take<__half>(static_cast<size_t>(B) * TN * CH);
  __half* yT16 = bp.take<__half>(static_cast<size_t>(B) * CH * TN);
  __half* t1 = bp.take<__half>(static_cast<size_t>(B) * CH * c.cls_token_inter);
  float* yT32 = bp.take<float>(static_cast<size_t>(B) * CH * TN);
  float* xy = bp.take<float>(static_cast<size_t>(B) * TN * CH);
  __half* z16 = bp.take<__half>(static_cast<size_t>(B) * TN * CH);
  __half* c1 = bp.take<__half>(static_cast<size_t>(B) * TN * c.cls_hidden_inter);
  float* mn32 = bp.take<float>(static_cast<size_t>(B) * TN * CH);
  __half* mn16 = bp.take<__half>(static_cast<size_t>(B) * TN * CH);
  float* logits = bp.take<float>(static_cast<size_t>(B) * TN * NC);
  float* probs_fallback = bp.take<float>(static_cast<size_t>(B) * TN * NC);
  const int Lp0 = TN + 2 * PAD;
  __half* p16 = bp.take<__half>(static_cast<size_t>(B) * Lp0 * NC);
  __half* d16 = bp.take<__half>(static_cast<size_t>(B) * Lp0 * c.code_dim);
  __half* bufA = bp.take<__half>(static_cast<size_t>(B) * Lp0 * W);
  __half* bufB = bp.take<__half>(static_cast<size_t>(B) * Lp0 * W);
  const int Lj = c.tok_joints, Lpj = Lj + 2 * PAD;
  float* x32 = bp.take<float>(static_cast<size_t>(B) * Lpj * W);
  float* out6 = bp.take<float>(static_cast<size_t>(B) * Lpj * 8);
  TailWs tail;
  tail_carve(bp, e->smpl->m, B, &tail);
  const size_t total = (bp.off + 1023) & ~size_t(1023);
  if (!build) return total;

  // ---------------------------------------------------------------- steps
  e->steps.clear();
  StepList S{e->steps};
  int err = THMR_OK;
  e->stamps = stamps;
  auto slot = [&]() -> unsigned long long* { return S.size() < static_cast<size_t>(kMaxStamps - 1) ? stamps + S.size() : nullptr; };
  auto add_gemm = [&](GemmDesc d) {
    d.stamp = slot();
    GemmPlan plan;
    const int s = gemm_make_plan(d, &plan);
    if (s != THMR_OK) { err = s; return; }
    S.flops = 2.0 * d.M * d.N * d.K;
    S.bytes = 0;
    S.push_back([plan](const RunCtx&, cudaStream_t st) -> int { return gemm_launch(plan, st); });
  };
  auto linear = [&](const __half* A, int lda, int rows, const void* Wt, int N, int K, const float* bias, int act,
                    float* o32, __half* o16, const float* resid = nullptr) {
    GemmDesc d;
    d.A = A; d.lda = lda; d.a_rows = rows;
    d.B = static_cast<const __half*>(Wt); d.ldb = K;
    d.M = rows; d.N = N; d.K = K;
    d.bias = bias; d.act = act; d.resid = resid; d.ldr = N;
    d.out32 = o32; d.ld32 = N; d.out16 = o16; d.ld16 = N;
    if (!c.concurrent && gemm_sk_flag_count(rows, N) <= n_skf) d.sk_flags = skf;   // (stream-K spins across CTA pairs)
    add_gemm(d);
  };
  auto ln = [&](const float* in, const float* g, const float* b, __half* o16, float* o32, int R, int C, float eps,
                int relu, int out_t) {
    S.flops = 0;
    S.bytes = static_cast<double>(R) * C * (4 + (o16 ? 2 : 0) + (o32 ? 4 : 0));
    unsigned long long* sp = slot();
    S.push_back([=](const RunCtx&, cudaStream_t st) -> int {
      return layernorm_launch(in, g, b, o16, 0, o32, R, C, eps, relu, out_t, st, sp);
    });
  };

  // ---- ViT backbone (vit.py:320-343)
  {
    const int S_ = c.image_size, x0 = (c.image_size - c.crop_w) / 2, Wc = c.crop_w, P = c.patch, pad = c.patch_pad;
    S.tag("vit.patch_im2col", 0, static_cast<double>(B) * 3 * c.image_size * c.crop_w * 4 + static_cast<double>(M) * KP * 2);
    unsigned long long* sp = slot();
    S.push_back([=](const RunCtx& r, cudaStream_t st) -> int {
      const long total_t = static_cast<long>(B) * gh * gw * 3 * P;
      im2col_patch_kernel<<<static_cast<unsigned>((total_t + 255) / 256), 256, 0, st>>>(r.img, a0, B, S_, x0, Wc, P, pad,
                                                                                       gh, gw, sp);
      THMR_CUDA(cudaGetLastError());
      return THMR_OK;
    });
    S.tag("vit.patch_embed_gemm");
    GemmDesc d;
    d.A = a0; d.lda = KP; d.a_rows = M;
    d.B = static_cast<const __half*>(w.patch_w); d.ldb = KP;
    d.M = M; d.N = D; d.K = KP;
    d.bias = w.patch_b; d.resid = w.pos; d.ldr = D; d.resid_mod = T;
    d.out32 = x; d.ld32 = D;
    add_gemm(d);
  }
  for (int i = 0; i < c.vit_depth; ++i) {
    const thmr_vit_block& bw = e->blocks[i];
    S.tag("vit.layernorm");
    ln(x, bw.ln1_g, bw.ln1_b, xn, nullptr, M, D, c.vit_ln_eps, 0, 0);
    S.tag("vit.qkv_gemm");
    linear(xn, D, M, bw.qkv_w, 3 * D, D, bw.qkv_b, kActNone, nullptr, qkv);
    {
      // 4*N*N*d FLOPs per head (QK^T + PV); Q,K,V read + O written once in fp16
      S.tag("vit.attention", 4.0 * B * H * 192.0 * 192.0 * 80.0, 4.0 * M * D * 2);
      AttnPlan ap;
      const int s = attention_make_plan(qkv, 3 * D, B, H, ao, D, nullptr, &ap);
      if (s != THMR_OK) err = s;
      ap.p.stamp = slot();
      S.push_back([ap](const RunCtx&, cudaStream_t st) -> int { return attention_dispatch(ap, st); });
    }
    S.tag("vit.proj_gemm");
    linear(ao, D, M, bw.proj_w, D, D, bw.proj_b, kActNone, x, nullptr, x);
    S.tag("vit.layernorm");
    ln(x, bw.ln2_g, bw.ln2_b, xn, nullptr, M, D, c.vit_ln_eps, 0, 0);
    S.tag("vit.fc1_gelu_gemm");
    linear(xn, D, M, bw.fc1_w, c.vit_mlp_ratio * D, D, bw.fc1_b, kActGelu, nullptr, hbuf);
    S.tag("vit.fc2_gemm");
    linear(hbuf, c.vit_mlp_ratio * D, M, bw.fc2_w, D, c.vit_mlp_ratio * D, bw.fc2_b, kActNone, x, nullptr, x);
  }
  {
    S.tag("vit.layernorm", 0, static_cast<double>(M) * D * 6);
    const float* g = w.last_g; const float* b = w.last_b;
    const float eps = c.vit_ln_eps;
    unsigned long long* sp = slot();
    S.push_back([=](const RunCtx& r, cudaStream_t st) -> int {
      float* t32 = r.vit_tokens_only ? r.vit_tokens_only : r.out.vit_tokens;
      return layernorm_launch(x, g, b, feat, 0, t32, M, D, eps, 0, 0, st, sp);
    });
  }
  e->vit_steps = S.size();

  // ---- decoder (pose_transformer.py:191-201,349-357): K/V of all layers in one GEMM
  S.tag("dec.to_kv_gemm");
  linear(feat, D, M, w.kv_w, L * 2 * inner, D, nullptr, kActNone, nullptr, kv);
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
    ln(tok, dw.ln0_g, dw.ln0_b, y16, nullptr, B, E, c.ln_eps, 0, 0);
    linear(y16, E, B, dw.sa_v_w, inner, E, nullptr, kActNone, nullptr, v16);
    linear(v16, inner, B, dw.sa_out_w, E, inner, dw.sa_out_b, kActNone, tok, nullptr, tok);
    ln(tok, dw.ln1_g, dw.ln1_b, y16, nullptr, B, E, c.ln_eps, 0, 0);
    linear(y16, E, B, dw.ca_q_w, inner, E, nullptr, kActNone, q32, nullptr);
    {
      const int ld = L * 2 * inner, koff = l * 2 * inner, voff = koff + inner, heads = c.dec_heads;
      const float scale = 1.0f / sqrtf(static_cast<float>(c.dec_dim_head));
      S.push_back([=](const RunCtx&, cudaStream_t st) -> int {
        dec_cross_attn_kernel<192><<<B * heads, 192, 0, st>>>(q32, kv, ld, koff, voff, scale, att16, heads);
        THMR_CUDA(cudaGetLastError());
        return THMR_OK;
      });
    }
    linear(att16, inner, B, dw.ca_out_w, E, inner, dw.ca_out_b, kActNone, tok, nullptr, tok);
    ln(tok, dw.ln2_g, dw.ln2_b, y16, nullptr, B, E, c.ln_eps, 0, 0);
    linear(y16, E, B, dw.ff1_w, c.dec_mlp_dim, E, dw.ff1_b, kActGelu, nullptr, hid16);
    linear(hid16, c.dec_mlp_dim, B, dw.ff2_w, E, c.dec_mlp_dim, dw.ff2_b, kActNone, tok, nullptr, tok);
  }
  // decoder output: optional tap + fp16 operand copy for the read-outs and the classifier
  S.push_back([=](const RunCtx& r, cudaStream_t st) -> int {
    if (r.out.token_out)
      THMR_CUDA(cudaMemcpyAsync(r.out.token_out, tok, sizeof(float) * B * E, cudaMemcpyDeviceToDevice, st));
    const long n4 = static_cast<long>(B) * E / 4;
    cast_f16_kernel<<<static_cast<unsigned>((n4 + 255) / 256), 256, 0, st>>>(tok, y16, n4);
    THMR_CUDA(cudaGetLastError());
    return THMR_OK;
  });
  // read-outs: decpose_grot | decpose_hands | decshape | deccam (token_head.py:99-105) in one GEMM
  linear(y16, E, B, w.readout_w, 32, E, w.readout_b, kActNone, readout, nullptr);

  // ---- token classifier (token_classifier.py:89-104)
  S.tag("cls.mixer_ops");
  linear(y16, E, B, w.mt_w, TN * CH, E, w.mt_b, kActNone, mt32, nullptr);
  ln(mt32, w.mt_ln_g, w.mt_ln_b, nullptr, cx, B, TN * CH, c.ln_eps, 1, 0);   // FCBlock: LN + ReLU -> x (B*T, H)
  for (int i = 0; i < c.cls_blocks; ++i) {
    const thmr_mixer_block& mw = e->mixer[i];
    // token mixing on the transposed (B*H, T) view (modules.py:56-59)
    ln(cx, mw.ln1_g, mw.ln1_b, yT16, nullptr, B * TN, CH, c.ln_eps, 0, TN);
    linear(yT16, TN, B * CH, mw.tok1_w, c.cls_token_inter, TN, mw.tok1_b, kActGelu, nullptr, t1);
    linear(t1, c.cls_token_inter, B * CH, mw.tok2_w, TN, c.cls_token_inter, mw.tok2_b, kActNone, yT32, nullptr);
    S.push_back([=](const RunCtx&, cudaStream_t st) -> int {
      const long n = static_cast<long>(B) * TN * CH;
      mixer_add_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(cx, yT32, nullptr, xy, B, TN, CH);
      THMR_CUDA(cudaGetLastError());
      return THMR_OK;
    });
    // channel mixing (modules.py:60-62): out = (x + y) + MLP_channel(LN2(x + y))
    ln(xy, mw.ln2_g, mw.ln2_b, z16, nullptr, B * TN, CH, c.ln_eps, 0, 0);
    linear(z16, CH, B * TN, mw.ch1_w, c.cls_hidden_inter, CH, mw.ch1_b, kActGelu, nullptr, c1);
    linear(c1, c.cls_hidden_inter, B * TN, mw.ch2_w, CH, c.cls_hidden_inter, mw.ch2_b, kActNone, cx, cx16, xy);
  }
  linear(cx16, CH, B * TN, w.mn_w, CH, CH, w.mn_b, kActNone, mn32, nullptr);
  ln(mn32, w.mn_ln_g, w.mn_ln_b, mn16, nullptr, B * TN, CH, c.ln_eps, 1, 0);
  linear(mn16, CH, B * TN, w.cls_w, NC, CH, w.cls_b, kActNone, logits, nullptr);
  S.push_back([=](const RunCtx& r, cudaStream_t st) -> int {
    float* p32 = r.out.cls_logits_softmax ? r.out.cls_logits_softmax : probs_fallback;
    // pad rows of p16 stay zero: they are cleared once at plan time and never written
    return softmax_rows_launch(logits, p32, p16, B * TN, NC, TN, Lp0, PAD, st);
  });

  S.tag("tok.decoder_ops");
  // ---- tokenizer: soft codebook lookup + Conv1d decoder (vanilla_pose_vqvae.py:294-297, 135-154)
  {
    GemmDesc d;   // dequantize_logits on the padded layout (pad rows are zero -> zero output rows)
    d.A = p16; d.lda = NC; d.a_rows = static_cast<long long>(B) * Lp0;
    d.B = static_cast<const __half*>(w.codebook_t); d.ldb = NC;
    d.M = B * Lp0; d.N = c.code_dim; d.K = NC;
    d.out16 = d16; d.ld16 = c.code_dim;
    add_gemm(d);
  }
  auto conv = [&](const __half* in, int Lcur, int cin, const thmr_conv& cw, int cout, int dil, int taps, int act,
                  int act32, float* o32, int ld32, __half* o16, const float* resid) {
    const int Lp = Lcur + 2 * PAD;
    GemmDesc d;
    d.A = in; d.lda = cin; d.a_rows = static_cast<long long>(B) * Lp;
    d.B = static_cast<const __half*>(cw.w); d.ldb = taps * cin;
    d.M = B * Lp; d.N = cout; d.K = taps * cin;
    d.bias = cw.b; d.act = act; d.act32 = act32;
    d.resid = resid; d.ldr = cout;
    d.out32 = o32; d.ld32 = ld32; d.out16 = o16; d.ld16 = cout;
    if (taps > 1) { d.taps = taps; d.cin = cin; d.tap_row0 = -dil; d.tap_stride = dil; }
    d.seq_pitch = Lp; d.seq_lo = PAD; d.seq_hi = PAD + Lcur;
    add_gemm(d);
  };
  int Lcur = TN;
  conv(d16, Lcur, c.code_dim, w.conv_in, W, 1, 3, kActRelu, 0, nullptr, 0, bufA, nullptr);
  for (int u = 0; u < c.n_upsample; ++u) {
    const int Lout = c.upsample_sizes[u], Lin = Lcur;
    S.push_back([=](const RunCtx&, cudaStream_t st) -> int {
      const long n = static_cast<long>(B) * (Lout + 2 * PAD) * (W / 8);
      upsample_rows_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(bufA, bufB, B, Lin, Lout, PAD, W / 8);
      THMR_CUDA(cudaGetLastError());
      return THMR_OK;
    });
    Lcur = Lout;
    const bool last = (u == c.n_upsample - 1);
    conv(bufB, Lcur, W, w.conv_up[u], W, 1, 3, kActRelu, last ? 1 : 0, last ? x32 : nullptr, W, bufA, nullptr);
  }
  // Resnet1D (resnet.py:51-82): x = x + conv1x1(relu(conv3_dil(relu(x)))), stored order = dilation descending
  for (int dd = 0; dd < c.tok_depth; ++dd) {
    int dil = 1;
    for (int k = 0; k < c.tok_depth - 1 - dd; ++k) dil *= c.tok_dilation_rate;
    conv(bufA, Lcur, W, w.res_conv1[dd], W, dil, 3, kActRelu, 0, nullptr, 0, bufB, nullptr);
    const bool lastb = (dd == c.tok_depth - 1);
    conv(bufB, Lcur, W, w.res_conv2[dd], W, 1, 1, lastb ? kActNone : kActRelu, 0, x32, W, bufA, x32);
  }
  conv(bufA, Lcur, W, w.conv_post, W, 1, 3, kActNone, 0, nullptr, 0, bufB, nullptr);
  conv(bufB, Lcur, W, w.conv_out, 6, 1, 3, kActNone, 0, out6, 8, nullptr, nullptr);

  const int s = add_tail_step(S, e, B, tail, readout, out6);
  if (s != THMR_OK) err = s;
  *status = err;
  // zero the padded fp16 probability buffer once (pad rows are never written afterwards)
  if (err == THMR_OK) {
    cudaError_t ce = cudaMemsetAsync(p16, 0, static_cast<size_t>(B) * Lp0 * NC * sizeof(__half), stream);
    if (ce == cudaSuccess) ce = cudaMemsetAsync(skf, 0, n_skf * sizeof(unsigned), stream);
    if (ce == cudaSuccess) ce = cudaMemsetAsync(stamps, 0, kMaxStamps * sizeof(unsigned long long), stream);
    if (ce != cudaSuccess) *status = fail(THMR_ERR_CUDA, "cudaMemsetAsync(p16 / flags): %s", cudaGetErrorString(ce));
  }
  return total;
}

}  // namespace thmr
