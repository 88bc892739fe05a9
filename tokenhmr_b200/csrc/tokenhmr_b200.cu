// Single translation unit of libtokenhmr_b200.so: device kernels (*.cuh) + the extern "C" ABI
// declared in include/tokenhmr_b200.h.
#include <algorithm>
#include <new>

#include "comm.cuh"
#include "common.cuh"
#include "engine.cuh"
#include "engine_strict.cuh"
#include "eval_kernels.cuh"
#include "preproc.cuh"
#include "tok_encoder.cuh"

using namespace thmr;

namespace {

template <typename T>
int dev_alloc(T** p, size_t n) {
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(p), std::max<size_t>(n, 1) * sizeof(T));
  if (e != cudaSuccess) return fail(THMR_ERR_NOMEM, "cudaMalloc(%zu bytes) failed: %s", n * sizeof(T), cudaGetErrorString(e));
  return THMR_OK;
}
template <typename T>
int dev_upload(T** p, const std::vector<T>& h) {
  THMR_TRY(dev_alloc(p, h.size()));
  if (!h.empty()) THMR_CUDA(cudaMemcpy(*p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
  return THMR_OK;
}
template <typename T>
int dev_clone(T** p, const T* src, size_t n) {
  THMR_TRY(dev_alloc(p, n));
  THMR_CUDA(cudaMemcpy(*p, src, n * sizeof(T), cudaMemcpyDefault));
  return THMR_OK;
}

}  // namespace

extern "C" {

int thmr_abi_version(void) { return 5; }

const char* thmr_last_error(void) { return last_error_buf(); }

int thmr_check_device_flags(void) {
  THMR_CUDA(cudaDeviceSynchronize());
  unsigned int flag = 0;
  THMR_CUDA(cudaMemcpyFromSymbol(&flag, g_pipeline_timeout, sizeof(flag)));
  if (flag) {
    unsigned int zero = 0;
    THMR_CUDA(cudaMemcpyToSymbol(g_pipeline_timeout, &zero, sizeof(zero)));
    return fail(THMR_ERR_TIMEOUT, "device pipeline wait timed out (mbarrier never completed)");
  }
  THMR_CUDA(cudaMemcpyFromSymbol(&flag, g_strict_overflow, sizeof(flag)));
  if (flag) {
    unsigned int zero = 0;
    THMR_CUDA(cudaMemcpyToSymbol(g_strict_overflow, &zero, sizeof(zero)));
    return fail(THMR_ERR_INVALID, "strict mode: an activation left the split-fp16 range (|a| >= 4094 or NaN)");
  }
  return THMR_OK;
}

// ------------------------------------------------------------------------------------------ GEMM / conv
int thmr_gemm_f16(const void* A, int lda, const void* B, int ldb, int M, int N, int K, const float* bias,
                  const float* resid, int ldr, int act, float* out32, int ld32, void* out16, int ld16, int block_n,
                  void* stream) {
  THMR_CHECK(A && B, "gemm: null operand");
  GemmDesc d;
  d.A = static_cast<const __half*>(A); d.lda = lda; d.a_rows = M;
  d.B = static_cast<const __half*>(B); d.ldb = ldb;
  d.M = M; d.N = N; d.K = K;
  d.bias = bias; d.resid = resid; d.ldr = ldr; d.act = act;
  d.out32 = out32; d.ld32 = ld32; d.out16 = static_cast<__half*>(out16); d.ld16 = ld16;
  d.force_bn = block_n;
  if (resid && resid == out32) d.sk_flags = default_sk_flags(gemm_sk_flag_count(M, N));
  GemmPlan plan;
  THMR_TRY(gemm_make_plan(d, &plan));
  return gemm_launch(plan, static_cast<cudaStream_t>(stream));
}

int thmr_conv1d_k3_f16(const void* x, int B, int L, int pad, int Cin, const void* w, int Cout, const float* bias,
                       int dilation, int act, float* out32, void* out16, void* stream) {
  THMR_CHECK(x && w && B > 0 && L > 0, "conv1d: bad arguments");
  THMR_CHECK(pad >= dilation && dilation >= 1, "conv1d: pad %d < dilation %d", pad, dilation);
  const int Lp = L + 2 * pad;
  GemmDesc d;
  d.A = static_cast<const __half*>(x); d.lda = Cin; d.a_rows = static_cast<long long>(B) * Lp;
  d.B = static_cast<const __half*>(w); d.ldb = 3 * Cin;
  d.M = B * Lp; d.N = Cout; d.K = 3 * Cin;
  d.bias = bias; d.act = act;
  d.out32 = out32; d.ld32 = Cout; d.out16 = static_cast<__half*>(out16); d.ld16 = Cout;
  d.taps = 3; d.cin = Cin; d.tap_row0 = -dilation; d.tap_stride = dilation;
  d.seq_pitch = Lp; d.seq_lo = pad; d.seq_hi = pad + L;
  GemmPlan plan;
  THMR_TRY(gemm_make_plan(d, &plan));
  return gemm_launch(plan, static_cast<cudaStream_t>(stream));
}

int thmr_layernorm(const float* x, const float* gamma, const float* beta, int R, int C, float eps, int relu,
                   void* y16, float* y32, void* stream) {
  THMR_CHECK(x && gamma && beta && (y16 || y32), "layernorm: null argument");
  return layernorm_launch(x, gamma, beta, static_cast<__half*>(y16), 0, y32, R, C, eps, relu, 0,
                          static_cast<cudaStream_t>(stream));
}

int thmr_vit_attention(const void* qkv, int B, int heads, void* out, float* dbg_scores, void* stream) {
  THMR_CHECK(qkv && out, "attention: null argument");
  AttnPlan plan;
  THMR_TRY(attention_make_plan(static_cast<const __half*>(qkv), 3 * heads * kAttHeadDim, B, heads,
                               static_cast<__half*>(out), heads * kAttHeadDim, dbg_scores, &plan));
  return attention_dispatch(plan, static_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------------------------------ VQ
// Screened (two-pass) arg-min, vq.cuh, for Q >= 8192.  THMR_VQ_SCREEN=0/1 selects the single exact pass / the screened
// path (read on every call, so that a test can compare the two in one process); both return identical indices.
constexpr int kVqScreenDefault = 1;
static bool vq_screen_enabled() {
  const char* e = getenv("THMR_VQ_SCREEN");
  return (e ? atoi(e) : kVqScreenDefault) != 0;
}
struct VqWs {
  __half* xs; __half* cs; float* x2; float* c2;                  // exact path / exact pass
  __half* xh; float* x2f; int* rows; int* count; float* cmax2;   // screened path
};
static void vq_carve(Bump& bp, int64_t Q, int K, int D, bool screen, VqWs* w) {
  memset(w, 0, sizeof(*w));
  const int64_t cap = screen ? (Q < kVqExactCap ? Q : kVqExactCap) : Q;
  w->xs = bp.take<__half>(static_cast<size_t>(cap) * 3 * D);
  w->cs = bp.take<__half>(static_cast<size_t>(K) * 3 * D);
  w->x2 = bp.take<float>(Q);
  w->c2 = bp.take<float>(K);
  if (screen) {
    w->xh = bp.take<__half>(static_cast<size_t>(Q < kVqScreenChunk ? Q : kVqScreenChunk) * D);
    w->x2f = bp.take<float>(cap);
    w->rows = bp.take<int>(Q);
    w->count = bp.take<int>(4);
    w->cmax2 = bp.take<float>(4);
  }
}

size_t thmr_vq_workspace_bytes(int64_t Q, int K, int D) {
  // the larger of the two layouts, so that the environment switch never invalidates a caller's buffer
  size_t need = 0;
  for (int screen = 0; screen < 2; ++screen) {
    Bump bp(nullptr);
    VqWs w;
    vq_carve(bp, Q, K, D, screen != 0, &w);
    if (bp.off > need) need = bp.off;
  }
  return (need + 1023) & ~size_t(1023);
}

int thmr_vq_argmin(const float* x, int64_t Q, const float* codebook, int K, int D, int64_t* idx, void* workspace,
                   void* stream) {
  THMR_CHECK(x && codebook && idx && workspace, "vq_argmin: null argument");
  THMR_CHECK(D % 64 == 0 && Q > 0 && K > 0 && K % 4 == 0 && Q < (1ll << 31), "vq_argmin: unsupported shape Q=%lld K=%d D=%d",
             (long long)Q, K, D);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool screen = vq_screen_enabled() && Q >= 8192 && K % 32 == 0;
  Bump bp(workspace);
  VqWs w;
  vq_carve(bp, Q, K, D, screen, &w);
  vq_split_rows_kernel<<<static_cast<unsigned>((K + 7) / 8), 256, 0, st>>>(codebook, w.cs, w.c2, K, D, 0);
  THMR_CUDA(cudaGetLastError());
  GemmDesc d;
  d.B = w.cs; d.ldb = 3 * D; d.N = K;
  d.alpha = 1.0f / (kVqScale * kVqScale);
  d.argmin_out = reinterpret_cast<long long*>(idx); d.col_sq = w.c2;
  d.force_bn = 256;
  GemmPlan plan;
  if (!screen) {
    vq_split_rows_kernel<<<static_cast<unsigned>((Q + 7) / 8), 256, 0, st>>>(x, w.xs, w.x2, Q, D, 1);
    THMR_CUDA(cudaGetLastError());
    d.A = w.xs; d.lda = 3 * D; d.a_rows = Q;
    d.M = static_cast<int>(Q); d.K = 3 * D;
    d.row_sq = w.x2;
    THMR_TRY(gemm_make_plan(d, &plan));
    return gemm_launch(plan, st);
  }
  // ---- pass 1: one fp16 product per pair (the first D columns of the split codebook are its hi part), L2-sized chunks
  vq_screen_prep_kernel<<<1, 256, 0, st>>>(w.c2, K, w.cmax2, w.count);
  THMR_CUDA(cudaGetLastError());
  for (int64_t q0 = 0; q0 < Q; q0 += kVqScreenChunk) {
    const int64_t n = (Q - q0) < kVqScreenChunk ? (Q - q0) : kVqScreenChunk;
    vq_hi_rows_kernel<<<static_cast<unsigned>((n + 7) / 8), 256, 0, st>>>(x + q0 * D, w.xh, w.x2 + q0, n, D);
    THMR_CUDA(cudaGetLastError());
    GemmDesc s = d;
    s.A = w.xh; s.lda = D; s.a_rows = n;
    s.M = static_cast<int>(n); s.K = D;
    s.argmin_out = reinterpret_cast<long long*>(idx) + q0; s.row_sq = w.x2 + q0;
    s.screen_rows = w.rows; s.screen_count = w.count; s.screen_cmax2 = w.cmax2;
    s.screen_rel = kVqScreenRel; s.screen_abs = kVqScreenAbs; s.screen_row0 = static_cast<int>(q0);
    THMR_TRY(gemm_make_plan(s, &plan));
    THMR_TRY(gemm_launch(plan, st));
  }
  // ---- pass 2: the queued rows through the exact split-precision GEMM, kVqExactCap rows per round (the count is only
  //      known on the device: every round is launched, rounds past the end find zero rows)
  const int64_t cap = Q < kVqExactCap ? Q : kVqExactCap;
  for (int64_t off = 0; off < Q; off += cap) {
    vq_gather_split_kernel<<<num_sms() * 4, 256, 0, st>>>(x, w.rows, w.count, static_cast<int>(off), static_cast<int>(cap),
                                                         w.xs, w.x2f, D);
    THMR_CUDA(cudaGetLastError());
    GemmDesc e = d;
    e.A = w.xs; e.lda = 3 * D; e.a_rows = cap;
    e.M = static_cast<int>(cap); e.K = 3 * D;
    e.row_sq = w.x2f;
    e.row_map = w.rows + off; e.m_dev = w.count; e.m_dev_off = static_cast<int>(off);
    THMR_TRY(gemm_make_plan(e, &plan));
    THMR_TRY(gemm_launch(plan, st));
  }
  return THMR_OK;
}

int thmr_vq_dequantize(const int64_t* idx, int64_t Q, const float* codebook, int D, float* out, void* stream) {
  THMR_CHECK(idx && codebook && out && D % 4 == 0, "vq_dequantize: bad argument");
  const long n = Q * (D / 4);
  vq_gather_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const long long*>(idx), codebook, out, Q, D / 4);
  THMR_CUDA(cudaGetLastError());
  return THMR_OK;
}

int thmr_vq_dequant_logits(const void* logits16, int64_t Q, int K, const void* codebook_t16, int D, float* out,
                           void* stream) {
  return thmr_gemm_f16(logits16, K, codebook_t16, K, static_cast<int>(Q), D, K, nullptr, nullptr, 0, THMR_ACT_NONE, out,
                       D, nullptr, 0, 0, stream);
}

int thmr_rot6d_to_rotmat(const float* x6, int64_t N, float* rot, void* stream) {
  THMR_CHECK(x6 && rot, "rot6d: null argument");
  rot6d_kernel<<<static_cast<unsigned>((N + 127) / 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(x6, rot, N);
  THMR_CUDA(cudaGetLastError());
  return THMR_OK;
}

// ------------------------------------------------------------------------------------------ evaluation
int thmr_regress_joints(const float* jreg, int J, const float* verts, int V, int B, float* joints, void* stream) {
  THMR_CHECK(jreg && verts && joints, "regress_joints: null argument");
  THMR_CHECK(J > 0 && V > 0 && B > 0, "regress_joints: bad shape J=%d V=%d B=%d", J, V, B);
  regress_joints_kernel<<<B * J, 256, 0, static_cast<cudaStream_t>(stream)>>>(jreg, verts, joints, J, V);
  THMR_CUDA(cudaGetLastError());
  return THMR_OK;
}

int thmr_eval_pose(const float* pred_kp, const float* gt_kp, int gt_stride, int J, const int32_t* keypoint_list, int K,
                   int pelvis_a, int pelvis_b, const float* pred_verts, const float* gt_verts, int V, int B,
                   float* mpjpe, float* re, float* pve, void* stream) {
  THMR_CHECK(pred_kp && gt_kp && keypoint_list && mpjpe && re, "eval_pose: null argument");
  THMR_CHECK(B > 0 && J > 0 && K > 0 && K <= kEvalMaxKp, "eval_pose: bad shape B=%d J=%d K=%d (K <= %d)", B, J, K,
             kEvalMaxKp);
  THMR_CHECK(gt_stride == 3 || gt_stride == 4, "eval_pose: gt_stride %d (3 or 4)", gt_stride);
  THMR_CHECK(pelvis_a >= 0 && pelvis_a < J && pelvis_b >= 0 && pelvis_b < J, "eval_pose: pelvis index out of range");
  THMR_CHECK(pve == nullptr || (pred_verts && gt_verts && V > 0), "eval_pose: pve needs both vertex sets");
  eval_pose_kernel<<<B, 256, 0, static_cast<cudaStream_t>(stream)>>>(pred_kp, gt_kp, gt_stride, J, keypoint_list, K,
                                                                     pelvis_a, pelvis_b, pred_verts, gt_verts, V, mpjpe,
                                                                     re, pve);
  THMR_CUDA(cudaGetLastError());
  return THMR_OK;
}

int thmr_cam_crop_to_full(const float* cam, const float* box_center, const float* box_size, const float* img_size,
                          float focal_length, int B, float* full_cam, void* stream) {
  THMR_CHECK(cam && box_center && box_size && img_size && full_cam, "cam_crop_to_full: null argument");
  THMR_CHECK(B > 0, "cam_crop_to_full: bad batch %d", B);
  cam_crop_to_full_kernel<<<(B + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(cam, box_center, box_size,
                                                                                       img_size, focal_length, full_cam, B);
  THMR_CUDA(cudaGetLastError());
  return THMR_OK;
}

// ------------------------------------------------------------------------------------------ pre-processing
size_t thmr_preprocess_workspace_bytes(int img_h, int img_w, int n) {
  if (img_h <= 0 || img_w <= 0 || n < 0) return 0;
  return pre_layout(img_h, img_w, n).total + 256;
}

// Host half of the pre-processing (no CUDA call): box -> centre / size / blur sigma / inverse affine map, in float32
// and double exactly as the reference computes them.
int thmr_preprocess_plan(const float* boxes_host, int n, const thmr_preproc_cfg* cfg, float* box_center_host,
                         float* box_size_host, float* sigma_host, double* inv_affine_host) {
  THMR_CHECK(boxes_host && cfg, "preprocess_plan: null argument");
  THMR_CHECK(n > 0, "preprocess_plan: no boxes");
  const int S = cfg->image_size;
  THMR_CHECK(S >= 16 && S <= 4096, "preprocess_plan: image_size %d", S);
  for (int i = 0; i < n; ++i) {
    const float* b = boxes_host + 4 * i;
    THMR_CHECK(b[2] > b[0] && b[3] > b[1], "preprocess: box %d is empty (%g,%g,%g,%g)", i, b[0], b[1], b[2], b[3]);
    volatile float sx_ = b[2] + b[0], sy_ = b[3] + b[1];
    const float cx = sx_ / 2.0f, cy = sy_ / 2.0f;
    volatile float dw = b[2] - b[0], dh = b[3] - b[1];
    volatile float sw = dw / 200.0f, sh = dh / 200.0f;           // self.scale
    volatile float w = sw * 200.0f, h = sh * 200.0f;             // scale * 200
    const float bsz = pre_bbox_size(w, h, cfg->bbox_w, cfg->bbox_h);
    if (box_center_host) { box_center_host[2 * i] = cx; box_center_host[2 * i + 1] = cy; }
    if (box_size_host) box_size_host[i] = bsz;
    volatile float f1 = bsz / static_cast<float>(S);
    volatile float f = f1 / 2.0f;
    float sigma = 0.f;
    if (f > 1.1f) {
      volatile float t = f - 1.0f;
      sigma = t / 2.0f;
    }
    if (sigma_host) sigma_host[i] = sigma;
    if (inv_affine_host) {
      // gen_trans_from_patch_cv (utils.py:81-129), scale 1, rot 0
      volatile float half = bsz * 0.5f;
      float src[3][2], dst[3][2];
      src[0][0] = cx; src[0][1] = cy;
      src[1][0] = cx; src[1][1] = static_cast<float>(static_cast<double>(cy) + static_cast<double>(half));
      src[2][0] = static_cast<float>(static_cast<double>(cx) + static_cast<double>(half)); src[2][1] = cy;
      const float hs = static_cast<float>(S * 0.5);
      dst[0][0] = hs; dst[0][1] = hs; dst[1][0] = hs; dst[1][1] = hs + hs; dst[2][0] = hs + hs; dst[2][1] = hs;
      double M[6];
      THMR_CHECK(pre_get_affine(src, dst, M), "preprocess: box %d gives a singular transform", i);
      pre_invert_affine(M, inv_affine_host + 6 * i);
    }
  }
  return THMR_OK;
}

int thmr_preprocess_boxes(const uint8_t* img_bgr, int img_h, int img_w, int64_t pitch_bytes, const float* boxes_host,
                          int n, const thmr_preproc_cfg* cfg, float* out_img, uint8_t* out_patch_u8,
                          float* box_center_host, float* box_size_host, float* sigma_host, void* workspace,
                          void* stream) {
  THMR_CHECK(img_bgr && boxes_host && cfg && out_img && workspace, "preprocess: null argument");
  THMR_CHECK(img_h > 1 && img_w > 1 && pitch_bytes >= 3LL * img_w, "preprocess: bad image %dx%d pitch %lld", img_h,
             img_w, static_cast<long long>(pitch_bytes));
  THMR_CHECK(n > 0, "preprocess: no boxes");
  const int S = cfg->image_size;
  for (int c = 0; c < 3; ++c) THMR_CHECK(cfg->std[c] > 0, "preprocess: std[%d] must be positive", c);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
  const PreLayout L = pre_layout(img_h, img_w, n);

  std::vector<uint8_t> blob(L.tmp_off, 0);
  PrePerson* persons = reinterpret_cast<PrePerson*>(blob.data() + L.persons_off);
  int* which = reinterpret_cast<int*>(blob.data() + L.which_off);
  float* lut = reinterpret_cast<float*>(blob.data() + L.lut_off);
  double* wts = reinterpret_cast<double*>(blob.data() + L.wts_off);
  double mean[3], sd[3];                                         // RGB order, 0..255 scale (vitdet_dataset.py:32-33)
  for (int c = 0; c < 3; ++c) { mean[c] = 255.0 * cfg->mean[c]; sd[c] = 255.0 * cfg->std[c]; }
  for (int c = 0; c < 3; ++c)
    for (int v = 0; v < 256; ++v) lut[c * 256 + v] = static_cast<float>((static_cast<double>(v) - mean[c]) / sd[c]);
  std::vector<float> sigma(n, 0.f), size(n);
  std::vector<double> inv(6 * static_cast<size_t>(n));
  std::vector<int> radius(n, 0);
  THMR_TRY(thmr_preprocess_plan(boxes_host, n, cfg, box_center_host, size.data(), sigma.data(), inv.data()));
  int n_u8 = 0;
  for (int i = 0; i < n; ++i) {
    if (box_size_host) box_size_host[i] = size[i];
    if (sigma_host) sigma_host[i] = sigma[i];
    memcpy(persons[i].iM, &inv[6 * static_cast<size_t>(i)], sizeof(double) * 6);
    if (sigma[i] > 0.f) {
      const double sg = static_cast<double>(sigma[i]);
      const int r = static_cast<int>(4.0 * sg + 0.5);
      THMR_CHECK(2 * r + 1 <= kPreMaxTaps, "preprocess: box %d needs a %d-tap blur (max %d)", i, 2 * r + 1, kPreMaxTaps);
      radius[i] = r;
      double* wi = wts + static_cast<size_t>(i) * kPreMaxTaps;
      double sum = 0;
      for (int k = -r; k <= r; ++k) { wi[k + r] = exp(-0.5 / (sg * sg) * static_cast<double>(k * k)); sum += wi[k + r]; }
      for (int k = 0; k <= 2 * r; ++k) wi[k] /= sum;
    } else {
      which[n_u8++] = i;
    }
  }
  THMR_CUDA(cudaMemcpyAsync(ws, blob.data(), blob.size(), cudaMemcpyHostToDevice, st));   // pageable: staged before return
  const PrePerson* d_persons = reinterpret_cast<const PrePerson*>(ws + L.persons_off);
  const int* d_which = reinterpret_cast<const int*>(ws + L.which_off);
  const float* d_lut = reinterpret_cast<const float*>(ws + L.lut_off);
  const double* d_wts = reinterpret_cast<const double*>(ws + L.wts_off);
  float* tmp = reinterpret_cast<float*>(ws + L.tmp_off);
  float* blur = reinterpret_cast<float*>(ws + L.blur_off);
  const int px_blocks = (S * S + 255) / 256;
  if (n_u8 > 0) {
    preproc_warp_u8_kernel<<<dim3(px_blocks, n_u8), 256, 0, st>>>(img_bgr, img_h, img_w, pitch_bytes, d_persons, d_which,
                                                                 d_lut, S, out_img, out_patch_u8);
    THMR_CUDA(cudaGetLastError());
  }
  for (int i = 0; i < n; ++i) {
    if (sigma[i] <= 0.f) continue;
    // source region the remap can touch: the box (+2 px for the bilinear footprint and rounding), clipped
    const double half = 0.5 * static_cast<double>(size[i]);
    const double cx = 0.5 * (static_cast<double>(boxes_host[4 * i]) + boxes_host[4 * i + 2]);
    const double cy = 0.5 * (static_cast<double>(boxes_host[4 * i + 1]) + boxes_host[4 * i + 3]);
    const int r = radius[i];
    int x0 = static_cast<int>(floor(cx - half)) - 3, x1 = static_cast<int>(ceil(cx + half)) + 4;
    int y0 = static_cast<int>(floor(cy - half)) - 3, y1 = static_cast<int>(ceil(cy + half)) + 4;
    x0 = std::max(x0, 0); y0 = std::max(y0, 0); x1 = std::min(x1, img_w); y1 = std::min(y1, img_h);
    if (x0 < x1 && y0 < y1) {
      const int vx0 = std::max(x0 - r, 0), vx1 = std::min(x1 + r, img_w);    // the column pass reads +-r around x
      const long long nv = 3LL * (vx1 - vx0) * (y1 - y0), nh = 3LL * (x1 - x0) * (y1 - y0);
      const double* wi = d_wts + static_cast<size_t>(i) * kPreMaxTaps;
      preproc_gauss_kernel<0><<<static_cast<unsigned>((nv + 255) / 256), 256, 0, st>>>(img_bgr, pitch_bytes, img_h, img_w,
                                                                                     wi, r, vx0, vx1, y0, y1, tmp);
      THMR_CUDA(cudaGetLastError());
      preproc_gauss_kernel<1><<<static_cast<unsigned>((nh + 255) / 256), 256, 0, st>>>(tmp, 0, img_h, img_w, wi, r, x0, x1,
                                                                                     y0, y1, blur);
      THMR_CUDA(cudaGetLastError());
    }
    PrePerson pp;
    memcpy(&pp, &persons[i], sizeof(pp));
    preproc_warp_f32_kernel<<<px_blocks, 256, 0, st>>>(blur, img_h, img_w, pp, i, S, mean[0], mean[1], mean[2], sd[0],
                                                       sd[1], sd[2], out_img);
    THMR_CUDA(cudaGetLastError());
  }
  return THMR_OK;
}

// ------------------------------------------------------------------------------------------ tokenizer encoder
int thmr_tok_encoder_create(const thmr_tok_encoder_desc* d, thmr_tok_encoder** out) {
  THMR_CHECK(d && out, "tok_encoder_create: null argument");
  THMR_CHECK(d->joints > 0 && d->in_dim > 0 && d->in_dim <= kEncCin0, "tok_encoder: joints %d in_dim %d (<= %d)", d->joints,
             d->in_dim, kEncCin0);
  THMR_CHECK(d->width % 64 == 0 && d->code_dim % 64 == 0 && d->nb_code % 4 == 0, "tok_encoder: width %d code_dim %d nb_code %d",
             d->width, d->code_dim, d->nb_code);
  THMR_CHECK(d->depth >= 1 && d->depth <= 8 && d->size_mul >= 1 && d->size_mul <= 8, "tok_encoder: depth %d size_mul %d",
             d->depth, d->size_mul);
  THMR_CHECK(d->conv_in.w && d->conv_down.w && d->conv_out.w && d->codebook, "tok_encoder: missing weights");
  for (int i = 0; i < d->size_mul; ++i) THMR_CHECK(d->conv_up[i].w, "tok_encoder: conv_up[%d] missing", i);
  for (int i = 0; i < d->depth; ++i)
    THMR_CHECK(d->res_conv1[i].w && d->res_conv2[i].w, "tok_encoder: resnet block %d missing", i);
  thmr_tok_encoder* e = new thmr_tok_encoder();
  e->d = *d;
  *out = e;
  return THMR_OK;
}

void thmr_tok_encoder_destroy(thmr_tok_encoder* e) { delete e; }

int thmr_tok_encoder_num_tokens(const thmr_tok_encoder* e) {
  if (!e) return 0;
  int Lmax, T;
  enc_seq_lens(e->d, &Lmax, &T);
  return T;
}

size_t thmr_tok_encoder_workspace_bytes(const thmr_tok_encoder* e, int batch) {
  if (!e || batch <= 0) return 0;
  EncWs ws;
  enc_carve(e->d, nullptr, batch, &ws);
  return ws.total + 1024;
}

int thmr_tok_encode(const thmr_tok_encoder* e, const float* pose6d, int B, int64_t* code_idx, float* latent,
                    void* workspace, void* stream) {
  THMR_CHECK(e && pose6d && code_idx && workspace, "tok_encode: null argument");
  THMR_CHECK(B > 0, "tok_encode: bad batch %d", B);
  void* ws = reinterpret_cast<void*>((reinterpret_cast<uintptr_t>(workspace) + 1023) & ~uintptr_t(1023));
  return enc_run(e, pose6d, B, code_idx, latent, ws, static_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------------------------------ SMPL
void thmr_smpl_destroy(thmr_smpl* s) {
  if (!s) return;
  SmplModel& m = s->m;
  cudaFree(m.v_template); cudaFree(m.shapedirs); cudaFree(m.J_template); cudaFree(m.J_shapedirs);
  cudaFree(m.posedirsT); cudaFree(m.w_idx); cudaFree(m.w_val); cudaFree(m.jx_ptr); cudaFree(m.jx_idx);
  cudaFree(m.jx_val); cudaFree(m.extra_vid); cudaFree(m.joint_map); cudaFree(s->parents_dev);
  delete s;
}

int thmr_smpl_create(const thmr_smpl_desc* d, thmr_smpl** out) {
  THMR_CHECK(d && out, "smpl_create: null argument");
  THMR_CHECK(d->num_verts > 0 && d->num_betas > 0 && d->num_betas <= 10, "smpl_create: V=%d betas=%d", d->num_verts,
             d->num_betas);
  THMR_CHECK(d->v_template && d->shapedirs && d->posedirs && d->J_regressor && d->lbs_weights && d->parents_host &&
                 d->extra_vertex_ids_host && d->joint_map_host,
             "smpl_create: missing tensor");
  thmr_smpl* s = new (std::nothrow) thmr_smpl();
  if (!s) return fail(THMR_ERR_NOMEM, "smpl_create: out of host memory");
  SmplModel& m = s->m;
  const int V = d->num_verts, nb = d->num_betas;
  m.V = V; m.nb = nb; m.n_extra = d->joint_regressor_extra ? d->n_extra : 0;
  auto bail = [&](int code) { thmr_smpl_destroy(s); return code; };
#define SM_TRY(e) do { int _r = (e); if (_r != THMR_OK) return bail(_r); } while (0)
  SM_TRY(dev_clone(&m.v_template, d->v_template, static_cast<size_t>(V) * 3));
  SM_TRY(dev_clone(&m.shapedirs, d->shapedirs, static_cast<size_t>(V) * 3 * nb));
  for (int j = 0; j < kSmplJ; ++j) m.parents[j] = d->parents_host[j];
  SM_TRY(dev_upload(&s->parents_dev, std::vector<int>(m.parents, m.parents + kSmplJ)));
  // J_template / J_shapedirs
  float* Jreg = nullptr;
  SM_TRY(dev_clone(&Jreg, d->J_regressor, static_cast<size_t>(kSmplJ) * V));
  SM_TRY(dev_alloc(&m.J_template, kSmplJ * 3));
  SM_TRY(dev_alloc(&m.J_shapedirs, static_cast<size_t>(kSmplJ) * 3 * nb));
  smpl_jreg_kernel<<<kSmplJ * 3 * (nb + 1), 256>>>(Jreg, m.v_template, m.shapedirs, m.J_template, m.J_shapedirs, V, nb);
  // posedirs -> transposed split fp16
  float* pd = nullptr;
  SM_TRY(dev_clone(&pd, d->posedirs, static_cast<size_t>(kSmplPF) * 3 * V));
  {
    // rows padded to a multiple of 4 (zero rows): the blend GEMM's N equals the 16-byte aligned offsets pitch
    const size_t rows_pad = (static_cast<size_t>(3) * V + 3) / 4 * 4;
    SM_TRY(dev_alloc(&m.posedirsT, rows_pad * 3 * kSmplPFPad));
    if (cudaMemset(m.posedirsT, 0, rows_pad * 3 * kSmplPFPad * sizeof(__half)) != cudaSuccess)
      return bail(fail(THMR_ERR_CUDA, "smpl_create: memset posedirs"));
  }
  {
    const long n = static_cast<long>(3) * V * kSmplPFPad;
    smpl_pack_posedirs_kernel<<<static_cast<unsigned>((n + 255) / 256), 256>>>(pd, m.shapedirs, m.v_template, nb,
                                                                               m.posedirsT, 3 * V);
  }
  cudaError_t ce = cudaDeviceSynchronize();
  cudaFree(Jreg);
  cudaFree(pd);
  if (ce != cudaSuccess) return bail(fail(THMR_ERR_CUDA, "smpl_create: %s", cudaGetErrorString(ce)));
  // skinning weights -> ELL
  {
    std::vector<float> W(static_cast<size_t>(V) * kSmplJ);
    if (cudaMemcpy(W.data(), d->lbs_weights, W.size() * sizeof(float), cudaMemcpyDefault) != cudaSuccess)
      return bail(fail(THMR_ERR_CUDA, "smpl_create: copy lbs_weights"));
    int ell = 1;
    for (int v = 0; v < V; ++v) {
      int n = 0;
      for (int j = 0; j < kSmplJ; ++j) n += (W[static_cast<size_t>(v) * kSmplJ + j] != 0.f);
      ell = std::max(ell, n);
    }
    std::vector<int> idx(static_cast<size_t>(V) * ell, 0);
    std::vector<float> val(static_cast<size_t>(V) * ell, 0.f);
    for (int v = 0; v < V; ++v) {
      int n = 0;
      for (int j = 0; j < kSmplJ; ++j) {
        const float w = W[static_cast<size_t>(v) * kSmplJ + j];
        if (w != 0.f) { idx[static_cast<size_t>(v) * ell + n] = j; val[static_cast<size_t>(v) * ell + n] = w; ++n; }
      }
    }
    m.ell = ell;
    SM_TRY(dev_upload(&m.w_idx, idx));
    SM_TRY(dev_upload(&m.w_val, val));
  }
  // extra joint regressor -> CSR
  {
    std::vector<int> ptr(1, 0), idx;
    std::vector<float> val;
    if (m.n_extra > 0) {
      std::vector<float> Jx(static_cast<size_t>(m.n_extra) * V);
      if (cudaMemcpy(Jx.data(), d->joint_regressor_extra, Jx.size() * sizeof(float), cudaMemcpyDefault) != cudaSuccess)
        return bail(fail(THMR_ERR_CUDA, "smpl_create: copy joint_regressor_extra"));
      for (int r = 0; r < m.n_extra; ++r) {
        for (int v = 0; v < V; ++v) {
          const float w = Jx[static_cast<size_t>(r) * V + v];
          if (w != 0.f) { idx.push_back(v); val.push_back(w); }
        }
        ptr.push_back(static_cast<int>(idx.size()));
      }
    }
    SM_TRY(dev_upload(&m.jx_ptr, ptr));
    SM_TRY(dev_upload(&m.jx_idx, idx));
    SM_TRY(dev_upload(&m.jx_val, val));
  }
  for (int i = 0; i < 21; ++i)
    if (d->extra_vertex_ids_host[i] < 0 || d->extra_vertex_ids_host[i] >= V)
      return bail(fail(THMR_ERR_INVALID, "smpl_create: extra vertex id %d out of range", d->extra_vertex_ids_host[i]));
  SM_TRY(dev_upload(&m.extra_vid, std::vector<int>(d->extra_vertex_ids_host, d->extra_vertex_ids_host + 21)));
  SM_TRY(dev_upload(&m.joint_map, std::vector<int>(d->joint_map_host, d->joint_map_host + 25)));
#undef SM_TRY
  *out = s;
  return THMR_OK;
}

size_t thmr_smpl_workspace_bytes(const thmr_smpl* s, int batch) {
  if (!s || batch <= 0) return 0;
  Bump bp(nullptr);
  SmplWs ws;
  smpl_carve(bp, s->m, batch, &ws);
  return (bp.off + 1023) & ~size_t(1023);
}

int thmr_lbs(const thmr_smpl* s, const float* pose, int pose2rot, const float* betas, int B, float* verts,
             float* joints, void* workspace, void* stream) {
  THMR_CHECK(s && pose && betas && verts && workspace && B > 0, "lbs: bad argument");
  Bump bp(workspace);
  SmplWs ws;
  smpl_carve(bp, s->m, B, &ws);
  return smpl_run(s, pose, pose2rot, betas, B, verts, joints, nullptr, nullptr, 0.f, 0.f, nullptr, nullptr, nullptr, ws,
                  nullptr, static_cast<cudaStream_t>(stream));
}

int thmr_smpl_forward(const thmr_smpl* s, const float* rotmats, const float* betas, int B, float* verts, float* joints,
                      const float* pred_cam, float focal_length, float image_size, float* cam_t, float* focal_out,
                      float* kp2d, void* workspace, void* stream) {
  THMR_CHECK(s && rotmats && betas && verts && joints && workspace && B > 0, "smpl_forward: bad argument");
  THMR_CHECK(!pred_cam || (cam_t && focal_out && kp2d), "smpl_forward: pred_cam given without camera outputs");
  Bump bp(workspace);
  SmplWs ws;
  smpl_carve(bp, s->m, B, &ws);
  return smpl_run(s, rotmats, 0, betas, B, verts, nullptr, joints, pred_cam, focal_length, image_size, cam_t, focal_out,
                  kp2d, ws, nullptr, static_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------------------------------ engine
int thmr_engine_create(const thmr_config* cfg, const thmr_weights* w, const thmr_smpl* smpl, thmr_engine** out) {
  THMR_CHECK(cfg && w && smpl && out, "engine_create: null argument");
  THMR_CHECK(cfg->vit_dim == cfg->vit_heads * kAttHeadDim, "engine_create: head_dim must be %d", kAttHeadDim);
  const int gh = (cfg->image_size + 2 * cfg->patch_pad - cfg->patch) / cfg->patch + 1;
  const int gw = (cfg->crop_w + 2 * cfg->patch_pad - cfg->patch) / cfg->patch + 1;
  THMR_CHECK(gh * gw == kAttTokens, "engine_create: %dx%d patches != %d tokens", gh, gw, kAttTokens);
  THMR_CHECK(cfg->dec_dim_head == 64 && cfg->dec_heads <= 8, "engine_create: decoder heads must be <=8 x 64");
  THMR_CHECK(cfg->n_upsample >= 1 && cfg->n_upsample <= 8 && cfg->tok_depth >= 1 && cfg->tok_depth <= 8,
             "engine_create: tokenizer depth");
  THMR_CHECK(cfg->upsample_sizes[cfg->n_upsample - 1] == cfg->tok_joints, "engine_create: last upsample != joints");
  THMR_CHECK(cfg->tok_width % 64 == 0 && cfg->code_dim % 64 == 0 && cfg->token_class_num % 8 == 0 &&
                 cfg->token_class_num <= 2048 && cfg->token_num % 8 == 0,
             "engine_create: tokenizer dims");
  int maxdil = 1;
  for (int k = 0; k < cfg->tok_depth - 1; ++k) maxdil *= cfg->tok_dilation_rate;
  THMR_CHECK(maxdil <= kTokPad, "engine_create: dilation %d exceeds sequence padding %d", maxdil, kTokPad);
  THMR_CHECK(smpl->m.nb <= 10 && smpl->m.n_extra + 25 <= 64, "engine_create: SMPL model shape");
  THMR_CHECK(w->blocks_host && w->dec_host && w->mixer_host, "engine_create: missing layer arrays");
  thmr_engine* e = new (std::nothrow) thmr_engine();
  if (!e) return fail(THMR_ERR_NOMEM, "engine_create: out of host memory");
  e->cfg = *cfg;
  e->w = *w;
  e->blocks.assign(w->blocks_host, w->blocks_host + cfg->vit_depth);
  e->dec.assign(w->dec_host, w->dec_host + cfg->dec_depth);
  e->mixer.assign(w->mixer_host, w->mixer_host + cfg->cls_blocks);
  e->w.blocks_host = nullptr; e->w.dec_host = nullptr; e->w.mixer_host = nullptr;
  e->smpl = smpl;
  *out = e;
  return THMR_OK;
}

void thmr_engine_destroy(thmr_engine* e) { delete e; }

size_t thmr_engine_workspace_bytes(const thmr_engine* e, int max_batch) {
  if (!e || max_batch <= 0) return 0;
  int st;
  if (e->cfg.strict) return engine_build_strict(const_cast<thmr_engine*>(e), nullptr, max_batch, false, &st, nullptr);
  return engine_build(const_cast<thmr_engine*>(e), nullptr, max_batch, false, &st, nullptr);
}

static int engine_prepare(thmr_engine* e, int B, void* workspace, cudaStream_t st) {
  THMR_CHECK(e && workspace && B > 0, "engine_forward: bad argument");
  THMR_CHECK((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0, "engine_forward: workspace not 1024-byte aligned");
  if (e->ws != workspace || e->B != B) {
    int status = THMR_OK;
    e->ws = nullptr;
    if (e->cfg.strict) engine_build_strict(e, workspace, B, true, &status, st);
    else engine_build(e, workspace, B, true, &status, st);
    if (status != THMR_OK) { e->steps.clear(); return status; }
    e->ws = workspace;
    e->B = B;
  }
  return THMR_OK;
}

int thmr_engine_forward(thmr_engine* e, const float* img, int B, const thmr_outputs* out, void* workspace,
                        void* stream) {
  THMR_CHECK(img && out, "engine_forward: null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  THMR_TRY(engine_prepare(e, B, workspace, st));
  RunCtx ctx{img, *out, nullptr};
  for (auto& step : e->steps) THMR_TRY(step.fn(ctx, st));
  return THMR_OK;
}

int thmr_engine_forward_stamped(thmr_engine* e, const float* img, int B, const thmr_outputs* out, void* workspace,
                                void* stream) {
  THMR_TRY(thmr_engine_forward(e, img, B, out, workspace, stream));
  THMR_CHECK(e->stamps != nullptr, "forward_stamped: this engine mode records no stamps");
  stamp_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(e->stamps + e->steps.size());
  THMR_CUDA(cudaGetLastError());
  return THMR_OK;
}

int thmr_engine_read_stamps(const thmr_engine* e, unsigned long long* host_ns, int cap) {
  THMR_CHECK(e && host_ns && e->stamps, "read_stamps: no stamps");
  const int n = static_cast<int>(e->steps.size()) + 1;
  THMR_CHECK(cap >= n && n <= kMaxStamps, "read_stamps: need room for %d entries", n);
  THMR_CUDA(cudaMemcpy(host_ns, e->stamps, sizeof(unsigned long long) * n, cudaMemcpyDeviceToHost));
  return n;
}

int thmr_engine_vit_forward(thmr_engine* e, const float* img, int B, float* tokens, void* workspace, void* stream) {
  THMR_CHECK(img && tokens, "vit_forward: null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  THMR_TRY(engine_prepare(e, B, workspace, st));
  RunCtx ctx{img, thmr_outputs{}, tokens};
  for (size_t i = 0; i < e->vit_steps; ++i) THMR_TRY(e->steps[i].fn(ctx, st));
  return THMR_OK;
}

int thmr_engine_num_steps(const thmr_engine* e) { return e ? static_cast<int>(e->steps.size()) : 0; }

int thmr_engine_step_info(const thmr_engine* e, int i, const char** name, double* flops, double* bytes) {
  THMR_CHECK(e && i >= 0 && i < static_cast<int>(e->steps.size()), "step_info: bad index");
  if (name) *name = e->steps[i].name;
  if (flops) *flops = e->steps[i].flops;
  if (bytes) *bytes = e->steps[i].bytes;
  return THMR_OK;
}

int thmr_engine_profile(thmr_engine* e, const float* img, int B, const thmr_outputs* out, void* workspace, void* stream,
                        float* step_ms, int cap) {
  THMR_CHECK(img && out && step_ms, "engine_profile: null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  THMR_TRY(engine_prepare(e, B, workspace, st));
  const int n = static_cast<int>(e->steps.size());
  THMR_CHECK(cap >= n, "engine_profile: step_ms holds %d entries, need %d", cap, n);
  std::vector<cudaEvent_t> ev(n + 1);
  for (auto& x : ev) THMR_CUDA(cudaEventCreate(&x));
  RunCtx ctx{img, *out, nullptr};
  int status = THMR_OK;
  THMR_CUDA(cudaEventRecord(ev[0], st));
  for (int i = 0; i < n && status == THMR_OK; ++i) {
    status = e->steps[i].fn(ctx, st);
    cudaEventRecord(ev[i + 1], st);
  }
  cudaError_t ce = cudaStreamSynchronize(st);
  if (status == THMR_OK && ce == cudaSuccess)
    for (int i = 0; i < n; ++i) cudaEventElapsedTime(&step_ms[i], ev[i], ev[i + 1]);
  for (auto& x : ev) cudaEventDestroy(x);
  if (ce != cudaSuccess) return fail(THMR_ERR_CUDA, "engine_profile: %s", cudaGetErrorString(ce));
  return status;
}

int thmr_engine_num_launches(const thmr_engine* e) {
  if (!e) return 0;
  int n = 0;
  for (const Step& s : e->steps) n += s.kernels;
  return n;
}

// ------------------------------------------------------------------------------------------ multi-GPU exchange
int thmr_comm_unique_id(void* id128) {
  THMR_CHECK(id128, "comm_unique_id: null argument");
  NcclApi* api = nccl_api();
  if (!api) return fail(THMR_ERR_CUDA, "libnccl.so.2 could not be loaded (%s)", dlerror() ? dlerror() : "no error text");
  NcclUniqueId id;
  THMR_NCCL(api, api->GetUniqueId(&id));
  memcpy(id128, &id, sizeof(id));
  return THMR_OK;
}

int thmr_comm_create(const void* id128, int nranks, int rank, thmr_comm** out) {
  THMR_CHECK(id128 && out, "comm_create: null argument");
  THMR_CHECK(nranks >= 1 && rank >= 0 && rank < nranks, "comm_create: rank %d of %d", rank, nranks);
  NcclApi* api = nccl_api();
  if (!api) return fail(THMR_ERR_CUDA, "libnccl.so.2 could not be loaded");
  thmr_comm* c = new (std::nothrow) thmr_comm();
  if (!c) return fail(THMR_ERR_NOMEM, "comm_create: out of host memory");
  NcclUniqueId id;
  memcpy(&id, id128, sizeof(id));
  THMR_CUDA(cudaGetDevice(&c->device));
  const int r = api->CommInitRank(&c->comm, nranks, id, rank);
  if (r != 0) {
    delete c;
    return fail(THMR_ERR_CUDA, "ncclCommInitRank(rank %d of %d) failed: %s", rank, nranks, api->GetErrorString(r));
  }
  c->nranks = nranks;
  c->rank = rank;
  *out = c;
  return THMR_OK;
}

void thmr_comm_destroy(thmr_comm* c) {
  if (!c) return;
  NcclApi* api = nccl_api();
  if (api && c->comm) api->CommDestroy(c->comm);
  delete c;
}

int thmr_comm_nranks(const thmr_comm* c) { return c ? c->nranks : 0; }
int thmr_comm_rank(const thmr_comm* c) { return c ? c->rank : -1; }

int thmr_allgather_outputs(const thmr_engine* e, thmr_comm* c, const thmr_outputs* g, int rows, void* stream) {
  THMR_CHECK(e && c && g && rows > 0, "allgather_outputs: bad argument");
  NcclApi* api = nccl_api();
  THMR_CHECK(api && c->comm, "allgather_outputs: communicator not initialised");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int nj = 25 + e->smpl->m.n_extra;
  struct Field { float* base; size_t per_image; };
  const Field fields[] = {
      {g->pred_vertices, static_cast<size_t>(e->smpl->m.V) * 3},
      {g->pred_keypoints_3d, static_cast<size_t>(nj) * 3},
      {g->pred_keypoints_2d, static_cast<size_t>(nj) * 2},
      {g->pred_cam, 3}, {g->pred_cam_t, 3}, {g->focal_length, 2},
      {g->rotmats, 24 * 9}, {g->betas, static_cast<size_t>(e->smpl->m.nb)},
      {g->cls_logits_softmax, static_cast<size_t>(e->cfg.token_num) * e->cfg.token_class_num},
  };
  THMR_NCCL(api, api->GroupStart());
  int status = THMR_OK;
  for (const Field& f : fields) {
    if (!f.base) continue;
    const size_t count = f.per_image * rows;
    const int r = api->AllGather(f.base + count * c->rank, f.base, count, kNcclFloat32, c->comm, st);
    if (r != 0 && status == THMR_OK) status = fail(THMR_ERR_CUDA, "ncclAllGather failed: %s", api->GetErrorString(r));
  }
  THMR_NCCL(api, api->GroupEnd());
  return status;
}

}  // extern "C"
