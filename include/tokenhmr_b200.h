/*
 * tokenhmr_b200 — C ABI of the B200-native TokenHMR inference engine (libtokenhmr_b200.so).
 *
 * The reference (saidwivedi/TokenHMR @ 198645f) has no FFI layer: its seam is the Python method
 * TokenHMR.forward(batch) (tokenhmr/lib/models/tokenhmr.py:330-338 -> forward_step :135-188) and the
 * sub-module calls inside it.  Every entry point below names the reference call it replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - functions return THMR_OK (0) or a negative thmr_status; thmr_last_error() holds the message
 *     (thread-local); nothing throws across this boundary;
 *   - the caller owns every buffer it passes (inputs, outputs, workspace, weights); weights must outlive
 *     the engine; the engine owns only the plans (TMA descriptors) and the repacked SMPL model;
 *   - calls on one engine must be serialised by the caller; all work is stream-ordered, there is no host
 *     synchronisation inside thmr_engine_forward, and it is CUDA-graph capturable after one eager call;
 *   - "f16" = IEEE binary16 (__half), row-major, innermost dimension contiguous.
 *
 * Numeric contract (DESIGN.md): every Linear / Conv / attention product rounds its two operands to f16 and
 * accumulates in fp32 on the tcgen05 tensor cores; LayerNorm, softmax, GELU, residual streams, 6D->rotation,
 * SMPL skinning and projection are fp32.
 */
#ifndef TOKENHMR_B200_H_
#define TOKENHMR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum thmr_status {
  THMR_OK = 0,
  THMR_ERR_INVALID = -1, /* bad argument */
  THMR_ERR_CUDA = -2,    /* CUDA runtime / driver error */
  THMR_ERR_TIMEOUT = -3, /* a device-side pipeline wait expired (kernel bug, not a data error) */
  THMR_ERR_NOMEM = -4
} thmr_status;

int thmr_abi_version(void);
const char* thmr_last_error(void);
/* Reads and clears the device-side pipeline-timeout flag (synchronises the device). */
int thmr_check_device_flags(void);

/* ================================================================================================
 * Stand-alone operators (each is also a stage of thmr_engine_forward)
 * ============================================================================================== */

enum { THMR_ACT_NONE = 0, THMR_ACT_GELU = 1, THMR_ACT_RELU = 2 };

/* nn.Linear as one tcgen05 GEMM:  y = x @ W^T (+ bias) (+ resid)      [vit.py:82-86,112,123; any F.linear]
 *   A [M,K] f16 (pitch lda), B = weight [N,K] f16 (pitch ldb), fp32 accumulate in TMEM.
 *   out32 (nullable) <- acc+bias+resid (fp32);  out16 (nullable) <- act(acc+bias+resid) (f16).
 *   resid (nullable, fp32, pitch ldr) may alias out32.  block_n: 0 = auto, else 32/64/128/256. */
int thmr_gemm_f16(const void* A, int lda, const void* B, int ldb, int M, int N, int K, const float* bias,
                  const float* resid, int ldr, int act, float* out32, int ld32, void* out16, int ld16, int block_n,
                  void* stream);

/* nn.Conv1d(Cin, Cout, 3, stride 1, padding = dilation, dilation) on channels-last zero-padded sequences
 * [resnet.py:47, vanilla_pose_vqvae.py:135-152] as an implicit tcgen05 GEMM.
 *   x   f16 [B, L + 2*pad, Cin]  (pad rows must be zero, pad >= dilation),  w f16 [Cout, 3*Cin] with
 *   k = tap*Cin + c (tap-major repack of the reference's [Cout, Cin, 3]),  bias fp32 [Cout].
 *   Outputs use the same padded layout (pad rows written as zero). */
int thmr_conv1d_k3_f16(const void* x, int B, int L, int pad, int Cin, const void* w, int Cout, const float* bias,
                       int dilation, int act, float* out32, void* out16, void* stream);

/* nn.LayerNorm over the last dim [vit.py:136,144,252; pose_transformer.py:29; modules.py:17,50,52].
 *   x fp32 [R,C] -> y16 (f16, nullable) and/or y32 (fp32, nullable); optional fused ReLU (modules.py:15-19). */
int thmr_layernorm(const float* x, const float* gamma, const float* beta, int R, int C, float eps, int relu,
                   void* y16, float* y32, void* stream);

/* ViT attention core  softmax(q k^T * 80^-0.5) v  for all heads [vit.py:113-122].
 *   qkv f16 [B*192, 3*H*80] exactly as produced by Attention.qkv (q heads, then k, then v);
 *   out f16 [B*192, H*80];  dbg_scores (nullable) fp32 [B*H,192,192] receives the raw q.k^T (tests). */
int thmr_vit_attention(const void* qkv, int B, int heads, void* out, float* dbg_scores, void* stream);

/* QuantizeEMAReset.quantize  [tokenization/models/quantize_cnn.py:80-86]:
 *   idx[q] = argmin_k ( sum x_q^2 - 2 x_q . c_k + sum c_k^2 ), first minimum, int64.
 *   x fp32 [Q,D], codebook fp32 [K,D] (D % 64 == 0).  workspace: thmr_vq_workspace_bytes(Q,K,D) bytes. */
size_t thmr_vq_workspace_bytes(int64_t Q, int K, int D);
int thmr_vq_argmin(const float* x, int64_t Q, const float* codebook, int K, int D, int64_t* idx, void* workspace,
                   void* stream);
/* QuantizeEMAReset.dequantize (F.embedding) [quantize_cnn.py:88-90]: out[q] = codebook[idx[q]]. */
int thmr_vq_dequantize(const int64_t* idx, int64_t Q, const float* codebook, int D, float* out, void* stream);
/* QuantizeEMAReset.dequantize_logits [quantize_cnn.py:92-93]: out = logits @ codebook.
 *   logits f16 [Q,K], codebook_t f16 [D,K] (transposed codebook), out fp32 [Q,D]. */
int thmr_vq_dequant_logits(const void* logits16, int64_t Q, int K, const void* codebook_t16, int D, float* out,
                           void* stream);

/* rot6d_to_rotmat [tokenhmr/lib/utils/geometry.py:64-84]: x fp32 [N,6] -> rot fp32 [N,3,3]. */
int thmr_rot6d_to_rotmat(const float* x6, int64_t N, float* rot, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Evaluation metrics and the crop->full camera (SURVEY §8 rows f1 / f3: the consumers of the forward's outputs)
 * ---------------------------------------------------------------------------------------------- */
/* torch.matmul(J_regressor_24_SMPL, vertices) [tokenhmr/lib/utils/pose_utils.py:213,219]:
 *   jreg fp32 [J,V] (dense), verts fp32 [B,V,3] -> joints fp32 [B,J,3]. */
int thmr_regress_joints(const float* jreg, int J, const float* verts, int V, int B, float* joints, void* stream);
/* Evaluator.__call__ + eval_pose + reconstruction_error + compute_similarity_transform
 * [tokenhmr/lib/utils/pose_utils.py:61-143,201-275], one batch, results in millimetres:
 *   pred_kp fp32 [B,J,3]; gt_kp fp32 [B,J,gt_stride] (gt_stride 3, or 4 when the confidence column is still there);
 *   keypoint_list int32 [K] device (K <= 64); pelvis = (kp[pelvis_a] + kp[pelvis_b]) / 2 of each set
 *   (pelvis_a == pelvis_b: 3DPW branch; 1,2: EMDB branch); pred_verts / gt_verts fp32 [B,V,3] (both NULL with pve
 *   NULL to skip the per-vertex error); mpjpe, re (PA-MPJPE), pve fp32 [B]. */
int thmr_eval_pose(const float* pred_kp, const float* gt_kp, int gt_stride, int J, const int32_t* keypoint_list, int K,
                   int pelvis_a, int pelvis_b, const float* pred_verts, const float* gt_verts, int V, int B,
                   float* mpjpe, float* re, float* pve, void* stream);
/* cam_crop_to_full [tokenhmr/lib/utils/renderer.py:13-23]: cam fp32 [B,3] (s,tx,ty), box_center [B,2], box_size [B],
 *   img_size [B,2] (w,h) -> full_cam fp32 [B,3] (tx,ty,tz). */
int thmr_cam_crop_to_full(const float* cam, const float* box_center, const float* box_size, const float* img_size,
                          float focal_length, int B, float* full_cam, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Input pre-processing (SURVEY §8 row f2: the step before the path)
 * ---------------------------------------------------------------------------------------------- */
typedef struct thmr_preproc_cfg {
  int image_size;          /* MODEL.IMAGE_SIZE: 256 */
  int bbox_w, bbox_h;      /* MODEL.BBOX_SHAPE: 192, 256 (0, 0 = None) */
  double mean[3], std[3];  /* MODEL.IMAGE_MEAN / IMAGE_STD, RGB order, 0..1 scale (multiplied by 255 inside) */
} thmr_preproc_cfg;

/* ViTDetDataset.__init__ / __getitem__ for all boxes of one frame
 * [tokenhmr/lib/datasets/vitdet_dataset.py:17-88 -> utils.py:14-33 (expand_to_aspect_ratio), :81-129
 * (gen_trans_from_patch_cv), :317-361 (generate_image_patch_cv2), :364-376 (convert_cvimg_to_tensor)]:
 *   img_bgr     uint8 [H, pitch_bytes] device, BGR interleaved as cv2.imread returns it;
 *   boxes_host  fp32 [n,4] (x0,y0,x1,y1) HOST (the detector's boxes, demo.py:64-70);
 *   out_img     fp32 [n,3,S,S] device = batch['img'] (RGB, (v - 255 mean) / (255 std));
 *   out_patch_u8 (nullable) uint8 [n,S,S,3] device: the BGR crop cv2.warpAffine returns (8-bit path only; bit exact);
 *   box_center_host [n,2], box_size_host [n], sigma_host [n] (each nullable, HOST): the item's 'box_center',
 *   'box_size' and the anti-alias sigma that was applied (0 = none).
 * Boxes wider than 2.2 * S pixels take the blurred path (Gaussian over the box's source region, then the remap on
 * fp32 data); the others are bit exact with cv2's 8-bit remap.  Stream-ordered; one pageable H2D copy of the
 * per-person parameters, so not graph-capturable.  workspace: thmr_preprocess_workspace_bytes(H, W, n) bytes. */
size_t thmr_preprocess_workspace_bytes(int img_h, int img_w, int n);
/* The host half alone (no CUDA call): 'box_center' [n,2], 'box_size' [n], blur sigma [n] and the inverse affine
 * map cv2.warpAffine derives from gen_trans_from_patch_cv's matrix, [n,6] doubles (each output nullable). */
int thmr_preprocess_plan(const float* boxes_host, int n, const thmr_preproc_cfg* cfg, float* box_center_host,
                         float* box_size_host, float* sigma_host, double* inv_affine_host);
int thmr_preprocess_boxes(const uint8_t* img_bgr, int img_h, int img_w, int64_t pitch_bytes, const float* boxes_host,
                          int n, const thmr_preproc_cfg* cfg, float* out_img, uint8_t* out_patch_u8,
                          float* box_center_host, float* box_size_host, float* sigma_host, void* workspace,
                          void* stream);

/* ------------------------------------------------------------------------------------------------
 * SMPL body model (smplx==0.1.28 SMPLLayer / lbs, wrapped by tokenhmr/lib/models/smpl_wrapper.py:10-41)
 * ---------------------------------------------------------------------------------------------- */
typedef struct thmr_smpl thmr_smpl;

typedef struct thmr_smpl_desc {
  int num_verts;                 /* 6890 */
  int num_betas;                 /* <= 10 */
  const float* v_template;       /* [V,3] */
  const float* shapedirs;        /* [V,3,num_betas] */
  const float* posedirs;         /* [207, 3V] */
  const float* J_regressor;      /* [24,V] */
  const float* lbs_weights;      /* [V,24] */
  const int32_t* parents_host;   /* [24], parents[0] = -1 */
  const float* joint_regressor_extra; /* [n_extra, V] (nullable) */
  int n_extra;                   /* 19 */
  const int32_t* extra_vertex_ids_host; /* [21] VertexJointSelector vertex ids */
  const int32_t* joint_map_host; /* [25] smpl_to_openpose (smpl_wrapper.py:19-20) */
} thmr_smpl_desc;

/* Copies / repacks the model into engine-owned device memory (the descriptor's buffers may be freed after). */
int thmr_smpl_create(const thmr_smpl_desc* desc, thmr_smpl** out);
void thmr_smpl_destroy(thmr_smpl* m);
size_t thmr_smpl_workspace_bytes(const thmr_smpl* m, int batch);

/* smplx.lbs.lbs(betas, pose, ..., pose2rot):  pose fp32 [B,24,3] axis-angle (pose2rot=1) or [B,24,3,3]
 * (pose2rot=0); betas fp32 [B,num_betas]  ->  verts fp32 [B,V,3], joints fp32 [B,24,3] (J_transformed). */
int thmr_lbs(const thmr_smpl* m, const float* pose, int pose2rot, const float* betas, int B, float* verts,
             float* joints, void* workspace, void* stream);

/* SMPL wrapper forward [smpl_wrapper.py:27-41 on top of SMPLLayer.forward]: rotation matrices in,
 * verts fp32 [B,V,3] and joints fp32 [B,25+n_extra,3] (OpenPose-mapped + regressed extra joints) out.
 * If pred_cam (fp32 [B,3], nullable) is given the tail of forward_step is fused in (tokenhmr.py:165-187):
 * cam_t [B,3], focal_out [B,2], kp2d [B,25+n_extra,2]. */
int thmr_smpl_forward(const thmr_smpl* m, const float* rotmats /* [B,24,3,3] */, const float* betas, int B,
                      float* verts, float* joints, const float* pred_cam, float focal_length, float image_size,
                      float* cam_t, float* focal_out, float* kp2d, void* workspace, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Tokenizer encoder + hard quantisation (SURVEY §8 row f4): EncodeTokens
 * [tokenization/models/vanilla_pose_vqvae.py:304-346 -> PoseSPEncoderV1 :42-111, quantize_cnn.py:74-86]
 * ---------------------------------------------------------------------------------------------- */
typedef struct thmr_tok_encoder thmr_tok_encoder;
/* f16 [Cout, taps*3*Cin] tap-major, per tap [hi | hi | lo] of w * 2^8 (split precision: the encoder's output is an
 * index and is computed at fp32 grade; packed by tokenhmr_b200/tokenizer.py); fp32 bias */
typedef struct thmr_tok_conv { const void* w; const float* b; } thmr_tok_conv;
typedef struct thmr_tok_encoder_desc {
  int joints, in_dim;              /* 21, 6 */
  int width, depth, dilation_rate; /* ARCH.WIDTH 512, DEPTH 2, DILATION_RATE 3 */
  int size_mul;                    /* ARCH.TOKEN_SIZE_MUL 4: Upsample(40) + (size_mul-1) x Upsample(x2) */
  int code_dim, nb_code;           /* 256, 2048 */
  thmr_tok_conv conv_in;           /* Conv1d(in_dim,W,3): [W, 3*64], the in_dim channels zero-padded to 64 per tap */
  thmr_tok_conv conv_up[8];        /* the size_mul Conv1d(W,W,3) that follow the Upsample layers */
  thmr_tok_conv conv_down;         /* Conv1d(W,W,4,stride 2,pad 1): [W, 4*W] */
  thmr_tok_conv res_conv1[8], res_conv2[8]; /* Resnet1D blocks in stored order (dilation rate^(depth-1) ... 1) */
  thmr_tok_conv conv_out;          /* Conv1d(W,code_dim,3) */
  const float* codebook;           /* fp32 [nb_code, code_dim] */
} thmr_tok_encoder_desc;

/* The descriptor is copied; the weight buffers stay caller-owned and must outlive the encoder. */
int thmr_tok_encoder_create(const thmr_tok_encoder_desc* desc, thmr_tok_encoder** out);
void thmr_tok_encoder_destroy(thmr_tok_encoder* e);
int thmr_tok_encoder_num_tokens(const thmr_tok_encoder* e);            /* T = 160 for the release tokenizer */
size_t thmr_tok_encoder_workspace_bytes(const thmr_tok_encoder* e, int batch);
/* EncodeTokens.forward: pose6d fp32 [B, joints, in_dim] -> code_idx int64 [B*T] (first minimum, as torch.min);
 * latent (nullable) fp32 [B*T, code_dim] receives the encoder output the quantiser saw. */
int thmr_tok_encode(const thmr_tok_encoder* e, const float* pose6d, int B, int64_t* code_idx, float* latent,
                    void* workspace, void* stream);

/* ================================================================================================
 * Engine: TokenHMR.forward(batch)  [tokenhmr.py:330-338 -> 135-188]
 * ============================================================================================== */
typedef struct thmr_engine thmr_engine;

typedef struct thmr_config {
  int image_size, crop_w, patch, patch_pad;           /* 256, 192, 16, 2 */
  int vit_dim, vit_depth, vit_heads, vit_mlp_ratio;   /* 1280, 32, 16, 4  (head_dim must be 80, 192 tokens) */
  float vit_ln_eps;                                   /* 1e-6 */
  int dec_dim, dec_depth, dec_heads, dec_dim_head, dec_mlp_dim; /* 1024, 6, 8, 64, 1024 */
  float ln_eps;                                       /* 1e-5 */
  int token_num, token_class_num, cls_hidden, cls_hidden_inter, cls_token_inter, cls_blocks; /* 160,2048,64,256,64,4 */
  int code_dim, tok_width, tok_depth, tok_dilation_rate, tok_joints; /* 256, 512, 2, 3, 21 */
  int n_upsample;                                     /* 4 */
  int upsample_sizes[8];                              /* 125, 90, 55, 21 */
  float focal_length;                                 /* 5000 */
  int strict;   /* 0: fp16 operands / fp32 accumulate (default).  1: every contraction in split fp16 (3 tensor-core
                 * products, ~2^-21 relative = fp32-grade, the reference's arithmetic: demo.py:35-37 runs fp32); all
                 * "w" matrices of thmr_weights are then f16 [out, 3*in] = [hi | hi | lo] of w * 2^8 (per tap for convs),
                 * as packed by tokenhmr_b200/weights.py with strict=True. */
  int concurrent; /* 0: the forward owns the GPU while it runs (default).  1: its kernels may share the GPU with other work
                   * (another forward of this engine's weights replayed on a second stream, TokenHMRPipeline(streams=2)):
                   * schedules that need every CTA of a grid to be resident at the same time (the stream-K reduce-add GEMM,
                   * whose CTA pairs wait for each other's partial tiles) are replaced by their whole-tile forms. */
} thmr_config;

/* Weight pointers, packed by the host loader (tokenhmr_b200/weights.py) from the reference state_dicts.
 * "w" matrices are f16 [out,in] (nn.Linear layout); vectors are fp32. */
typedef struct thmr_vit_block {
  const float *ln1_g, *ln1_b;
  const void* qkv_w; const float* qkv_b;      /* [3D,D] */
  const void* proj_w; const float* proj_b;    /* [D,D] */
  const float *ln2_g, *ln2_b;
  const void* fc1_w; const float* fc1_b;      /* [4D,D] */
  const void* fc2_w; const float* fc2_b;      /* [D,4D] */
} thmr_vit_block;

typedef struct thmr_dec_layer {
  const float *ln0_g, *ln0_b;
  const void* sa_v_w;                          /* V third of to_qkv: [inner, E] */
  const void* sa_out_w; const float* sa_out_b; /* [E, inner] */
  const float *ln1_g, *ln1_b;
  const void* ca_q_w;                          /* [inner, E] */
  const void* ca_out_w; const float* ca_out_b; /* [E, inner] */
  const float *ln2_g, *ln2_b;
  const void* ff1_w; const float* ff1_b;       /* [mlp, E] */
  const void* ff2_w; const float* ff2_b;       /* [E, mlp] */
} thmr_dec_layer;

typedef struct thmr_mixer_block {
  const float *ln1_g, *ln1_b;
  const void* tok1_w; const float* tok1_b;     /* [token_inter, T] */
  const void* tok2_w; const float* tok2_b;     /* [T, token_inter] */
  const float *ln2_g, *ln2_b;
  const void* ch1_w; const float* ch1_b;       /* [hidden_inter, H] */
  const void* ch2_w; const float* ch2_b;       /* [H, hidden_inter] */
} thmr_mixer_block;

typedef struct thmr_conv { const void* w; const float* b; } thmr_conv; /* w f16 [Cout, 3*Cin] tap-major (or [Cout,Cin]) */

typedef struct thmr_weights {
  /* ViT */
  const void* patch_w; const float* patch_b;   /* [D, 3*P*P] */
  const float* pos;                            /* [192, D] = pos_embed[1:] + pos_embed[0] */
  const thmr_vit_block* blocks_host;           /* host array [vit_depth] */
  const float *last_g, *last_b;
  /* decoder */
  const float* token0;                         /* [E] = to_token_embedding.bias + pos_embedding */
  const void* kv_w;                            /* [dec_depth * 2*inner, D]: to_kv of all layers stacked */
  const thmr_dec_layer* dec_host;              /* host array [dec_depth] */
  const void* readout_w; const float* readout_b; /* [32, E]: grot(6) hands(12) shape(10) cam(3) + 1 zero row */
  const float *init_pose, *init_betas, *init_cam; /* [144], [10], [3] */
  /* token classifier */
  const void* mt_w; const float* mt_b; const float *mt_ln_g, *mt_ln_b; /* Linear E -> T*H, LN(T*H) */
  const thmr_mixer_block* mixer_host;          /* host array [cls_blocks] */
  const void* mn_w; const float* mn_b; const float *mn_ln_g, *mn_ln_b; /* Linear H->H, LN(H) */
  const void* cls_w; const float* cls_b;       /* [classes, H] */
  /* tokenizer */
  const void* codebook_t;                      /* f16 [code_dim, nb_code] */
  thmr_conv conv_in;                           /* code_dim -> W */
  thmr_conv conv_up[8];                        /* after each Upsample */
  thmr_conv res_conv1[8], res_conv2[8];        /* Resnet1D blocks in stored order (dilation rate^(depth-1) ... 1) */
  thmr_conv conv_post, conv_out;               /* W -> W, W -> 6 */
} thmr_weights;

typedef struct thmr_outputs {                  /* all fp32, caller-allocated; any pointer may be NULL */
  float* cls_logits_softmax;  /* [B,160,2048] */
  float* pred_cam;            /* [B,3] */
  float* rotmats;             /* [B,24,3,3]: global_orient = [:, :1], body_pose = [:, 1:] */
  float* betas;               /* [B,10] */
  float* pred_cam_t;          /* [B,3] */
  float* focal_length;        /* [B,2] */
  float* pred_keypoints_3d;   /* [B,44,3] */
  float* pred_vertices;       /* [B,V,3] */
  float* pred_keypoints_2d;   /* [B,44,2] */
  /* optional taps for stage-level parity tests */
  float* vit_tokens;          /* [B,192,D] backbone output (token-major) */
  float* token_out;           /* [B,E] decoder output */
  float* pose6d;              /* [B,144] */
} thmr_outputs;

int thmr_engine_create(const thmr_config* cfg, const thmr_weights* w, const thmr_smpl* smpl, thmr_engine** out);
void thmr_engine_destroy(thmr_engine* e);
size_t thmr_engine_workspace_bytes(const thmr_engine* e, int max_batch);
/* img fp32 [B,3,image_size,image_size] (batch['img']).  `workspace` must hold
 * thmr_engine_workspace_bytes(e, B) bytes, 1024-byte aligned. */
int thmr_engine_forward(thmr_engine* e, const float* img, int B, const thmr_outputs* out, void* workspace,
                        void* stream);
/* Number of kernels one forward at the batch size of the last forward launches, copies not counted
 * (for bench.py's gpu_launches). */
int thmr_engine_num_launches(const thmr_engine* e);
/* Timed replay for roofline accounting: the forward is a list of launch groups ("steps"); this runs one
 * forward with a CUDA event between steps (synchronises the stream at the end) and returns per-step
 * milliseconds.  thmr_engine_step_info gives each step's label and algorithmic FLOPs / HBM bytes. */
int thmr_engine_num_steps(const thmr_engine* e);
int thmr_engine_step_info(const thmr_engine* e, int i, const char** name, double* flops, double* bytes);
int thmr_engine_profile(thmr_engine* e, const float* img, int B, const thmr_outputs* out, void* workspace,
                        void* stream, float* step_ms, int cap);
/* In-graph timing.  Every kernel of the default-mode forward writes the GPU's global nanosecond timer into its step's
 * slot when it starts; thmr_engine_forward_stamped = thmr_engine_forward + one trailing 1-warp kernel that stamps the
 * end.  Capture it in a CUDA graph, replay, then thmr_engine_read_stamps (synchronous D2H): host_ns[i] = start of step i
 * (0 = that step launched no stamped kernel: its time belongs to the previous step), host_ns[n_steps] = end.  Kernels of a
 * stream run back to back, so the differences are each step's share of the real replay, with no events in between.
 * Returns the number of entries (n_steps + 1) or a negative status. */
int thmr_engine_forward_stamped(thmr_engine* e, const float* img, int B, const thmr_outputs* out, void* workspace,
                                void* stream);
int thmr_engine_read_stamps(const thmr_engine* e, unsigned long long* host_ns, int cap);
/* Backbone only: ViT.forward [vit.py:341-343]: img -> tokens fp32 [B,192,D] (token-major). */
int thmr_engine_vit_forward(thmr_engine* e, const float* img, int B, float* tokens, void* workspace, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Multi-GPU exchange (SURVEY.md section 8b/8e).  The path shards by image with no data-path collective;
 * the one exchange is an all-gather of the per-image outputs (BASELINE.json configs[2]: "NCCL all-gather of
 * SMPL params/vertices").  In-place design: each output field is ONE device buffer of nranks * rows_per_rank
 * images on every rank; rank r runs thmr_engine_forward with its thmr_outputs pointing at rows
 * [r * rows_per_rank, (r+1) * rows_per_rank) of those buffers, then thmr_allgather_outputs() fills in the other
 * ranks' rows with one grouped ncclAllGather (sendbuff = recvbuff + rank * count), stream-ordered and
 * CUDA-graph capturable together with the forward.  Replaces the reference's single-process
 * `model(batch)` over the whole batch (tokenhmr/eval.py:146-147) when the batch is split over GPUs.
 * NCCL is loaded at run time (libnccl.so.2; override with THMR_NCCL_LIB). */
typedef struct thmr_comm thmr_comm;
/* 128-byte NCCL unique id, created on one rank and distributed to the others by the caller (any transport). */
int thmr_comm_unique_id(void* id128);
/* Collective over all ranks; uses the calling thread's current CUDA device. */
int thmr_comm_create(const void* id128, int nranks, int rank, thmr_comm** out);
void thmr_comm_destroy(thmr_comm* c);
int thmr_comm_nranks(const thmr_comm* c);
int thmr_comm_rank(const thmr_comm* c);
/* `global`: base pointers of the nranks * rows_per_rank buffers (NULL fields are skipped; the taps are never
 * gathered; cls_logits_softmax is gathered only when its pointer is non-NULL: 1.3 MB per image). */
int thmr_allgather_outputs(const thmr_engine* e, thmr_comm* c, const thmr_outputs* global, int rows_per_rank,
                           void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TOKENHMR_B200_H_ */
