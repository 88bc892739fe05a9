"""CPU oracle for TokenHMR's per-image forward path.  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this
module; the product (tokenhmr_b200/) never does.

This is a plain-PyTorch (CPU, fp32) functional restatement of what the reference computes between
batch['img'] and the output dict, each function citing the reference file:line it follows
(reference = saidwivedi/TokenHMR @ 198645f).  It takes the flat state dict produced by
tokenhmr_b200.synth.make_state_dict (same names as the reference checkpoints).

Pinning status
  * ViT, decoder, token classifier, tokenizer decoder, quantizer, rot6d, projection: PINNED against the
    reference's own modules executed in the build container (oracle/ref_import.py imports them file by
    file; oracle/make_golden.py stores their outputs under tests/golden/; tests/test_oracle_pinned.py
    checks this restatement against those goldens).
  * SMPL (smplx==0.1.28 lbs / SMPLLayer / VertexJointSelector): third-party, absent from /root/reference
    and not installable offline -> restated from the published algorithm (oracle/smpl_oracle.py),
    anchored on the reference call sites only: PARITY UNPINNED for that stage.

`emulate_fp16=True` reproduces the engine's numeric contract on the CPU: every Linear / conv /
attention matmul rounds its two operands to fp16 and accumulates in fp32; LayerNorm, softmax, GELU,
residuals and all SMPL math stay fp32.  With emulate_fp16=False this is the reference's fp32 path.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch
import torch.nn.functional as F

from . import smpl_oracle

Tensor = torch.Tensor


class Numerics:
    """Operand rounding policy (fp32 reference, or the engine's fp16-operand / fp32-accumulate contract)."""

    def __init__(self, emulate_fp16: bool = False):
        self.emulate_fp16 = emulate_fp16

    def q(self, x: Tensor) -> Tensor:
        return x.half().float() if self.emulate_fp16 else x

    def linear(self, x: Tensor, w: Tensor, b: Optional[Tensor] = None) -> Tensor:
        return F.linear(self.q(x), self.q(w), b)

    def matmul(self, a: Tensor, b: Tensor) -> Tensor:
        return torch.matmul(self.q(a), self.q(b))

    def conv1d(self, x: Tensor, w: Tensor, b: Tensor, padding: int, dilation: int = 1, stride: int = 1) -> Tensor:
        return F.conv1d(self.q(x), self.q(w), b, stride=stride, padding=padding, dilation=dilation)

    def conv2d(self, x: Tensor, w: Tensor, b: Tensor, stride: int, padding: int) -> Tensor:
        return F.conv2d(self.q(x), self.q(w), b, stride=stride, padding=padding)


# ------------------------------------------------------------------------------------------------
# ViT-H/16 backbone
# ------------------------------------------------------------------------------------------------
def vit_forward(sd: Dict[str, Tensor], img: Tensor, cfg, nm: Numerics, prefix: str = "backbone.") -> Tensor:
    """ViT.forward + forward_features (vit.py:320-343).  img (B,3,256,256) -> tokens (B,192,1280).

    Returns token-major features: the reference's final permute/reshape to (B,1280,16,12) (vit.py:337) is
    undone by the head's rearrange 'b c h w -> b (h w) c' (token_head.py:69), so both are skipped."""
    g = lambda n: sd[prefix + n]
    x = img[:, :, :, cfg.crop_x0:cfg.image_size - cfg.crop_x0]                       # vit.py:342
    x = nm.conv2d(x, g("patch_embed.proj.weight"), g("patch_embed.proj.bias"),
                  stride=cfg.patch, padding=cfg.patch_pad)                          # vit.py:168,172
    x = x.flatten(2).transpose(1, 2)                                                # vit.py:175
    pos = g("pos_embed")
    x = x + pos[:, 1:] + pos[:, :1]                                                 # vit.py:327
    B, N, C = x.shape
    H, hd = cfg.vit_heads, cfg.head_dim
    scale = hd ** -0.5                                                              # vit.py:102
    for i in range(cfg.vit_depth):                                                  # vit.py:329-333
        p = f"blocks.{i}."
        y = F.layer_norm(x, (C,), g(p + "norm1.weight"), g(p + "norm1.bias"), cfg.vit_ln_eps)
        qkv = nm.linear(y, g(p + "attn.qkv.weight"), g(p + "attn.qkv.bias"))        # vit.py:112
        qkv = qkv.reshape(B, N, 3, H, hd).permute(2, 0, 3, 1, 4)                    # vit.py:113
        q, k, v = qkv[0], qkv[1], qkv[2]
        if nm.emulate_fp16:
            # engine contract: q,k,v stored as fp16; scores scaled after the fp32-accumulated dot;
            # unnormalised exp rounded to fp16 for the PV product; row sum kept in fp32.
            q, k, v = nm.q(q), nm.q(k), nm.q(v)
            s = torch.matmul(q, k.transpose(-2, -1)) * scale
            s = s - s.amax(dim=-1, keepdim=True)
            pexp = torch.exp(s)
            o = torch.matmul(nm.q(pexp), v) / pexp.sum(dim=-1, keepdim=True)
        else:
            q = q * scale                                                           # vit.py:116
            attn = (q @ k.transpose(-2, -1)).softmax(dim=-1)                        # vit.py:117-119
            o = attn @ v                                                            # vit.py:122
        o = o.transpose(1, 2).reshape(B, N, C)
        x = x + nm.linear(o, g(p + "attn.proj.weight"), g(p + "attn.proj.bias"))    # vit.py:123,149
        y = F.layer_norm(x, (C,), g(p + "norm2.weight"), g(p + "norm2.bias"), cfg.vit_ln_eps)
        h = F.gelu(nm.linear(y, g(p + "mlp.fc1.weight"), g(p + "mlp.fc1.bias")))    # vit.py:83-84 (erf GELU)
        x = x + nm.linear(h, g(p + "mlp.fc2.weight"), g(p + "mlp.fc2.bias"))        # vit.py:85,150
    x = F.layer_norm(x, (C,), g("last_norm.weight"), g("last_norm.bias"), cfg.vit_ln_eps)   # vit.py:335
    return x


# ------------------------------------------------------------------------------------------------
# One-token transformer decoder
# ------------------------------------------------------------------------------------------------
def decoder_forward(sd: Dict[str, Tensor], context: Tensor, cfg, nm: Numerics,
                    prefix: str = "smpl_head.transformer.") -> Tensor:
    """TransformerDecoder.forward with a zero (B,1,1) token (token_head.py:91-96,
    pose_transformer.py:349-357, 191-201).  context (B,192,1280) -> token_out (B,1024)."""
    g = lambda n: sd[prefix + n]
    B = context.shape[0]
    E, Hh, dh = cfg.dec_dim, cfg.dec_heads, cfg.dec_dim_head
    inner = Hh * dh
    scale = dh ** -0.5
    # to_token_embedding(zeros) = bias; += pos_embedding (pose_transformer.py:350,354)
    x = (g("to_token_embedding.bias") + g("pos_embedding")[0, 0]).unsqueeze(0).expand(B, E).clone()
    for l in range(cfg.dec_depth):
        p = f"transformer.layers.{l}."
        # -- self-attention over a single token (pose_transformer.py:75-86): softmax over one key == 1,
        #    so the block reduces to to_out(v); the q,k thirds of to_qkv do not influence the output.
        y = F.layer_norm(x, (E,), g(p + "0.norm.weight"), g(p + "0.norm.bias"), cfg.ln_eps)
        v = nm.linear(y, g(p + "0.fn.to_qkv.weight")[2 * inner:3 * inner])
        x = nm.linear(v, g(p + "0.fn.to_out.0.weight"), g(p + "0.fn.to_out.0.bias")) + x
        # -- cross-attention (pose_transformer.py:111-124); to_kv / to_q have no bias, context is not normed
        y = F.layer_norm(x, (E,), g(p + "1.norm.weight"), g(p + "1.norm.bias"), cfg.ln_eps)
        kv = nm.linear(context, g(p + "1.fn.to_kv.weight"))                        # (B,192,2*inner)
        k, vv = kv.chunk(2, dim=-1)
        q = nm.linear(y, g(p + "1.fn.to_q.weight"))                                # (B,inner)
        if nm.emulate_fp16:
            k, vv = nm.q(k), nm.q(vv)                                              # engine stores K/V as fp16
        qh = q.view(B, Hh, 1, dh)
        kh = k.view(B, -1, Hh, dh).permute(0, 2, 1, 3)
        vh = vv.view(B, -1, Hh, dh).permute(0, 2, 1, 3)
        dots = torch.matmul(qh, kh.transpose(-1, -2)) * scale                       # pose_transformer.py:117
        attn = dots.softmax(dim=-1)
        out = torch.matmul(attn, vh).permute(0, 2, 1, 3).reshape(B, inner)
        x = nm.linear(out, g(p + "1.fn.to_out.0.weight"), g(p + "1.fn.to_out.0.bias")) + x
        # -- feed-forward (pose_transformer.py:43-52)
        y = F.layer_norm(x, (E,), g(p + "2.norm.weight"), g(p + "2.norm.bias"), cfg.ln_eps)
        h = F.gelu(nm.linear(y, g(p + "2.fn.net.0.weight"), g(p + "2.fn.net.0.bias")))
        x = nm.linear(h, g(p + "2.fn.net.3.weight"), g(p + "2.fn.net.3.bias")) + x
    return x


# ------------------------------------------------------------------------------------------------
# Token classifier (MLP-Mixer) + tokenizer decode
# ------------------------------------------------------------------------------------------------
def classifier_logits_softmax(sd: Dict[str, Tensor], tok: Tensor, cfg, nm: Numerics,
                              prefix: str = "smpl_head.decpose.") -> Tensor:
    """TokenClassfier.forward up to the softmax (token_classifier.py:89-104; modules.py:11-63).
    tok (B,1024) -> cls_logits_softmax (B,160,2048)."""
    g = lambda n: sd[prefix + n]
    B = tok.shape[0]
    T, H = cfg.token_num, cfg.cls_hidden
    f = nm.linear(tok, g("mixer_trans.ff.0.weight"), g("mixer_trans.ff.0.bias"))
    f = F.relu(F.layer_norm(f, (T * H,), g("mixer_trans.ff.1.weight"), g("mixer_trans.ff.1.bias"), cfg.ln_eps))
    x = f.reshape(B, T, H)                                                          # token_classifier.py:94
    for i in range(cfg.cls_blocks):                                                 # modules.py:55-63
        p = f"mixer_head.{i}."
        y = F.layer_norm(x, (H,), g(p + "layernorm1.weight"), g(p + "layernorm1.bias"), cfg.ln_eps)
        y = y.transpose(2, 1)
        y = F.gelu(nm.linear(y, g(p + "MLP_token.ff.0.weight"), g(p + "MLP_token.ff.0.bias")))
        y = nm.linear(y, g(p + "MLP_token.ff.3.weight"), g(p + "MLP_token.ff.3.bias"))
        y = y.transpose(2, 1)
        z = F.layer_norm(x + y, (H,), g(p + "layernorm2.weight"), g(p + "layernorm2.bias"), cfg.ln_eps)
        z = F.gelu(nm.linear(z, g(p + "MLP_channel.ff.0.weight"), g(p + "MLP_channel.ff.0.bias")))
        z = nm.linear(z, g(p + "MLP_channel.ff.3.weight"), g(p + "MLP_channel.ff.3.bias"))
        x = x + y + z
    x = nm.linear(x, g("mixer_norm_layer.ff.0.weight"), g("mixer_norm_layer.ff.0.bias"))
    x = F.relu(F.layer_norm(x, (H,), g("mixer_norm_layer.ff.1.weight"), g("mixer_norm_layer.ff.1.bias"), cfg.ln_eps))
    logits = nm.linear(x, g("class_pred_layer.weight"), g("class_pred_layer.bias"))  # token_classifier.py:101
    return logits.softmax(-1)                                                       # token_classifier.py:104


def upsample_nearest_index(out_len: int, in_len: int) -> torch.Tensor:
    """nn.Upsample(size=out_len), mode='nearest' (legacy): src = floor(dst * in/out), computed in fp32
    exactly like ATen's nearest_neighbor_compute_source_index (scale = in/out as float)."""
    scale = torch.tensor(in_len / out_len, dtype=torch.float32)
    idx = torch.floor(torch.arange(out_len, dtype=torch.float32) * scale).to(torch.int64)
    return idx.clamp_(max=in_len - 1)


def tokenizer_decode(sd: Dict[str, Tensor], probs: Tensor, cfg, nm: Numerics,
                     prefix: str = "tokenizer.") -> Tensor:
    """DecodeTokens.forward (vanilla_pose_vqvae.py:294-297): soft codebook lookup
    (quantize_cnn.py:92-93) + PoseSPDecoderV1.decoder (vanilla_pose_vqvae.py:135-154, resnet.py:51-82).
    probs (B,160,2048) -> 6D body pose (B,21,6)."""
    g = lambda n: sd[prefix + n]
    t = "decoder.decoder."
    feat = nm.matmul(probs, g("quantizer.codebook"))                                # (B,160,256)
    x = feat.permute(0, 2, 1)                                                       # (B,256,160)
    x = F.relu(nm.conv1d(x, g(t + "0.weight"), g(t + "0.bias"), padding=1))
    idx = 2
    for size in cfg.upsample_sizes:                                                 # Upsample, Conv1d, ReLU
        x = x[:, :, upsample_nearest_index(size, x.shape[-1])]
        x = F.relu(nm.conv1d(x, g(f"{t}{idx + 1}.weight"), g(f"{t}{idx + 1}.bias"), padding=1))
        idx += 3
    # Resnet1D(reverse_dilation=True): blocks stored in order [dil = rate**(depth-1), ..., 1] (resnet.py:72-77)
    dils = [cfg.tok_dilation_rate ** d for d in range(cfg.tok_depth)][::-1]
    for d, dil in enumerate(dils):
        r = f"{t}{idx}.0.model.{d}."
        h = nm.conv1d(F.relu(x), g(r + "conv1.weight"), g(r + "conv1.bias"), padding=dil, dilation=dil)
        h = nm.conv1d(F.relu(h), g(r + "conv2.weight"), g(r + "conv2.bias"), padding=0)
        x = x + h                                                                   # resnet.py:51-68
    x = nm.conv1d(x, g(f"{t}{idx}.1.weight"), g(f"{t}{idx}.1.bias"), padding=1)
    x = nm.conv1d(x, g(f"{t}{idx + 1}.weight"), g(f"{t}{idx + 1}.bias"), padding=1)  # (B,6,21)
    return x.permute(0, 2, 1)                                                       # postprocess :156-159


def tokenizer_encode(sd: Dict[str, Tensor], pose6d: Tensor, cfg, nm: Numerics, prefix: str = "tokenizer."):
    """EncodeTokens.forward (vanilla_pose_vqvae.py:334-342): PoseSPEncoderV1 (:42-111: preprocess :88-92, the
    Sequential built at :65-86 with Resnet1D reverse_dilation=True, resnet.py:70-82) + QuantizeEMAReset.preprocess /
    quantize (quantize_cnn.py:74-86).  pose6d (B,21,6) -> (code_idx (B*T,) int64, latent (B*T, code_dim))."""
    g = lambda n: sd[prefix + n]
    e = "encoder.encoder."
    B = pose6d.shape[0]
    x = pose6d.reshape(B, pose6d.shape[1], -1).permute(0, 2, 1)                     # (B,6,21)
    x = F.relu(nm.conv1d(x, g(e + "0.weight"), g(e + "0.bias"), padding=1))
    x = x[:, :, upsample_nearest_index(((cfg.tok_joints * 2) // 10) * 10, x.shape[-1])]   # nn.Upsample(40), :69
    x = F.relu(nm.conv1d(x, g(e + "3.weight"), g(e + "3.bias"), padding=1))
    idx = 5
    for _ in range(cfg.tok_size_mul - 1):                                           # Upsample(x2), Conv1d, ReLU :73-76
        x = x[:, :, upsample_nearest_index(2 * x.shape[-1], x.shape[-1])]
        x = F.relu(nm.conv1d(x, g(f"{e}{idx + 1}.weight"), g(f"{e}{idx + 1}.bias"), padding=1))
        idx += 3
    x = nm.conv1d(x, g(f"{e}{idx}.0.weight"), g(f"{e}{idx}.0.bias"), padding=1, stride=2)   # Conv1d(W,W,4,2,1) :80-83
    dils = [cfg.tok_dilation_rate ** d for d in range(cfg.tok_depth)][::-1]
    for d, dil in enumerate(dils):
        r = f"{e}{idx}.1.model.{d}."
        h = nm.conv1d(F.relu(x), g(r + "conv1.weight"), g(r + "conv1.bias"), padding=dil, dilation=dil)
        h = nm.conv1d(F.relu(h), g(r + "conv2.weight"), g(r + "conv2.bias"), padding=0)
        x = x + h
    x = nm.conv1d(x, g(f"{e}{idx + 1}.weight"), g(f"{e}{idx + 1}.bias"), padding=1)          # (B,code_dim,T) :86
    lat = x.permute(0, 2, 1).contiguous().view(-1, x.shape[1])                      # preprocess, quantize_cnn.py:74-78
    return vq_quantize(lat, g("quantizer.codebook")), lat


def vq_quantize(x: Tensor, codebook: Tensor, chunk: int = 65536) -> Tensor:
    """QuantizeEMAReset.quantize (quantize_cnn.py:80-86): first-minimum index of
    sum(x^2) - 2 x @ codebook^T + sum(codebook^2); row-chunked (identical per-row arithmetic) so that 1 M
    queries do not materialise an 8 GB distance matrix."""
    k_w = codebook.t()
    c2 = torch.sum(k_w ** 2, dim=0, keepdim=True)
    out = []
    for i in range(0, x.shape[0], chunk):
        xc = x[i:i + chunk]
        distance = torch.sum(xc ** 2, dim=-1, keepdim=True) - 2 * torch.matmul(xc, k_w) + c2
        out.append(torch.min(distance, dim=-1)[1])
    return torch.cat(out)


def vq_top2_gap(x: Tensor, codebook: Tensor) -> Tensor:
    """Distance gap between the best and second-best code per query (near-tie detector for index parity)."""
    k_w = codebook.t()
    d = torch.sum(x ** 2, dim=-1, keepdim=True) - 2 * torch.matmul(x, k_w) + torch.sum(k_w ** 2, dim=0, keepdim=True)
    t = d.topk(2, dim=-1, largest=False).values
    return t[:, 1] - t[:, 0]


def vq_dequantize(idx: Tensor, codebook: Tensor) -> Tensor:
    """QuantizeEMAReset.dequantize (quantize_cnn.py:88-90)."""
    return F.embedding(idx, codebook)


def rot6d_to_rotmat(x: Tensor) -> Tensor:
    """geometry.py:64-84: Gram-Schmidt, rows of the result are b1, b2, b3.  (N*6,) -> (N,3,3)."""
    x = x.reshape(-1, 2, 3).permute(0, 2, 1).contiguous()
    a1, a2 = x[:, :, 0], x[:, :, 1]
    b1 = F.normalize(a1)
    b2 = F.normalize(a2 - torch.einsum("bi,bi->b", b1, a2).unsqueeze(-1) * b1)
    b3 = torch.cross(b1, b2, dim=-1)
    return torch.stack((b1, b2, b3), dim=-2)


def head_forward(sd: Dict[str, Tensor], context: Tensor, cfg, nm: Numerics, prefix: str = "smpl_head."):
    """SMPLTokenDecoderHead.forward with IEF_ITERS=1, TRANSFORMER_INPUT='zero' (token_head.py:65-128)."""
    g = lambda n: sd[prefix + n]
    B = context.shape[0]
    tok = decoder_forward(sd, context, cfg, nm, prefix + "transformer.")
    pred_grot = nm.linear(tok, g("decpose_grot.weight"), g("decpose_grot.bias"))            # :99
    probs = classifier_logits_softmax(sd, tok, cfg, nm, prefix + "decpose.")
    bpose = tokenizer_decode(sd, probs, cfg, nm).reshape(B, -1)                              # :100, cls :107
    pred_hands = nm.linear(tok, g("decpose_hands.weight"), g("decpose_hands.bias"))         # :101
    pred_body_pose = torch.cat([pred_grot, bpose, pred_hands], -1) + g("init_body_pose")    # :103
    pred_betas = nm.linear(tok, g("decshape.weight"), g("decshape.bias")) + g("init_betas")  # :104
    pred_cam = nm.linear(tok, g("deccam.weight"), g("deccam.bias")) + g("init_cam")          # :105
    rotmats = rot6d_to_rotmat(pred_body_pose).view(B, cfg.num_joints, 3, 3)                  # :123
    return {"global_orient": rotmats[:, [0]], "body_pose": rotmats[:, 1:], "betas": pred_betas}, pred_cam, \
        {"cls_logits_softmax": probs, "token_out": tok, "pred_body_pose_6d": pred_body_pose}


def perspective_projection(points: Tensor, translation: Tensor, focal_length: Tensor) -> Tensor:
    """geometry.py:86-124 with rotation = I and camera_center = 0."""
    p = points + translation.unsqueeze(1)
    p = p / p[:, :, -1].unsqueeze(-1)
    return p[:, :, :-1] * focal_length.unsqueeze(1)


def forward(sd: Dict[str, Tensor], smpl: Dict[str, Tensor], img: Tensor, cfg,
            emulate_fp16: bool = False, return_intermediates: bool = False) -> Dict[str, Tensor]:
    """TokenHMR.forward(batch) == forward_step(batch, train=False) (tokenhmr.py:135-188, 330-338)."""
    nm = Numerics(emulate_fp16)
    B = img.shape[0]
    feats = vit_forward(sd, img, cfg, nm)                                                    # tokenhmr.py:151
    params, pred_cam, aux = head_forward(sd, feats, cfg, nm)                                 # :153
    out: Dict[str, Tensor] = {}
    out["cls_logits_softmax"] = aux["cls_logits_softmax"]                                    # :157-158
    out["pred_cam"] = pred_cam                                                               # :159
    out["pred_smpl_params"] = {k: v.clone() for k, v in params.items()}                      # :160
    focal = cfg.focal_length * torch.ones(B, 2, dtype=img.dtype)                             # :165
    cam_t = torch.stack([pred_cam[:, 1], pred_cam[:, 2],
                         2 * focal[:, 0] / (cfg.image_size * pred_cam[:, 0] + 1e-9)], dim=-1)  # :166-168
    out["pred_cam_t"] = cam_t
    out["focal_length"] = focal
    verts, joints = smpl_oracle.smpl_forward(smpl, params["global_orient"], params["body_pose"],
                                             params["betas"])                               # :173-176
    out["pred_keypoints_3d"] = joints.reshape(B, -1, 3)
    out["pred_vertices"] = verts.reshape(B, -1, 3)
    out["pred_keypoints_2d"] = perspective_projection(joints, cam_t, focal / cfg.image_size)  # :183-187
    if return_intermediates:
        out["_vit_tokens"] = feats
        out["_token_out"] = aux["token_out"]
        out["_pred_body_pose_6d"] = aux["pred_body_pose_6d"]
    return out
