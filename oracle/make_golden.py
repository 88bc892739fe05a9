"""Generate tests/golden/*.npz by running the LIVE reference modules (oracle/ref_import.py) on seeded
synthetic weights and inputs.  Run in the build container (needs /root/reference):

    python -m oracle.make_golden            # tiny (depth-2) + stage goldens, ~10 s
    python -m oracle.make_golden --release  # also the full ViT-H depth-32 forward (B=2), ~1 min, 2.6 GB RAM

The weights are not stored: tests regenerate them from the same seeds (tokenhmr_b200/synth.py).  TEST
INFRASTRUCTURE ONLY.
"""
from __future__ import annotations

import argparse
import hashlib
from pathlib import Path

import numpy as np
import torch

from tokenhmr_b200 import synth
from tokenhmr_b200.config import release_config, tiny_config

from . import ref_import, smpl_oracle

GOLDEN = Path(__file__).resolve().parent.parent / "tests" / "golden"
W_SEED, SMPL_SEED, IMG_SEED = 1234, 3, 0


def forward_golden(ns, cfg, batch: int, name: str, img_seed: int = IMG_SEED, vert_stride: int = 1) -> None:
    """vert_stride > 1 (the bs=64 golden): vertices every `vert_stride`-th, no token / probability sub-samples."""
    sd = synth.make_state_dict(cfg, W_SEED)
    smpl = synth.make_smpl(cfg, SMPL_SEED)
    img = synth.make_images(batch, cfg, img_seed)
    bb = ref_import.build_backbone(ns, sd, cfg)
    head = ref_import.build_head(ns, sd, cfg)
    out = ref_import.reference_forward(ns, bb, head, smpl, img, cfg)
    probs = out["cls_logits_softmax"]
    top2 = probs.topk(2, dim=-1).values
    if vert_stride > 1:
        np.savez_compressed(
            GOLDEN / name,
            meta=np.array([W_SEED, SMPL_SEED, img_seed, batch, cfg.vit_depth, cfg.num_verts, vert_stride]),
            cls_argmax=probs.argmax(-1).numpy().astype(np.int16),
            cls_maxprob=top2[..., 0].numpy(), cls_second_prob=top2[..., 1].numpy(),
            pred_cam=out["pred_cam"].numpy(), pred_cam_t=out["pred_cam_t"].numpy(),
            betas=out["pred_smpl_params"]["betas"].numpy(),
            global_orient=out["pred_smpl_params"]["global_orient"].numpy(),
            pred_keypoints_3d=out["pred_keypoints_3d"].numpy(),
            pred_vertices_sub=out["pred_vertices"][:, ::vert_stride].numpy(),
            pred_keypoints_2d=out["pred_keypoints_2d"].numpy())
        print("wrote", name)
        return
    np.savez_compressed(
        GOLDEN / name,
        meta=np.array([W_SEED, SMPL_SEED, img_seed, batch, cfg.vit_depth, cfg.num_verts]),
        vit_tokens_sub=out["_vit_tokens"][:, ::8].numpy(),          # every 8th token, all channels
        cls_argmax=probs.argmax(-1).numpy().astype(np.int16),
        cls_maxprob=top2[..., 0].numpy(), cls_second_prob=top2[..., 1].numpy(),
        cls_probs_sub=probs[:, ::16].numpy().astype(np.float32),     # every 16th token position, all classes
        pred_cam=out["pred_cam"].numpy(), pred_cam_t=out["pred_cam_t"].numpy(),
        focal_length=out["focal_length"].numpy(),
        global_orient=out["pred_smpl_params"]["global_orient"].numpy(),
        body_pose=out["pred_smpl_params"]["body_pose"].numpy(),
        betas=out["pred_smpl_params"]["betas"].numpy(),
        pred_keypoints_3d=out["pred_keypoints_3d"].numpy(), pred_vertices=out["pred_vertices"].numpy(),
        pred_keypoints_2d=out["pred_keypoints_2d"].numpy())
    print("wrote", name)


def stage_goldens(ns) -> None:
    cfg = release_config()
    g = torch.Generator().manual_seed(7)
    # --- QuantizeEMAReset.quantize / dequantize / dequantize_logits (quantize_cnn.py:80-93)
    qz = ns.quantize_cnn.QuantizeEMAReset(cfg.nb_code, cfg.code_dim)
    codebook = torch.randn(cfg.nb_code, cfg.code_dim, generator=torch.Generator().manual_seed(1))
    qz.codebook = codebook
    x_rand = torch.randn(4096, cfg.code_dim, generator=torch.Generator().manual_seed(2))
    pick = torch.randint(0, cfg.nb_code, (4096,), generator=g)
    x_near = codebook[pick] + 0.05 * torch.randn(4096, cfg.code_dim, generator=g)
    with torch.no_grad():
        idx_rand = qz.quantize(x_rand)
        idx_near = qz.quantize(x_near)
        k_w = codebook.t()
        d = (x_rand ** 2).sum(-1, keepdim=True) - 2 * x_rand @ k_w + (k_w ** 2).sum(0, keepdim=True)
        top2 = d.topk(2, dim=-1, largest=False).values
        logits = torch.softmax(4 * torch.randn(64, cfg.nb_code, generator=g), -1)
        deq = qz.dequantize_logits(logits)
    np.savez_compressed(GOLDEN / "vq_quantize.npz", idx_rand=idx_rand.numpy(), idx_near=idx_near.numpy(),
                        pick=pick.numpy(), gap_rand=(top2[:, 1] - top2[:, 0]).numpy(),
                        logits=logits.numpy(), dequant_logits=deq.numpy())
    # --- rot6d_to_rotmat + perspective_projection (geometry.py:64-124)
    x6 = torch.randn(256, 6, generator=g)
    pts = torch.randn(4, 44, 3, generator=g) + torch.tensor([0., 0., 20.])
    tr = torch.randn(4, 3, generator=g)
    fl = torch.full((4, 2), 5000. / 256)
    with torch.no_grad():
        R = ns.geometry.rot6d_to_rotmat(x6)
        proj = ns.geometry.perspective_projection(pts, translation=tr, focal_length=fl)
    np.savez_compressed(GOLDEN / "geometry.npz", x6=x6.numpy(), rotmat=R.numpy(), pts=pts.numpy(), tr=tr.numpy(),
                        fl=fl.numpy(), proj=proj.numpy())
    # --- SMPL lbs restatement (UNPINNED: produced by oracle/smpl_oracle.py in float64, stored as regression
    #     fixture so later changes to the restatement are visible)
    smpl = synth.make_smpl(cfg, SMPL_SEED)
    aa = 0.3 * torch.randn(8, 24, 3, generator=g)
    betas = torch.randn(8, 10, generator=g)
    R = smpl_oracle.batch_rodrigues(aa.double().view(-1, 3)).view(8, 24, 3, 3)
    v, j = smpl_oracle.smpl_forward(smpl, R[:, :1], R[:, 1:], betas.double(), dtype=torch.float64)
    np.savez_compressed(GOLDEN / "smpl_lbs_f64.npz", aa=aa.numpy(), betas=betas.numpy(),
                        verts=v.numpy().astype(np.float32), joints=j.numpy().astype(np.float32))
    print("wrote stage goldens")


def eval_goldens() -> None:
    """Evaluator / eval_pose / compute_similarity_transform (pose_utils.py:61-275) and cam_crop_to_full
    (renderer.py:13-23) run from the LIVE reference on seeded inputs."""
    from . import eval_oracle
    ev = ref_import.load_eval_modules()
    V, J = 512, 44
    kl = list(range(25, 39))                       # the 14 LSP joints (datasets_eval.yaml KEYPOINT_LIST)
    out, batch = eval_oracle.synthetic_eval_batch(6, V=V, J=J, seed=11)
    clone = lambda d: {k: (v.clone() if torch.is_tensor(v) else list(v)) for k, v in d.items()}
    e1 = ev.pose_utils.Evaluator(dataset_length=16, keypoint_list=kl, pelvis_ind=39,
                                 metrics=['mode_re', 'mode_mpjpe', 'mode_pve'], dataset='3DPW-TEST')
    e1(clone(out), clone(batch))
    g = torch.Generator().manual_seed(12)
    jreg = torch.rand(24, V, generator=g) * (torch.rand(24, V, generator=g) < 0.06)
    jreg = jreg / jreg.sum(-1, keepdim=True)
    e2 = ev.pose_utils.Evaluator(dataset_length=16, keypoint_list=list(range(24)), pelvis_ind=39,
                                 metrics=['mode_re', 'mode_mpjpe', 'mode_pve'], J_regressor_24_SMPL=jreg, dataset='EMDB')
    e2(clone(out), clone(batch))
    cam = torch.cat([0.6 + 0.5 * torch.rand(6, 1, generator=g), 0.2 * torch.randn(6, 2, generator=g)], -1)
    center = torch.rand(6, 2, generator=g) * torch.tensor([1920., 1080.])
    size = 150 + 400 * torch.rand(6, generator=g)
    img_size = torch.tensor([[1920., 1080.]]).repeat(6, 1)
    full = ev.renderer.cam_crop_to_full(cam, center, size, img_size, 5000. / 256 * img_size.max(dim=1)[0])
    full_const = ev.renderer.cam_crop_to_full(cam, center, size, img_size)
    np.savez_compressed(
        GOLDEN / "evaluator.npz", meta=np.array([6, V, J, 11], np.int64), keypoint_list=np.array(kl, np.int32),
        pred_vertices=out["pred_vertices"].numpy(), pred_keypoints_3d=out["pred_keypoints_3d"].numpy(),
        gt_vertices=batch["vertices"].numpy(), gt_keypoints_3d=batch["keypoints_3d"].numpy(),
        mpjpe=e1.mode_mpjpe[:6].astype(np.float32), re=e1.mode_re[:6].astype(np.float32),
        pve=e1.mode_pve[:6].astype(np.float32), jreg=jreg.numpy(), emdb_mpjpe=e2.mode_mpjpe[:6].astype(np.float32),
        emdb_re=e2.mode_re[:6].astype(np.float32), emdb_pve=e2.mode_pve[:6].astype(np.float32),
        cam=cam.numpy(), center=center.numpy(), size=size.numpy(), img_size=img_size.numpy(),
        full_cam_scaled=full.numpy(), full_cam=full_const.numpy())
    print("wrote evaluator golden")


def preproc_scene(seed: int = 21, H: int = 208, W: int = 272):
    """Small synthetic BGR frame (smooth structure + noise) and person boxes that cover every branch of
    ViTDetDataset.__getitem__: interior box, boxes crossing the frame border, a wide box (aspect-ratio expansion
    on the other side) and two boxes wider than 2.2 x 256 px (anti-alias blur, sigma 0.60 and 1.46)."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    base = 127 + 70 * np.sin(xx / 9.0)[..., None] * np.cos(yy / 13.0)[..., None] * np.array([1.0, 0.6, -0.8])
    img = (base + rng.normal(0, 18, (H, W, 3))).clip(0, 255).astype(np.uint8)
    boxes = np.array([[60.3, 20.2, 180.7, 190.9], [-40.0, -30.0, 120.0, 150.0], [150.5, 100.25, 300.0, 230.0],
                      [20.0, 80.0, 250.0, 130.0], [-250.0, -300.0, 520.0, 540.0], [-900.0, -700.0, 1100.0, 1000.0]],
                     np.float32)
    return img, boxes


def preproc_goldens() -> None:
    """ViTDetDataset items (vitdet_dataset.py:44-88) from the LIVE reference class, cv2 4.x + scipy real,
    skimage.filters.gaussian shimmed onto scipy.ndimage (ref_import.load_dataset_modules)."""
    ds_mod = ref_import.load_dataset_modules()
    img, boxes = preproc_scene()
    ds = ds_mod.vitdet_dataset.ViTDetDataset(ref_import.dataset_cfg(), img, boxes)
    items = [ds[i] for i in range(len(boxes))]
    imgs = np.stack([it["img"] for it in items]).astype(np.float32)
    # the 8-bit crops are stored as bytes (the float image is a table lookup of them); blurred crops as float16-safe
    # float32 planes
    m = 255.0 * np.array([0.485, 0.456, 0.406]); s = 255.0 * np.array([0.229, 0.224, 0.225])
    u8 = np.stack([np.rint(imgs[i] * s[:, None, None] + m[:, None, None]).clip(0, 255).astype(np.uint8) for i in range(len(items))])
    is_u8 = np.array([np.array_equal(((u8[i].astype(np.float64) - m[:, None, None]) / s[:, None, None]).astype(np.float32),
                                     imgs[i]) for i in range(len(items))])
    np.savez_compressed(
        GOLDEN / "preproc.npz", meta=np.array([21, img.shape[0], img.shape[1]], np.int64), boxes=boxes,
        box_center=np.stack([it["box_center"] for it in items]).astype(np.float32),
        box_size=np.array([it["box_size"] for it in items], np.float32),
        img_size=np.stack([it["img_size"] for it in items]),
        is_u8=is_u8, rgb_u8=u8[is_u8], img_blur=imgs[~is_u8],
        cv2_version=np.array(__import__("cv2").__version__), numpy_version=np.array(np.__version__))
    print("wrote preproc golden:", int(is_u8.sum()), "8-bit crops,", int((~is_u8).sum()), "blurred crops")


def encoder_goldens(ns) -> None:
    """EncodeTokens.forward (vanilla_pose_vqvae.py:334-342) from the LIVE reference class on seeded 6D poses, with the
    synthetic codebook and with a codebook drawn from the encoder's own latents (so that the indices are spread)."""
    from tokenhmr_b200.config import release_config as rc
    cfg = rc()
    sd = synth.make_tokenizer_encoder_state_dict(cfg, 1234)
    g = torch.Generator().manual_seed(31)
    x = torch.randn(6, cfg.tok_joints, 6, generator=g)
    with torch.no_grad():
        enc = ref_import.build_encode_tokens(ns, sd, cfg)
        idx_a = enc(x)
        lat = enc.quantizer.preprocess(enc.encoder(x))
        # second codebook: latents of other poses + noise
        xb = torch.randn(16, cfg.tok_joints, 6, generator=g)
        lat_b = enc.quantizer.preprocess(enc.encoder(xb))
        cb = lat_b[torch.randperm(lat_b.shape[0], generator=g)[:cfg.nb_code]] + 0.05 * torch.randn(cfg.nb_code, cfg.code_dim, generator=g)
        cb = cb.half().float()                      # stored as fp16 (1 MB): the codebook IS these rounded values
        sd2 = dict(sd)
        sd2["tokenizer.quantizer.codebook"] = cb
        enc2 = ref_import.build_encode_tokens(ns, sd2, cfg)
        idx_b = enc2(x)
    np.savez_compressed(GOLDEN / "tok_encoder.npz", meta=np.array([1234, 31, 6], np.int64), x=x.numpy(),
                        idx_synth=idx_a.numpy().astype(np.int32), idx_latent_cb=idx_b.numpy().astype(np.int32),
                        latent_sub=lat[::7].numpy(), codebook_latent=cb.numpy().astype(np.float16))
    print("wrote tok_encoder golden:", idx_a.unique().numel(), "/", idx_b.unique().numel(), "distinct codes")


def _digest(a: np.ndarray) -> np.ndarray:
    return np.array(hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest())


def live_parity_goldens(ns) -> None:
    """What the *_equals_live_reference tests compare the restatements with, from the LIVE reference on inputs other
    than the goldens above.  Large arrays are kept as a fixed strided sample (a prime stride, so that every token and
    channel is visited); the bit-exact pre-processing crops are kept as a sample plus the SHA-256 of the whole crop."""
    from . import eval_oracle
    # --- forward of the reference modules (tiny config, weights 99, SMPL 5, images 11, batch 3) and the hard quantiser
    cfg = tiny_config(vit_depth=2)
    sd, smpl = synth.make_state_dict(cfg, 99), synth.make_smpl(cfg, 5)
    img = synth.make_images(3, cfg, 11)
    out = ref_import.reference_forward(ns, ref_import.build_backbone(ns, sd, cfg), ref_import.build_head(ns, sd, cfg),
                                       smpl, img, cfg)
    cb, x = small_vq_inputs()
    qz = ns.quantize_cnn.QuantizeEMAReset(64, 32)
    qz.codebook = cb
    with torch.no_grad():
        idx = qz.quantize(x)
    np.savez_compressed(
        GOLDEN / "forward_tiny_d2_seed99.npz", meta=np.array([99, 5, 11, 3], np.int64), stride=127,
        vit_tokens_flat=out["_vit_tokens"].flatten()[::127].numpy(),
        cls_probs_flat=out["cls_logits_softmax"].flatten()[::127].numpy(),
        cls_argmax=out["cls_logits_softmax"].argmax(-1).numpy().astype(np.int16),
        **{k: out[k].numpy() for k in ("pred_cam", "pred_keypoints_3d", "pred_vertices", "pred_keypoints_2d")},
        vq_idx=idx.numpy().astype(np.int16))
    # --- Evaluator metrics and compute_similarity_transform (pose_utils.py) on two seeded batches
    ev = ref_import.load_eval_modules()
    kl = list(range(25, 39))
    arrays = {}
    for seed in (0, 5):
        o, b = eval_oracle.synthetic_eval_batch(5, V=300, seed=seed)
        e = ev.pose_utils.Evaluator(dataset_length=8, keypoint_list=kl, pelvis_ind=39,
                                    metrics=['mode_re', 'mode_mpjpe', 'mode_pve'], dataset='3DPW-TEST')
        e({k: v.clone() for k, v in o.items()}, {k: (v.clone() if torch.is_tensor(v) else v) for k, v in b.items()})
        arrays.update({f"mpjpe_{seed}": e.mode_mpjpe[:5], f"re_{seed}": e.mode_re[:5], f"pve_{seed}": e.mode_pve[:5],
                       f"similarity_{seed}": ev.pose_utils.compute_similarity_transform(
                           o["pred_keypoints_3d"], b["keypoints_3d"][..., :3]).numpy()})
    np.savez_compressed(GOLDEN / "evaluator_seeds.npz", keypoint_list=np.array(kl, np.int32), **arrays)
    # --- ViTDetDataset items: boxes inside, across the border and larger than the frame, with and without BBOX_SHAPE
    ds_mod = ref_import.load_dataset_modules()
    frame, boxes = live_preproc_scene()
    arrays = {}
    for name, shape in (("shape", (192, 256)), ("noshape", None)):
        ds = ds_mod.vitdet_dataset.ViTDetDataset(ref_import.dataset_cfg(bbox_shape=shape), frame, boxes)
        items = [ds[i] for i in range(len(boxes))]
        arrays.update({f"{name}_img_flat": np.stack([it["img"].ravel()[::251] for it in items]),
                       f"{name}_img_sha256": np.stack([_digest(it["img"]) for it in items]),
                       f"{name}_img_dtype": np.array(str(items[0]["img"].dtype)),
                       f"{name}_box_center": np.stack([it["box_center"] for it in items]),
                       f"{name}_box_size": np.array([it["box_size"] for it in items], np.float32)})
    np.savez_compressed(GOLDEN / "preproc_live.npz", boxes=boxes, stride=251, **arrays)
    # --- EncodeTokens (encoder seed 77, poses seed 4)
    rcfg = release_config()
    sd = synth.make_tokenizer_encoder_state_dict(rcfg, 77)
    enc = ref_import.build_encode_tokens(ns, sd, rcfg)
    x = torch.randn(3, rcfg.tok_joints, 6, generator=torch.Generator().manual_seed(4))
    with torch.no_grad():
        idx, lat = enc(x), enc.quantizer.preprocess(enc.encoder(x))
    np.savez_compressed(GOLDEN / "tok_encoder_seed77.npz", meta=np.array([77, 4, 3], np.int64), stride=31,
                        idx=idx.numpy().astype(np.int32), latent_flat=lat.flatten()[::31].numpy())
    print("wrote live parity goldens")


def small_vq_inputs():
    """A 64 x 32 codebook and 500 queries (seed 13)."""
    g = torch.Generator().manual_seed(13)
    return torch.randn(64, 32, generator=g), torch.randn(500, 32, generator=g)


def live_preproc_scene():
    """Random 300 x 420 BGR frame and four boxes (inside, across the border, up to the far corner, larger than the frame:
    the last one takes the anti-alias blur)."""
    rng = np.random.default_rng(9)
    frame = rng.integers(0, 256, (300, 420, 3), dtype=np.uint8)
    boxes = np.float32([[30.5, 20.25, 200.0, 280.0], [-50, -60, 180, 200], [100, 50, 419, 299], [-400, -300, 800, 700]])
    return frame, boxes


def rodrigues_goldens(ns) -> None:
    """Axis-angle -> rotation matrix by the reference's OWN two implementations (geometry.aa_to_rotmat, via a quaternion,
    geometry.py:5-46; rotation_utils.axis_angle_to_matrix, rotation_utils.py:411-443).  smplx's batch_rodrigues is not in
    the tree (parity of the SMPL stage stays unpinned), but its first step must agree with these: a cross-check of
    oracle/smpl_oracle.batch_rodrigues and of thmr_lbs(pose2rot=1) that does come from reference code."""
    import importlib
    rot = importlib.import_module("lib.utils.rotation_utils")
    g = torch.Generator().manual_seed(17)
    aa = torch.cat([1.2 * torch.randn(120, 3, generator=g), 1e-4 * torch.randn(8, 3, generator=g)])
    with torch.no_grad():
        R_quat = ns.geometry.aa_to_rotmat(aa)
        R_p3d = rot.axis_angle_to_matrix(aa)
    np.savez_compressed(GOLDEN / "rodrigues_ref.npz", aa=aa.numpy(), R_aa_to_rotmat=R_quat.numpy(),
                        R_axis_angle_to_matrix=R_p3d.numpy())
    print("wrote rodrigues golden")


def vq_large_golden(ns) -> None:
    """QuantizeEMAReset.quantize (quantize_cnn.py:80-86) from the LIVE reference class on 65536 unstructured queries: large
    enough for the screened two-pass schedule of thmr_vq_argmin (Q >= 8192, several exact-pass row blocks), so that the
    library's default path is compared with the reference itself and not only with its own exact pass.  The whole distance
    matrix (512 MB) is formed at once, exactly as the reference does."""
    cfg = release_config()
    qz = ns.quantize_cnn.QuantizeEMAReset(cfg.nb_code, cfg.code_dim)
    codebook = torch.randn(cfg.nb_code, cfg.code_dim, generator=torch.Generator().manual_seed(1))
    qz.codebook = codebook
    x = torch.randn(65536, cfg.code_dim, generator=torch.Generator().manual_seed(12))
    with torch.no_grad():
        idx = qz.quantize(x)
        k_w = codebook.t()
        d = (x ** 2).sum(-1, keepdim=True) - 2 * x @ k_w + (k_w ** 2).sum(0, keepdim=True)
        top2 = d.topk(2, dim=-1, largest=False).values
    np.savez_compressed(GOLDEN / "vq_quantize_64k.npz", idx=idx.numpy().astype(np.int16),
                        gap=(top2[:, 1] - top2[:, 0]).numpy().astype(np.float32))
    print("wrote vq_quantize_64k.npz")


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--release", action="store_true")
    ap.add_argument("--only", default="", help="'eval': write only tests/golden/evaluator.npz")
    args = ap.parse_args()
    torch.set_num_threads(max(1, torch.get_num_threads()))
    GOLDEN.mkdir(parents=True, exist_ok=True)
    if args.only == "eval":
        eval_goldens()
        return
    if args.only == "preproc":
        preproc_goldens()
        return
    if args.only == "rodrigues":
        rodrigues_goldens(ref_import.load_modules())
        return
    if args.only == "encoder":
        encoder_goldens(ref_import.load_modules())
        return
    if args.only == "vq":
        vq_large_golden(ref_import.load_modules())
        return
    if args.only == "parity":
        live_parity_goldens(ref_import.load_modules())
        return
    if args.only == "forward":
        ns = ref_import.load_modules()
        forward_golden(ns, tiny_config(vit_depth=2), 2, "forward_tiny_d2.npz")
        if args.release:
            forward_golden(ns, release_config(), 2, "forward_release_d32.npz")
            forward_golden(ns, release_config(), 64, "forward_release_d32_bs64.npz", img_seed=5, vert_stride=16)
        return
    ns = ref_import.load_modules()
    stage_goldens(ns)
    vq_large_golden(ns)
    eval_goldens()
    preproc_goldens()
    encoder_goldens(ns)
    rodrigues_goldens(ns)
    live_parity_goldens(ns)
    forward_golden(ns, tiny_config(vit_depth=2), 2, "forward_tiny_d2.npz")
    if args.release:
        forward_golden(ns, release_config(), 2, "forward_release_d32.npz")
        forward_golden(ns, release_config(), 64, "forward_release_d32_bs64.npz", img_seed=5, vert_stride=16)


if __name__ == "__main__":
    main()
