"""Pins the CPU oracle against the golden vectors produced by the LIVE reference modules (oracle/make_golden.py)."""
import numpy as np
import torch

from oracle import smpl_oracle
from oracle import tokenhmr_oracle as O
from oracle.make_golden import small_vq_inputs
from tokenhmr_b200 import synth
from tokenhmr_b200.config import release_config, tiny_config

W_SEED, SMPL_SEED, IMG_SEED = 1234, 3, 0


def _check_forward(golden, cfg, batch):
    g = np.load(golden)
    assert list(g["meta"][:4]) == [W_SEED, SMPL_SEED, IMG_SEED, batch]
    sd, smpl = synth.make_state_dict(cfg, W_SEED), synth.make_smpl(cfg, SMPL_SEED)
    img = synth.make_images(batch, cfg, IMG_SEED)
    with torch.no_grad():
        out = O.forward(sd, smpl, img, cfg, return_intermediates=True)
    t = lambda k: torch.from_numpy(g[k])
    tol = dict(rtol=0, atol=2e-6)
    torch.testing.assert_close(out["_vit_tokens"][:, ::8], t("vit_tokens_sub"), rtol=0, atol=2e-5)
    torch.testing.assert_close(out["cls_logits_softmax"][:, ::16], t("cls_probs_sub"), rtol=0, atol=1e-5)
    assert np.array_equal(out["cls_logits_softmax"].argmax(-1).numpy().astype(np.int16), g["cls_argmax"])
    for k in ("pred_cam", "focal_length"):
        torch.testing.assert_close(out[k], t(k), **tol)
    torch.testing.assert_close(out["pred_cam_t"], t("pred_cam_t"), rtol=1e-5, atol=1e-5)
    for k in ("global_orient", "body_pose", "betas"):
        torch.testing.assert_close(out["pred_smpl_params"][k], t(k), rtol=0, atol=5e-6)
    for k in ("pred_keypoints_3d", "pred_vertices", "pred_keypoints_2d"):
        torch.testing.assert_close(out[k], t(k), rtol=1e-5, atol=2e-5)


def test_forward_tiny_matches_reference_golden(golden_dir):
    _check_forward(golden_dir / "forward_tiny_d2.npz", tiny_config(vit_depth=2), 2)


def test_forward_release_matches_reference_golden(golden_dir):
    torch.set_num_threads(max(1, torch.get_num_threads()))
    _check_forward(golden_dir / "forward_release_d32.npz", release_config(), 2)


def test_vq_quantize_64k_matches_reference_golden(golden_dir):
    """65536 queries (the size class that takes the library's screened two-pass schedule): the restatement equals the LIVE
    reference's QuantizeEMAReset.quantize on every row."""
    g = np.load(golden_dir / "vq_quantize_64k.npz")
    cb = torch.randn(2048, 256, generator=torch.Generator().manual_seed(1))
    x = torch.randn(65536, 256, generator=torch.Generator().manual_seed(12))
    assert np.array_equal(O.vq_quantize(x, cb).numpy(), g["idx"].astype(np.int64))
    gap = O.vq_top2_gap(x, cb).numpy()
    assert np.allclose(gap, g["gap"], rtol=0, atol=1e-4)


def test_vq_quantize_matches_reference_golden(golden_dir):
    g = np.load(golden_dir / "vq_quantize.npz")
    cb = torch.randn(2048, 256, generator=torch.Generator().manual_seed(1))
    x = torch.randn(4096, 256, generator=torch.Generator().manual_seed(2))
    assert np.array_equal(O.vq_quantize(x, cb).numpy(), g["idx_rand"])
    gg = torch.Generator().manual_seed(7)
    pick = torch.randint(0, 2048, (4096,), generator=gg)
    xn = cb[pick] + 0.05 * torch.randn(4096, 256, generator=gg)
    idx = O.vq_quantize(xn, cb).numpy()
    assert np.array_equal(idx, g["idx_near"]) and np.array_equal(idx, g["pick"])
    # quantize(codebook[i]) == i, dequantize(quantize(.)) returns codebook rows (invariants from the code)
    assert torch.equal(O.vq_quantize(cb, cb), torch.arange(2048))
    assert torch.equal(O.vq_dequantize(torch.from_numpy(idx), cb), cb[torch.from_numpy(idx)])
    torch.testing.assert_close(torch.from_numpy(g["logits"]) @ cb, torch.from_numpy(g["dequant_logits"]), rtol=1e-5, atol=1e-5)


def test_geometry_matches_reference_golden(golden_dir):
    g = np.load(golden_dir / "geometry.npz")
    torch.testing.assert_close(O.rot6d_to_rotmat(torch.from_numpy(g["x6"])), torch.from_numpy(g["rotmat"]), rtol=0, atol=1e-6)
    proj = O.perspective_projection(torch.from_numpy(g["pts"]), torch.from_numpy(g["tr"]), torch.from_numpy(g["fl"]))
    torch.testing.assert_close(proj, torch.from_numpy(g["proj"]), rtol=1e-5, atol=1e-5)
    eye6 = torch.tensor([[1., 0., 0., 0., 1., 0.]])
    torch.testing.assert_close(O.rot6d_to_rotmat(eye6)[0], torch.eye(3))


def test_upsample_index_matches_torch():
    import torch.nn as nn
    for lin, lout in [(160, 125), (125, 90), (90, 55), (55, 21)]:
        x = torch.arange(lin, dtype=torch.float32).view(1, 1, lin)
        want = nn.Upsample(lout)(x)[0, 0].long()
        assert torch.equal(O.upsample_nearest_index(lout, lin), want)


def test_restatement_equals_live_reference_modules(golden_dir):
    """Other seeds, other batch: the functional restatement reproduces what the reference modules computed
    (oracle/make_golden.py live_parity_goldens) bit for bit."""
    g = np.load(golden_dir / "forward_tiny_d2_seed99.npz")
    cfg = tiny_config(vit_depth=2)
    w_seed, smpl_seed, img_seed, batch = (int(v) for v in g["meta"])
    sd, smpl = synth.make_state_dict(cfg, w_seed), synth.make_smpl(cfg, smpl_seed)
    img = synth.make_images(batch, cfg, img_seed)
    with torch.no_grad():
        out = O.forward(sd, smpl, img, cfg, return_intermediates=True)
    t, stride = (lambda k: torch.from_numpy(g[k])), int(g["stride"])
    torch.testing.assert_close(out["_vit_tokens"].flatten()[::stride], t("vit_tokens_flat"), rtol=0, atol=1e-6)
    torch.testing.assert_close(out["cls_logits_softmax"].flatten()[::stride], t("cls_probs_flat"), rtol=0, atol=1e-6)
    assert np.array_equal(out["cls_logits_softmax"].argmax(-1).numpy().astype(np.int16), g["cls_argmax"])
    for k in ("pred_cam", "pred_keypoints_3d", "pred_vertices", "pred_keypoints_2d"):
        torch.testing.assert_close(out[k], t(k), rtol=0, atol=1e-6)
    # hard quantiser of the reference
    cb, x = small_vq_inputs()
    assert np.array_equal(O.vq_quantize(x, cb).numpy(), g["vq_idx"].astype(np.int64))


def test_fp16_emulation_stays_close_to_fp32():
    cfg = tiny_config(vit_depth=2)
    sd, smpl = synth.make_state_dict(cfg), synth.make_smpl(cfg)
    img = synth.make_images(2, cfg)
    with torch.no_grad():
        a = O.forward(sd, smpl, img, cfg, emulate_fp16=False)
        b = O.forward(sd, smpl, img, cfg, emulate_fp16=True)
    err = ((a["pred_vertices"] - b["pred_vertices"]).abs().max() / a["pred_vertices"].abs().max()).item()
    assert 0 < err < 2e-3


# ------------------------------------------------------------------------------------------------ evaluation (f1/f3)
def _eval_golden(golden_dir):
    g = np.load(golden_dir / "evaluator.npz")
    t = lambda k: torch.from_numpy(g[k])
    out = {"pred_vertices": t("pred_vertices"), "pred_keypoints_3d": t("pred_keypoints_3d")}
    batch = {"vertices": t("gt_vertices"), "keypoints_3d": t("gt_keypoints_3d"), "imgname": ["x"] * 6}
    return g, out, batch


def test_evaluator_restatement_matches_reference_golden(golden_dir):
    from oracle import eval_oracle as E
    g, out, batch = _eval_golden(golden_dir)
    m, r, p = E.evaluate_batch(out, batch, list(g["keypoint_list"]), 39)
    for got, key in ((m, "mpjpe"), (r, "re"), (p, "pve")):
        np.testing.assert_allclose(got.numpy(), g[key], rtol=2e-5, atol=1e-3)
    jreg = torch.from_numpy(g["jreg"])
    m, r, p = E.evaluate_batch(out, batch, list(range(24)), 39, jreg, "EMDB")
    for got, key in ((m, "emdb_mpjpe"), (r, "emdb_re"), (p, "emdb_pve")):
        np.testing.assert_allclose(got.numpy(), g[key], rtol=2e-5, atol=1e-3)
    t = lambda k: torch.from_numpy(g[k])
    np.testing.assert_allclose(E.cam_crop_to_full(t("cam"), t("center"), t("size"), t("img_size")).numpy(),
                               g["full_cam"], rtol=1e-6, atol=1e-6)


def test_evaluator_restatement_equals_live_reference(golden_dir):
    """Metrics and Procrustes alignment against what the reference's Evaluator computed on two seeded batches."""
    from oracle import eval_oracle as E
    g = np.load(golden_dir / "evaluator_seeds.npz")
    kl = list(g["keypoint_list"])
    for seed in (0, 5):
        out, batch = E.synthetic_eval_batch(5, V=300, seed=seed)
        m, r, p = E.evaluate_batch(out, batch, kl, 39)
        np.testing.assert_allclose(m.numpy(), g[f"mpjpe_{seed}"], rtol=1e-6)
        np.testing.assert_allclose(r.numpy(), g[f"re_{seed}"], rtol=1e-5)
        np.testing.assert_allclose(p.numpy(), g[f"pve_{seed}"], rtol=1e-6)
        S1, S2 = out["pred_keypoints_3d"], batch["keypoints_3d"][..., :3]
        torch.testing.assert_close(E.compute_similarity_transform(S1, S2), torch.from_numpy(g[f"similarity_{seed}"]),
                                   rtol=1e-5, atol=1e-5)


def test_procrustes_known_answers():
    """A similarity-transformed copy aligns back exactly; a reflected copy must NOT be matched by a reflection."""
    from oracle import eval_oracle as E
    g = torch.Generator().manual_seed(1)
    S2 = torch.randn(3, 14, 3, generator=g)
    c, s = np.cos(0.7), np.sin(0.7)
    R = torch.tensor([[c, -s, 0.], [s, c, 0.], [0., 0., 1.]], dtype=torch.float32)
    S1 = 1.7 * S2 @ R.T + torch.tensor([0.3, -0.2, 0.9])
    assert E.reconstruction_error(S1, S2).max() < 1e-5
    mirrored = S2 * torch.tensor([1., 1., -1.])
    assert E.reconstruction_error(mirrored, S2).min() > 0.1
