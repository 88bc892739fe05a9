"""Input pre-processing (SURVEY §8 row f2).  CPU part: pins oracle/preproc_oracle.py against the golden items the
LIVE reference ViTDetDataset produced (two scenes) and against cv2 / scipy themselves; checks the C-ABI
host planner (no CUDA call) bit for bit.  GPU part: thmr_preprocess_boxes vs the oracle and the goldens."""
import hashlib

import numpy as np
import pytest
import torch

from oracle import preproc_oracle as P
from oracle.make_golden import live_preproc_scene, preproc_scene

MEAN = 255.0 * np.array(P.DEFAULT_MEAN)
STD = 255.0 * np.array(P.DEFAULT_STD)


def _golden(golden_dir):
    g = np.load(golden_dir / "preproc.npz")
    img, boxes = preproc_scene(int(g["meta"][0]), int(g["meta"][1]), int(g["meta"][2]))
    assert np.array_equal(boxes, g["boxes"])
    ref = np.empty((len(boxes), 3, 256, 256), np.float32)
    ref[g["is_u8"]] = ((g["rgb_u8"].astype(np.float64) - MEAN[:, None, None]) / STD[:, None, None]).astype(np.float32)
    ref[~g["is_u8"]] = g["img_blur"]
    return g, img, boxes, ref


# ------------------------------------------------------------------------------------------------ oracle pinning
def test_oracle_matches_reference_golden_bit_for_bit(golden_dir):
    g, img, boxes, ref = _golden(golden_dir)
    for i, box in enumerate(boxes):
        it = P.vitdet_item(img, box)
        assert (it["sigma"] is None) == bool(g["is_u8"][i])
        assert np.array_equal(it["box_center"], g["box_center"][i]) and it["box_size"] == g["box_size"][i]
        assert np.array_equal(it["img_size"], g["img_size"][i])
        assert np.array_equal(it["img"], ref[i]), f"box {i}: max abs {np.abs(it['img'] - ref[i]).max()}"


def test_oracle_pieces_match_cv2_and_scipy():
    cv2 = pytest.importorskip("cv2")
    ndi = pytest.importorskip("scipy.ndimage")
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (150, 210, 3), dtype=np.uint8)
    for cx, cy, size in [(100.3, 70.7, 120.0), (10.0, 8.0, 250.5), (205.2, 140.9, 500.0), (105, 75, 37.3)]:
        c = np.float32([cx, cy])
        M = P.gen_trans(c[0], c[1], np.float32(size), 256)
        half = np.float32(np.float32(size) * np.float32(0.5))
        src = np.float32([[c[0], c[1]], [c[0], c[1] + half], [c[0] + half, c[1]]])
        dst = np.float32([[128, 128], [128, 256], [256, 128]])
        assert np.array_equal(M, cv2.getAffineTransform(src, dst))
        want = cv2.warpAffine(img, M, (256, 256), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
        assert np.array_equal(P.warp_affine_u8(img, M, 256, 256), want)
        f64 = img.astype(np.float64) * 0.731
        want = cv2.warpAffine(f64, M, (256, 256), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
        assert np.array_equal(P.warp_affine_f64(f64, M, 256, 256), want)
    for sigma in (0.0989, 0.6, 1.4603, 3.2):
        want = ndi.gaussian_filter(img.astype(float), [sigma, sigma, 0.0], mode="nearest", truncate=4.0)
        np.testing.assert_allclose(P.gaussian_blur(img, sigma), want, rtol=0, atol=1e-12)


def test_oracle_equals_live_reference_dataset(golden_dir):
    """Every crop equals the reference ViTDetDataset's bit for bit: a strided sample is compared value by value, the whole
    crop through its SHA-256."""
    g = np.load(golden_dir / "preproc_live.npz")
    img, boxes = live_preproc_scene()
    assert np.array_equal(boxes, g["boxes"])
    stride = int(g["stride"])
    for name, shape in (("shape", (192, 256)), ("noshape", None)):
        for i in range(len(boxes)):
            it = P.vitdet_item(img, boxes[i], bbox_shape=shape)
            assert str(it["img"].dtype) == str(g[f"{name}_img_dtype"])
            assert np.array_equal(it["img"].ravel()[::stride], g[f"{name}_img_flat"][i]), f"{name} box {i}"
            assert hashlib.sha256(np.ascontiguousarray(it["img"]).tobytes()).hexdigest() == g[f"{name}_img_sha256"][i]
            assert np.array_equal(it["box_center"], g[f"{name}_box_center"][i]) and it["box_size"] == g[f"{name}_box_size"][i]


# ------------------------------------------------------------------------------------------------ host planner
def test_host_planner_matches_oracle_bit_for_bit(built_lib):
    from tokenhmr_b200.preprocess import plan_boxes
    rng = np.random.default_rng(3)
    n = 1500
    x0, y0 = rng.uniform(-200, 3000, n), rng.uniform(-200, 2000, n)
    w, h = rng.uniform(5, 2500, n), rng.uniform(5, 2500, n)
    boxes = np.stack([x0, y0, x0 + w, y0 + h], 1).astype(np.float32)
    for shape in ((192, 256), None):
        pl = plan_boxes(boxes, bbox_shape=shape)
        for i in range(n):
            c, s = P.box_center_scale(boxes[i:i + 1])
            size = P.bbox_size(s[0], shape)
            sigma = P.blur_sigma(size, 256)
            assert np.array_equal(c[0], pl["box_center"][i]) and size == pl["box_size"][i]
            assert (0.0 if sigma is None else sigma) == pl["sigma"][i]
            if i < 300:
                iM = P.invert_affine(P.gen_trans(c[0, 0], c[0, 1], size, 256))
                assert np.array_equal(iM, pl["inv_affine"][i])


def test_planner_rejects_empty_boxes(built_lib):
    from tokenhmr_b200._lib import ThmrError
    from tokenhmr_b200.preprocess import plan_boxes
    with pytest.raises(ThmrError, match="empty"):
        plan_boxes(np.float32([[10, 10, 10, 50]]))


# ------------------------------------------------------------------------------------------------ GPU parity
@pytest.mark.gpu
def test_gpu_preprocess_matches_reference_golden(cuda_dev, golden_dir):
    from tokenhmr_b200.preprocess import ViTDetPreprocessor
    g, img, boxes, ref = _golden(golden_dir)
    batch = ViTDetPreprocessor(device=cuda_dev)(img, boxes, return_patch=True)
    torch.cuda.synchronize()
    got = batch["img"].cpu().numpy()
    u8 = g["is_u8"]
    assert np.array_equal(batch["_sigma"] == 0, u8)
    # 8-bit path: bit exact, both the byte crop cv2 returns and the normalised tensor
    assert np.array_equal(batch["_patch_bgr_u8"].cpu().numpy()[u8][..., ::-1].transpose(0, 3, 1, 2), g["rgb_u8"])
    assert np.array_equal(got[u8], ref[u8])
    # blurred path: the Gaussian is stored as fp32 between the passes (reference: float64) -> 1e-5 of the 0..255 range
    err = np.abs(got[~u8] - ref[~u8]).max()
    assert err < 2e-5, err
    assert np.array_equal(batch["box_center"].cpu().numpy(), g["box_center"])
    assert np.array_equal(batch["box_size"].cpu().numpy(), g["box_size"])
    assert np.array_equal(batch["img_size"].cpu().numpy(), g["img_size"])


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,n", [(97, 131, 5), (720, 1280, 16), (1080, 1920, 8)])
def test_gpu_preprocess_vs_oracle(cuda_dev, H, W, n):
    from tokenhmr_b200.preprocess import ViTDetPreprocessor
    rng = np.random.default_rng(H + n)
    img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    cx, cy = rng.uniform(0, W, n), rng.uniform(0, H, n)
    w, h = rng.uniform(20, 0.9 * W, n), rng.uniform(20, 0.9 * H, n)
    boxes = np.stack([cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2], 1).astype(np.float32)
    pre = ViTDetPreprocessor(device=cuda_dev)
    batch = pre(torch.from_numpy(img).to(cuda_dev), boxes, return_patch=True)
    got = batch["img"].cpu().numpy()
    n_blur = 0
    for i in range(n):
        it = P.vitdet_item(img, boxes[i])
        if it["sigma"] is None:
            assert np.array_equal(batch["_patch_bgr_u8"][i].cpu().numpy(), it["patch"]), f"box {i}"
            assert np.array_equal(got[i], it["img"]), f"box {i}"
        else:
            n_blur += 1
            assert np.abs(got[i] - it["img"]).max() < 2e-5, f"box {i} sigma {it['sigma']}"
    if W >= 1280:
        assert n_blur > 0


@pytest.mark.gpu
def test_gpu_preprocess_feeds_the_engine_surface(cuda_dev):
    """The batch dict has the keys / dtypes demo.py:72-118 reads after the DataLoader collate."""
    from tokenhmr_b200.preprocess import ViTDetPreprocessor
    img = np.zeros((64, 80, 3), np.uint8)
    img[..., 0], img[..., 1], img[..., 2] = 10, 20, 30                         # B, G, R
    batch = ViTDetPreprocessor(device=cuda_dev)(img, np.float32([[10, 10, 60, 50]]))
    assert batch["img"].shape == (1, 3, 256, 256) and batch["img"].dtype == torch.float32
    centre = batch["img"][0, :, 128, 128].cpu().numpy()                         # RGB planes of a constant frame
    want = ((np.array([30.0, 20.0, 10.0]) - MEAN) / STD).astype(np.float32)
    assert np.array_equal(centre, want)
    assert batch["img"][0, :, 0, 0].cpu().numpy().tolist() == ((0 - MEAN) / STD).astype(np.float32).tolist()  # border = 0
    assert batch["personid"].tolist() == [0] and batch["img_size"].tolist() == [[80.0, 64.0]]
