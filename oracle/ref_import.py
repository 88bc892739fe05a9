"""Import the reference's own PyTorch modules file by file (build container only).  TEST INFRASTRUCTURE.

/root/reference cannot be imported as a package here: lib/models/__init__.py pulls pytorch_lightning,
yacs, smplx, pyrender, ... none of which are installed (SURVEY.md §8c).  The individual model files
import fine once
  * empty namespace packages stand in for the package __init__ files (so relative imports resolve
    without executing them),
  * `timm.models.layers` is shimmed (only import of timm: backbones/vit.py:10),
  * `smplx` is stubbed (import-time body-model load in tokenization/models/vanilla_pose_vqvae.py:10-17),
  * torch.Tensor.cuda is neutralised on a CPU-only host (quantize_cnn.py:18 hard-codes .cuda()).
Nothing is copied: the modules execute from the reference tree where they lie.  This file is used by
oracle/make_golden.py, which writes tests/golden/*.npz; the tests compare with those files and never need
the reference tree.
"""
from __future__ import annotations

import argparse
import importlib
import importlib.util
import os
import sys
import tempfile
import types
from pathlib import Path
from typing import Dict

import numpy as np
import torch

REF_ROOT = Path(os.environ.get("TOKENHMR_REFERENCE", "/root/reference"))


def available() -> bool:
    """True when the reference tree is present and readable (a tree the user may not enter counts as absent)."""
    try:
        return (REF_ROOT / "tokenhmr" / "lib" / "models" / "backbones" / "vit.py").is_file()
    except OSError:
        return False


def _namespace(name: str, path: Path) -> None:
    if name in sys.modules:
        return
    m = types.ModuleType(name)
    m.__path__ = [str(path)]
    m.__package__ = name
    sys.modules[name] = m


def _install_shims() -> None:
    # --- timm.models.layers: drop_path, to_2tuple, trunc_normal_
    if "timm" not in sys.modules:
        timm = types.ModuleType("timm")
        models = types.ModuleType("timm.models")
        layers = types.ModuleType("timm.models.layers")

        def to_2tuple(x):
            return tuple(x) if isinstance(x, (tuple, list)) else (x, x)

        def trunc_normal_(t, mean=0., std=1., a=-2., b=2.):
            return torch.nn.init.trunc_normal_(t, mean=mean, std=std, a=a, b=b)

        def drop_path(x, drop_prob: float = 0., training: bool = False):
            if drop_prob == 0. or not training:
                return x
            raise RuntimeError("drop_path in training mode is outside the inference path")

        layers.to_2tuple, layers.trunc_normal_, layers.drop_path = to_2tuple, trunc_normal_, drop_path
        timm.models, models.layers = models, layers
        sys.modules.update({"timm": timm, "timm.models": models, "timm.models.layers": layers})
    # --- smplx stub (only so that `from smplx import SMPLHLayer, SMPLXLayer` and the import-time
    #     `body_model = SMPLHLayer(path, ...)` in vanilla_pose_vqvae.py succeed; never used on the path)
    if "smplx" not in sys.modules:
        smplx = types.ModuleType("smplx")

        class _Layer(torch.nn.Module):
            def __init__(self, *a, **k):
                super().__init__()

        smplx.SMPLLayer = smplx.SMPLHLayer = smplx.SMPLXLayer = _Layer
        sys.modules["smplx"] = smplx
    if not torch.cuda.is_available():
        torch.Tensor.cuda = lambda self, *a, **k: self  # quantize_cnn.py:18


def load_modules() -> types.SimpleNamespace:
    """Returns the reference modules on the forward path (imported from REF_ROOT, unmodified)."""
    if not available():
        raise FileNotFoundError(f"reference tree not found at {REF_ROOT}")
    _install_shims()
    lib = REF_ROOT / "tokenhmr" / "lib"
    _namespace("lib", lib)
    _namespace("lib.models", lib / "models")
    _namespace("lib.models.backbones", lib / "models" / "backbones")
    _namespace("lib.models.components", lib / "models" / "components")
    _namespace("lib.models.heads", lib / "models" / "heads")
    _namespace("lib.utils", lib / "utils")
    _namespace("tokenization", REF_ROOT / "tokenization")
    _namespace("tokenization.models", REF_ROOT / "tokenization" / "models")
    ns = types.SimpleNamespace()
    ns.vit = importlib.import_module("lib.models.backbones.vit")
    ns.geometry = importlib.import_module("lib.utils.geometry")
    ns.pose_transformer = importlib.import_module("lib.models.components.pose_transformer")
    ns.quantize_cnn = importlib.import_module("tokenization.models.quantize_cnn")
    import contextlib, io
    with contextlib.redirect_stdout(io.StringIO()):
        ns.vqvae = importlib.import_module("tokenization.models.vanilla_pose_vqvae")
        ns.token_classifier = importlib.import_module("lib.models.heads.token_classifier")
        ns.token_head = importlib.import_module("lib.models.heads.token_head")
    return ns


def load_eval_modules() -> types.SimpleNamespace:
    """The reference's evaluation helpers: lib/utils/pose_utils.py (imports cleanly: cv2 + torch) and
    lib/utils/renderer.py for cam_crop_to_full (module-level imports of pyrender / trimesh / yacs are stubbed; the
    function itself is plain torch, renderer.py:13-23)."""
    load_modules()
    class _Anything(types.ModuleType):   # annotations such as List[pyrender.Node] are evaluated at import
        def __getattr__(self, k):
            return type(k, (), {})

    for name in ("pyrender", "trimesh"):
        if name not in sys.modules:
            sys.modules[name] = _Anything(name)
    if "yacs" not in sys.modules:
        yacs, yc = types.ModuleType("yacs"), types.ModuleType("yacs.config")
        yc.CfgNode = dict
        yacs.config = yc
        sys.modules.update({"yacs": yacs, "yacs.config": yc})
    ns = types.SimpleNamespace()
    ns.pose_utils = importlib.import_module("lib.utils.pose_utils")
    prev = os.environ.get("PYOPENGL_PLATFORM")
    ns.renderer = importlib.import_module("lib.utils.renderer")   # sets PYOPENGL_PLATFORM at import
    if prev is None:
        os.environ.pop("PYOPENGL_PLATFORM", None)
    else:
        os.environ["PYOPENGL_PLATFORM"] = prev
    return ns


def load_dataset_modules() -> types.SimpleNamespace:
    """The reference's inference pre-processing: lib/datasets/vitdet_dataset.py and lib/datasets/utils.py (SURVEY
    §8 row f2).  cv2 and scipy are real here; skimage is absent, so `skimage.filters.gaussian` is a shim that does
    what skimage itself does for this call (uint8 -> float64 with preserve_range, scipy.ndimage.gaussian_filter
    over the image axes, mode 'nearest', truncate 4.0); `skimage.transform.rotate/resize` (training-only crop
    path, utils.py:6) and yacs.config.CfgNode (annotation only) are stubbed."""
    load_modules()
    if "skimage" not in sys.modules:
        import scipy.ndimage as ndi
        sk, skf, skt = types.ModuleType("skimage"), types.ModuleType("skimage.filters"), types.ModuleType("skimage.transform")

        def gaussian(image, sigma=1, *, mode="nearest", cval=0, preserve_range=False, truncate=4.0, channel_axis=None):
            assert preserve_range and channel_axis is not None, "only the vitdet_dataset.py:66 call is shimmed"
            img = image if image.dtype.char in "df" else image.astype(float)
            sig = [float(sigma)] * img.ndim
            sig[channel_axis] = 0.0
            return ndi.gaussian_filter(img, sig, mode=mode, cval=cval, truncate=truncate)

        def _unused(*a, **k):
            raise RuntimeError("skimage.transform is outside the inference path")

        skf.gaussian, skt.rotate, skt.resize = gaussian, _unused, _unused
        sk.filters, sk.transform = skf, skt
        sys.modules.update({"skimage": sk, "skimage.filters": skf, "skimage.transform": skt})
    if "yacs" not in sys.modules:
        yacs, yc = types.ModuleType("yacs"), types.ModuleType("yacs.config")
        yc.CfgNode = dict
        yacs.config = yc
        sys.modules.update({"yacs": yacs, "yacs.config": yc})
    _namespace("lib.datasets", REF_ROOT / "tokenhmr" / "lib" / "datasets")
    ns = types.SimpleNamespace()
    ns.utils = importlib.import_module("lib.datasets.utils")
    ns.vitdet_dataset = importlib.import_module("lib.datasets.vitdet_dataset")
    return ns


def dataset_cfg(image_size: int = 256, bbox_shape=(192, 256)):
    """The MODEL keys ViTDetDataset reads (vitdet_dataset.py:31-33,52); values of the release model_config.yaml."""
    return _Cfg({"MODEL": {"IMAGE_SIZE": image_size, "IMAGE_MEAN": [0.485, 0.456, 0.406],
                           "IMAGE_STD": [0.229, 0.224, 0.225], "BBOX_SHAPE": list(bbox_shape) if bbox_shape else None}})


class _Cfg(dict):
    """Duck-typed stand-in for the yacs CfgNode the reference constructors read (attribute + .get access)."""

    def __getattr__(self, k):
        try:
            v = self[k]
        except KeyError as e:
            raise AttributeError(k) from e
        return _Cfg(v) if isinstance(v, dict) and not isinstance(v, _Cfg) else v


def _sub(sd: Dict[str, torch.Tensor], prefix: str) -> Dict[str, torch.Tensor]:
    return {k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)}


def build_backbone(ns, sd, cfg):
    """vit() (vit.py:12-24) with the synthetic backbone.* weights, eval mode."""
    assert cfg.vit_dim == 1280 and cfg.vit_heads == 16, "reference vit() is fixed to ViT-H"
    if cfg.vit_depth == 32:
        model = ns.vit.vit()
    else:  # same class, fewer blocks (tests)
        model = ns.vit.ViT(img_size=(256, 192), patch_size=16, embed_dim=1280, depth=cfg.vit_depth, num_heads=16,
                           ratio=1, use_checkpoint=False, mlp_ratio=4, qkv_bias=True, drop_path_rate=0.55)
    model.load_state_dict(_sub(sd, "backbone."), strict=True)
    torch.nn.Module.eval(model)  # ViT.train() does not return self (vit.py:345-348)
    return model


def build_head(ns, sd, cfg):
    """SMPLTokenDecoderHead (token_head.py:20-63) built by the reference constructor: duck-typed cfg, a
    temporary mean-params .npz and a torch.load patched to hand back the synthetic tokenizer 'checkpoint'
    ({'hparams': ..., 'net': ...}, vanilla_pose_vqvae.py:265-301)."""
    tok_sd = {k[len("tokenizer."):]: v for k, v in sd.items() if k.startswith("tokenizer.")}
    arch = argparse.Namespace(ROT_TYPE="rot6d", CODE_DIM=cfg.code_dim, NB_CODE=cfg.nb_code, DOWN_T=1,
                              WIDTH=cfg.tok_width, DEPTH=cfg.tok_depth, DILATION_RATE=cfg.tok_dilation_rate,
                              TOKEN_SIZE_DIV=cfg.tok_size_div, TOKEN_SIZE_MUL=4)
    fake_ckpt = {"hparams": argparse.Namespace(ARCH=arch), "net": tok_sd}
    with tempfile.TemporaryDirectory() as td:
        npz = os.path.join(td, "smpl_mean_params.npz")
        np.savez(npz, pose=sd["smpl_head.init_body_pose"][0].numpy(), shape=sd["smpl_head.init_betas"][0].numpy(),
                 cam=sd["smpl_head.init_cam"][0].numpy())
        rcfg = _Cfg({
            "MODEL": {"SMPL_HEAD": {"TYPE": "token", "JOINT_REP": "6d", "TRANSFORMER_INPUT": "zero", "IEF_ITERS": 1,
                                    "TOKENIZER": {"TOKENIZER_TYPE": "Vanilla", "TOKEN_CODE_DIM": cfg.code_dim,
                                                  "TOKEN_NUM": cfg.token_num,
                                                  "TOKEN_CLASS_NUM": cfg.token_class_num},
                                    "TRANSFORMER_DECODER": {"depth": cfg.dec_depth, "heads": cfg.dec_heads,
                                                            "mlp_dim": cfg.dec_mlp_dim,
                                                            "dim_head": cfg.dec_dim_head, "dropout": 0.0,
                                                            "emb_dropout": 0.0, "norm": "layer",
                                                            "context_dim": cfg.vit_dim}},
                      "TOKENIZER_CHECKPOINT_PATH": "synthetic-tokenizer.pth"},
            "SMPL": {"NUM_BODY_JOINTS": cfg.num_joints - 1, "MEAN_PARAMS": npz},
        })
        real_load = torch.load
        torch.load = lambda *a, **k: fake_ckpt
        import contextlib, io
        try:
            with contextlib.redirect_stdout(io.StringIO()):
                head = ns.token_head.SMPLTokenDecoderHead(rcfg)
        finally:
            torch.load = real_load
    own = {k: v for k, v in _sub(sd, "smpl_head.").items()}
    missing, unexpected = head.load_state_dict(own, strict=False)
    assert not unexpected, unexpected
    assert not missing, missing
    head.eval()
    return head


def build_encode_tokens(ns, sd, cfg):
    """EncodeTokens (vanilla_pose_vqvae.py:304-346) built by the reference constructor from a synthetic tokenizer
    'checkpoint' ({'hparams', 'net'}); `sd` holds tokenizer.encoder.* and tokenizer.quantizer.codebook."""
    tok_sd = {k[len("tokenizer."):]: v for k, v in sd.items()
              if k.startswith(("tokenizer.encoder.", "tokenizer.quantizer."))}
    arch = argparse.Namespace(ROT_TYPE="rot6d", CODE_DIM=cfg.code_dim, NB_CODE=cfg.nb_code, DOWN_T=1,
                              WIDTH=cfg.tok_width, DEPTH=cfg.tok_depth, DILATION_RATE=cfg.tok_dilation_rate,
                              TOKEN_SIZE_DIV=cfg.tok_size_div, TOKEN_SIZE_MUL=cfg.tok_size_mul)
    fake_ckpt = {"hparams": argparse.Namespace(ARCH=arch), "net": tok_sd}
    real_load = torch.load
    torch.load = lambda *a, **k: fake_ckpt
    import contextlib, io
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            enc = ns.vqvae.EncodeTokens("synthetic-tokenizer.pth")
    finally:
        torch.load = real_load
    enc.eval()
    return enc


def reference_forward(ns, backbone, head, smpl, img, cfg):
    """TokenHMR.forward_step (tokenhmr.py:135-188) glue around the LIVE reference backbone / head / geometry;
    only the smplx call (tokenhmr.py:176) goes to the unpinned restatement in smpl_oracle."""
    from . import smpl_oracle
    with torch.no_grad():
        B = img.shape[0]
        feats = backbone(img)                                          # (B,1280,16,12)
        params, pred_cam, lists = head(feats)
        out = {"cls_logits_softmax": lists["cls_logits_softmax"], "pred_cam": pred_cam,
               "pred_smpl_params": {k: v.clone() for k, v in params.items()}}
        focal = cfg.focal_length * torch.ones(B, 2)
        cam_t = torch.stack([pred_cam[:, 1], pred_cam[:, 2],
                             2 * focal[:, 0] / (cfg.image_size * pred_cam[:, 0] + 1e-9)], dim=-1)
        out["pred_cam_t"], out["focal_length"] = cam_t, focal
        verts, joints = smpl_oracle.smpl_forward(smpl, params["global_orient"], params["body_pose"],
                                                 params["betas"])
        out["pred_keypoints_3d"], out["pred_vertices"] = joints, verts
        out["pred_keypoints_2d"] = ns.geometry.perspective_projection(
            joints, translation=cam_t, focal_length=focal / cfg.image_size)
        out["_vit_tokens"] = feats.flatten(2).transpose(1, 2).contiguous()
    return out
