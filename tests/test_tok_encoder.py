"""Tokenizer encoder + hard quantisation (SURVEY §8 row f4).  CPU: the oracle restatement of EncodeTokens.forward is
pinned against the golden indices and latents the LIVE reference class produced.  GPU:
thmr_tok_encode vs the oracle (index agreement, latent error) and the goldens."""
import numpy as np
import pytest
import torch

from oracle import tokenhmr_oracle as O
from tokenhmr_b200 import synth
from tokenhmr_b200.config import release_config


def _golden(golden_dir):
    g = np.load(golden_dir / "tok_encoder.npz")
    cfg = release_config()
    sd = synth.make_tokenizer_encoder_state_dict(cfg, int(g["meta"][0]))
    sd2 = dict(sd)
    sd2["tokenizer.quantizer.codebook"] = torch.from_numpy(g["codebook_latent"].astype(np.float32))
    return g, cfg, sd, sd2, torch.from_numpy(g["x"])


def test_oracle_matches_reference_golden(golden_dir):
    g, cfg, sd, sd2, x = _golden(golden_dir)
    with torch.no_grad():
        idx, lat = O.tokenizer_encode(sd, x, cfg, O.Numerics(False))
        idx2, _ = O.tokenizer_encode(sd2, x, cfg, O.Numerics(False))
    assert idx.shape == (x.shape[0] * 160,) and idx.dtype == torch.int64
    np.testing.assert_allclose(lat[::7].numpy(), g["latent_sub"], rtol=0, atol=2e-5)
    assert np.array_equal(idx.numpy(), g["idx_synth"])
    assert np.array_equal(idx2.numpy(), g["idx_latent_cb"])
    assert len(np.unique(g["idx_latent_cb"])) > 300          # the second codebook spreads the indices


def test_oracle_equals_live_reference_encoder(golden_dir):
    """Other weights, other poses: indices and latents equal what the reference EncodeTokens computed."""
    g = np.load(golden_dir / "tok_encoder_seed77.npz")
    w_seed, x_seed, batch = (int(v) for v in g["meta"])
    cfg = release_config()
    sd = synth.make_tokenizer_encoder_state_dict(cfg, w_seed)
    x = torch.randn(batch, cfg.tok_joints, 6, generator=torch.Generator().manual_seed(x_seed))
    with torch.no_grad():
        idx, lat = O.tokenizer_encode(sd, x, cfg, O.Numerics(False))
    assert torch.equal(idx, torch.from_numpy(g["idx"].astype(np.int64)))
    torch.testing.assert_close(lat.flatten()[::int(g["stride"])], torch.from_numpy(g["latent_flat"]), rtol=0, atol=1e-6)


def test_encoder_state_dict_shares_the_codebook_with_the_forward_weights():
    cfg = release_config()
    a = synth.make_tokenizer_encoder_state_dict(cfg)
    assert a["tokenizer.encoder.encoder.0.weight"].shape == (cfg.tok_width, 6, 3)
    assert a["tokenizer.encoder.encoder.14.0.weight"].shape == (cfg.tok_width, cfg.tok_width, 4)
    assert a["tokenizer.encoder.encoder.15.weight"].shape == (cfg.code_dim, cfg.tok_width, 3)
    from tokenhmr_b200.synth import _Maker
    m = _Maker(1234)
    m.normal("tokenizer.quantizer.codebook", (cfg.nb_code, cfg.code_dim), 1.0)
    assert torch.equal(a["tokenizer.quantizer.codebook"], m.sd["tokenizer.quantizer.codebook"])


# The encoder runs in split precision (fp32-grade): its indices must EQUAL the fp32 reference's.  The only admissible
# differences are queries whose two nearest codes are closer than the fp32 evaluation noise of the distance itself
# (d = |x|^2 - 2 x.c + |c|^2 cancels ~3 digits: with |x|^2 ~ 1e2..1e3 the fp32 noise of d is ~1e-4): gated per element.
TIE_GAP = 2e-3
MAX_TIE_FRAC = 0.005


def _assert_indices_exact(idx_gpu, ref_idx, gap, what):
    diff = idx_gpu.cpu() != ref_idx
    frac = diff.float().mean().item()
    worst = gap[diff].max().item() if diff.any() else 0.0
    print(f"{what}: {int(diff.sum())} of {diff.numel()} indices differ, largest reference top-2 gap among them {worst:.2e}")
    assert (gap[diff] < TIE_GAP).all(), (what, gap[diff])
    assert frac <= MAX_TIE_FRAC, (what, frac)


@pytest.mark.gpu
def test_gpu_encode_matches_reference_golden(cuda_dev, golden_dir):
    from tokenhmr_b200.tokenizer import EncodeTokens
    g, cfg, sd, sd2, x = _golden(golden_dir)
    with torch.no_grad():
        _, lat32 = O.tokenizer_encode(sd, x, cfg, O.Numerics(False))       # == the live reference (pinned above)
    for s, key in ((sd, "idx_synth"), (sd2, "idx_latent_cb")):
        enc = EncodeTokens(cfg, s, device=cuda_dev)
        idx, lat = enc(x, return_latent=True)
        torch.cuda.synchronize()
        assert idx.shape == (x.shape[0] * 160,) and idx.dtype == torch.int64 and enc.num_tokens == 160
        ref_lat = torch.from_numpy(g["latent_sub"])
        err = (lat.cpu()[::7] - ref_lat).abs().max().item() / ref_lat.abs().max().item()
        assert err < 2e-5, err                             # fp32-grade through 9 conv layers
        gap = O.vq_top2_gap(lat32, s["tokenizer.quantizer.codebook"])
        _assert_indices_exact(idx, torch.from_numpy(g[key].astype(np.int64)), gap, key)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 7, 64, 300])
def test_gpu_encode_vs_fp32_oracle(cuda_dev, B):
    from tokenhmr_b200.tokenizer import EncodeTokens
    cfg = release_config()
    sd = synth.make_tokenizer_encoder_state_dict(cfg, 5)
    x = torch.randn(B, cfg.tok_joints, 6, generator=torch.Generator().manual_seed(B))
    with torch.no_grad():
        _, lat32 = O.tokenizer_encode(sd, x, cfg, O.Numerics(False))
    # spread the indices: codebook from the latents themselves (+ noise), as in the golden
    gsel = torch.Generator().manual_seed(1)
    rows = lat32[torch.randint(0, lat32.shape[0], (cfg.nb_code,), generator=gsel)]
    sd["tokenizer.quantizer.codebook"] = rows + 0.05 * torch.randn(cfg.nb_code, cfg.code_dim, generator=gsel)
    ref_idx = O.vq_quantize(lat32, sd["tokenizer.quantizer.codebook"])
    gap = O.vq_top2_gap(lat32, sd["tokenizer.quantizer.codebook"])
    enc = EncodeTokens(cfg, sd, device=cuda_dev)
    idx, lat = enc(x.to(cuda_dev), return_latent=True)
    torch.cuda.synchronize()
    err = (lat.cpu() - lat32).abs().max().item() / lat32.abs().max().item()
    assert err < 2e-5, err
    _assert_indices_exact(idx, ref_idx, gap, f"B={B}")
    # a second call reuses the workspace and is bit-identical; B = 300 spans two kEncChunk passes
    idx_b = enc(x.to(cuda_dev))
    assert torch.equal(idx, idx_b)
    if B > 1:                                        # batch independence: the first pose alone gives the same tokens
        assert torch.equal(enc(x[:1].to(cuda_dev)), idx[:160])


@pytest.mark.gpu
def test_gpu_encode_rejects_bad_shapes(cuda_dev):
    from tokenhmr_b200._lib import ThmrError
    from tokenhmr_b200.tokenizer import EncodeTokens
    cfg = release_config()
    enc = EncodeTokens(cfg, synth.make_tokenizer_encoder_state_dict(cfg, 5), device=cuda_dev)
    with pytest.raises(ThmrError, match="pose must be"):
        enc(torch.zeros(2, 20, 6))
