"""CPU check of the host-side graph logic: drive cvvae_b200's engine + wrapper through the torch
restatement of the operator set (tests/fake_ops.py) and compare with the reference's golden outputs.

This validates padding modes/offsets, time interleave, attention plumbing, tiling/chunking/blending and the
state-dict schema without a GPU.  The CUDA kernels themselves are covered by the `-m gpu` tests.
"""
import json
import os

import numpy as np
import pytest
import torch

from cvvae_b200 import CVVAEModel, CVVAESD3Model
from fake_ops import FakeOps
from golden_data import stored
from oracle import cvvae_oracle as O

GOLD = os.path.join(os.path.dirname(__file__), "golden")
with open(os.path.join(GOLD, "manifest.json")) as f:
    MANIFEST = json.load(f)
CASES = {c["name"]: c for c in MANIFEST["cases"]}


def build_model(case, ops_factory=FakeOps):
    widths = [case["ch"] * m for m in (1, 2, 4, 4)]
    if case["variant"] == "sd21":
        m = CVVAEModel(ch=case["ch"], **case["wrap"])
        cfg = O.VAEConfig(variant="sd21", ch=case["ch"], **case["wrap"])
    else:
        m = CVVAESD3Model(block_out_channels=widths, **case["wrap"])
        cfg = O.VAEConfig(variant="sd3", ch=case["ch"], z_channels=16, **case["wrap"])
    m.load_state_dict(O.make_state_dict(cfg, MANIFEST["weight_seed"]), strict=True)
    m._ops_factory = ops_factory
    return m, cfg


@pytest.mark.parametrize("name", sorted(CASES))
def test_engine_graph_matches_reference(name):
    case = CASES[name]
    m, _ = build_model(case)
    gold = np.load(os.path.join(GOLD, name + ".npz"))
    x = O.synthetic_video(case["shape"], MANIFEST["input_seed"])
    post = m.encode(x).latent_dist
    rec = m.decode(post.mode()).sample
    # fp32 library kernels in a different association order than the reference: tight but not bit-exact
    assert list(rec.shape) == case["outputs"]["recon"]
    np.testing.assert_allclose(post.parameters.numpy(), gold["moments"], rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(stored(gold, "recon", rec.numpy()), gold["recon"], rtol=1e-4, atol=5e-5)
    if "recon_4d" in gold.files:
        z = post.mode()
        z4 = z.permute(0, 2, 1, 3, 4).reshape(-1, z.shape[1], *z.shape[3:])
        rec4 = m.decode(z4, num_frames=1).sample
        np.testing.assert_allclose(rec4.numpy(), gold["recon_4d"], rtol=1e-4, atol=5e-5)
    if "recon_4dlat" in gold.files:
        z = post.mode()
        z4 = z.permute(0, 2, 1, 3, 4).reshape(-1, z.shape[1], *z.shape[3:])
        np.testing.assert_allclose(m.decode(z4).sample.numpy(), gold["recon_4dlat"], rtol=1e-4, atol=5e-5)


def test_surface_matches_reference_contract(tmp_path):
    m = CVVAEModel(ch=32)
    # config access both ways, reference defaults (modeling_vae.py:26-50)
    assert m.config.scaling_factor == 0.18215 and m.config["spatial_n_compress"] == 8
    assert (m.encode_n_frames_a_time, m.decode_n_frames_a_time, m.pixel_tile_size, m.latent_tile_size) == (16, 4, 576, 72)
    m.save_pretrained(str(tmp_path / "vae3d"))
    m2 = CVVAEModel.from_pretrained(str(tmp_path), subfolder="vae3d", torch_dtype=torch.float16)
    assert m2.dtype == torch.float16 and m2.config.ch == 32
    for (k1, v1), (k2, v2) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert k1 == k2 and torch.equal(v1.half(), v2)
    # no silent CPU path in production
    m3 = CVVAEModel(ch=32).half()
    with pytest.raises(RuntimeError, match="CUDA"):
        m3.encode(torch.zeros(1, 3, 1, 16, 16, dtype=torch.float16))
    # return_dict=False tuples and forward()
    m._ops_factory = FakeOps
    x = O.synthetic_video((1, 3, 5, 16, 16), 1)
    (post,) = m.encode(x, return_dict=False)
    (rec,) = m.decode(post.mode(), return_dict=False)
    out = m(x).sample
    assert torch.equal(out, rec) and rec.shape == x.shape
    assert m.encoder(x).shape == (1, 8, 2, 2, 2)


@pytest.mark.parametrize("variant", ["sd21", "sd3"])
def test_single_frame_time_tap_folding(variant):
    """T = 1 (image path): the engine folds the time taps of every 3x3x3 conv and computes only the kept half of the
    up_time convs; the result must equal the oracle's literal execution (pad, conv, interleave, drop)."""
    case = dict(variant=variant, ch=32, wrap=dict(tile_spatial_size=None, en_de_n_frames_a_time=None))
    m, cfg = build_model(case)
    sd = O.make_state_dict(cfg, MANIFEST["weight_seed"])
    x = O.synthetic_video((2, 3, 1, 40, 24), 5)
    want_post = O.encode(x, sd, cfg)
    want_rec = O.decode(want_post.mode(), sd, cfg)
    post = m.encode(x).latent_dist
    rec = m.decode(post.mode()).sample
    assert rec.shape == want_rec.shape == (2, 3, 1, 40, 24)
    np.testing.assert_allclose(post.parameters.numpy(), want_post.parameters.numpy(), rtol=1e-4, atol=2e-5)
    np.testing.assert_allclose(rec.numpy(), want_rec.numpy(), rtol=1e-4, atol=5e-5)
    folded = [k for k in m._engine().p if ".t1." in k and not k.endswith(".bias")]
    # 2x2 phases / 3x3 / tap-packed network-input convs (1 tap over 9*Cin channels): no time taps left
    assert folded and all(m._engine().p[k].shape[0] in (4, 9) or (".hwpack" in k and m._engine().p[k].shape[0] == 1) for k in folded)


def test_diagonal_gaussian_distribution_contract():
    """diffusers' DiagonalGaussianDistribution as the reference uses it (models/modeling_vae.py:223; training twin
    lvdm/modules/distributions/distributions.py:24-73): chunk, logvar clamp to [-30, 20], std = exp(0.5 logvar),
    sample(generator) = mean + std * randn (diffusers randn_tensor: drawn on the generator's device), mode = mean."""
    from cvvae_b200.modeling_vae import DiagonalGaussianDistribution
    g = torch.Generator().manual_seed(5)
    moments = torch.randn((2, 8, 3, 4, 5), generator=g) * 3
    moments[0, 4, 0, 0, 0], moments[0, 5, 0, 0, 0] = -100.0, 100.0      # outside the clamp
    d = DiagonalGaussianDistribution(moments)
    mean, logvar = torch.chunk(moments, 2, dim=1)
    assert d.parameters is moments and torch.equal(d.mean, mean) and torch.equal(d.mode(), mean)
    assert torch.equal(d.logvar, logvar.clamp(-30.0, 20.0))
    assert d.logvar.min().item() == -30.0 and d.logvar.max().item() == 20.0
    assert torch.equal(d.std, torch.exp(0.5 * d.logvar)) and torch.equal(d.var, torch.exp(d.logvar))
    g1, g2 = torch.Generator().manual_seed(11), torch.Generator().manual_seed(11)
    s = d.sample(generator=g1)
    want = d.mean + d.std * torch.randn(d.mean.shape, generator=g2, dtype=moments.dtype)
    assert torch.equal(s, want) and s.shape == mean.shape
    assert not torch.equal(d.sample(), d.sample())                       # global RNG when no generator is given
    det = DiagonalGaussianDistribution(moments, deterministic=True)
    assert torch.equal(det.sample(generator=torch.Generator().manual_seed(1)), det.mean) and det.std.abs().max().item() == 0


def test_forward_sample_posterior_uses_the_generator():
    """forward(sample, sample_posterior=True, generator=g) (models/modeling_vae.py:114-142) = decode(posterior.sample(g))."""
    case = dict(variant="sd21", ch=32, wrap=dict(tile_spatial_size=None, en_de_n_frames_a_time=None))
    m, _ = build_model(case)
    x = O.synthetic_video((1, 3, 5, 16, 16), 2)
    a = m(x, sample_posterior=True, generator=torch.Generator().manual_seed(7)).sample
    post = m.encode(x).latent_dist
    b = m.decode(post.sample(generator=torch.Generator().manual_seed(7))).sample
    assert torch.equal(a, b) and not torch.equal(a, m(x).sample)


def test_in_place_weight_update_repacks():
    """The pre-packed weight cache follows in-place parameter updates (copy_ under no_grad), like the reference modules;
    invalidate_weights() covers writes through `.data`, which carry no version counter."""
    case = dict(variant="sd21", ch=32, wrap=dict(tile_spatial_size=None, en_de_n_frames_a_time=None))
    m, _ = build_model(case)
    x = O.synthetic_video((1, 3, 1, 16, 16), 2)
    z0 = m.encode(x).latent_dist.parameters.clone()
    w = dict(m.named_parameters())["encoder.conv_in.weight"]
    with torch.no_grad():
        w.mul_(0.5)
    z1 = m.encode(x).latent_dist.parameters.clone()
    assert not torch.equal(z0, z1)
    w.data.mul_(2.0)
    m.invalidate_weights()
    assert torch.allclose(m.encode(x).latent_dist.parameters, z0, rtol=1e-5, atol=1e-6)


def test_chunk_tile_assembly_equals_reference_concatenation():
    """The single-copy assembly (every (chunk, tile) result written once into the pre-allocated clip) equals the
    reference's crop + cat over columns + cat over rows + cat over chunks (modeling_vae.py:181-191, 207-210)."""
    case = CASES["sd21_w32_tiled"]
    m, cfg = build_model(case)
    x = O.synthetic_video((1, 3, 13, 104, 120), 4)         # 3 chunks x (2 x 2) tiles
    mom = m.encode(x).latent_dist.parameters
    g = O.TileGeometry.of(cfg)
    outs = []
    for n in range(3):
        o = O._spatial_tiled(x[:, :, 4 * n:4 * n + 5], lambda t: m.encoder(t.contiguous()), g.pixel_tile, g.latent_tile, g.ratio, True)
        outs.append(o if n == 0 else o[:, :, 1:])
    assert torch.equal(mom, torch.cat(outs, dim=2))
