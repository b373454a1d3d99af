"""End-to-end GPU parity: CVVAEModel / CVVAESD3Model on the CUDA engine vs the reference's golden outputs
(fp32, produced by the unmodified reference) and vs the oracle run in the same 16-bit precision.

Gate (SURVEY.md section 7.4): element-wise rtol=1e-3/atol=1e-4 is the per-operator bar (tests/test_gpu_ops.py).  Two
differently ordered 16-bit pipelines cannot meet it end to end (the reference's own fp16 path misses it on
>60% of elements against its fp32 path), so end to end we require, against the fp32 golden of the UNMODIFIED reference:
  (i)   mean-abs error of this engine <= 1.0 x that of the reference algorithm evaluated in the same 16-bit dtype
        (oracle on torch-CUDA library kernels) - no slack factor, no absolute floor; the max-abs error, an extreme-value
        statistic of up to 3e5 outputs, <= 1.25 x (see tests/test_gpu_fullsize.py for the measured spread);
  (ii)  the fraction of elements inside rtol=1e-3/atol=1e-4 is >= the reference-16-bit path's own fraction (minus two
        binomial standard deviations of that count - the smallest fixtures have 256 moment elements);
both numbers are recorded per case (gpurun_out/e2e_*.json -> profiles/).
"""
import json
import os

import numpy as np
import pytest
import torch

from golden_data import stored
from oracle import cvvae_oracle as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
with open(os.path.join(GOLD, "manifest.json")) as f:
    MANIFEST = json.load(f)
CASES = {c["name"]: c for c in MANIFEST["cases"]}


def _build(case, dtype):
    from cvvae_b200 import CVVAEModel, CVVAESD3Model
    widths = [case["ch"] * m for m in (1, 2, 4, 4)]
    if case["variant"] == "sd21":
        m = CVVAEModel(ch=case["ch"], **case["wrap"])
        cfg = O.VAEConfig(variant="sd21", ch=case["ch"], **case["wrap"])
    else:
        m = CVVAESD3Model(block_out_channels=widths, **case["wrap"])
        cfg = O.VAEConfig(variant="sd3", ch=case["ch"], z_channels=16, **case["wrap"])
    sd = O.make_state_dict(cfg, MANIFEST["weight_seed"])
    m.load_state_dict(sd, strict=True)
    return m.to(dtype).cuda(), cfg, sd


def _err(a, b):
    d = (a.double() - b.double()).abs()
    return d.max().item(), d.mean().item()


def _pass_fraction(a, gold, rtol=1e-3, atol=1e-4):
    """Share of elements with |a - gold| <= atol + rtol |gold| (the north_star tolerance)."""
    a, gold = a.double(), gold.double()
    return ((a - gold).abs() <= atol + rtol * gold.abs()).double().mean().item()


def _gate(mine, ref, what):
    assert mine[0] <= 1.25 * ref[0] and mine[1] <= ref[1], f"{what}: engine error {mine} exceeds the reference-16-bit error {ref}"


@pytest.mark.parametrize("name", sorted(CASES))
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_engine_vs_reference_golden(name, dtype):
    case = CASES[name]
    if dtype == torch.bfloat16 and "w128" not in name:
        pytest.skip("bf16 covered on the full-width cases")
    m, cfg, sd = _build(case, dtype)
    gold = np.load(os.path.join(GOLD, name + ".npz"))
    g_mom = torch.from_numpy(gold["moments"])
    g_rec = torch.from_numpy(gold["recon"])
    x = O.synthetic_video(case["shape"], MANIFEST["input_seed"])
    xd = x.to(dtype).cuda()
    post = m.encode(xd).latent_dist
    rec = m.decode(post.mode()).sample
    torch.cuda.synchronize()
    assert post.parameters.shape == g_mom.shape and list(rec.shape) == case["outputs"]["recon"]
    assert torch.isfinite(rec).all() and torch.isfinite(post.parameters).all()
    # the reference algorithm in the same dtype on torch-CUDA (library kernels) = how far 16-bit drifts anyway
    sd16 = {k: v.to(dtype).cuda() for k, v in sd.items()}
    with torch.no_grad():
        rpost = O.encode(xd, sd16, cfg)
        rrec = O.decode(rpost.mode(), sd16, cfg)
    # reconstructions at the positions the fixture stores (all of them, or its fixed sample for the larger cases)
    rec_s, rrec_s = stored(gold, "recon", rec.cpu()), stored(gold, "recon", rrec.cpu())
    mine_m, mine_r = _err(post.parameters.cpu(), g_mom), _err(rec_s, g_rec)
    ref_m, ref_r = _err(rpost.parameters.cpu(), g_mom), _err(rrec_s, g_rec)
    # decode-only error with the SAME latent as the golden decode used
    z_gold = g_mom[:, : cfg.z_channels].to(dtype).cuda()
    rec2 = m.decode(z_gold).sample
    mine_r2 = _err(stored(gold, "recon", rec2.cpu()), g_rec)
    pf = dict(mine_moments=_pass_fraction(post.parameters.cpu(), g_mom), ref16_moments=_pass_fraction(rpost.parameters.cpu(), g_mom),
              mine_recon=_pass_fraction(rec_s, g_rec), ref16_recon=_pass_fraction(rrec_s, g_rec))
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, f"e2e_{name}_{str(dtype).split('.')[-1]}.json"), "w") as f:
        json.dump(dict(mine_moments=mine_m, mine_recon=mine_r, ref16_moments=ref_m, ref16_recon=ref_r,
                       mine_recon_from_gold_latent=mine_r2, pass_fraction_rtol1e_3_atol1e_4=pf), f, indent=1)
    _gate(mine_m, ref_m, "moments")
    _gate(mine_r, ref_r, "reconstruction")
    # ">= the reference-16-bit path's own fraction", up to the counting noise of the sample: the smallest fixtures have 256
    # moment elements, where one element is 0.4 % - two binomial standard deviations of the reference's count are allowed
    for key, n in (("moments", g_mom.numel()), ("recon", g_rec.numel())):
        ref_pf = pf["ref16_" + key]
        slack = 2.0 * (ref_pf * (1.0 - ref_pf) / n) ** 0.5
        assert pf["mine_" + key] >= ref_pf - slack, (key, pf, slack)
    if "recon_4dlat" in gold.files:
        # 4-D latents regrouped by the model's num_latent_frames: must be the same computation as the 5-D call
        z = post.mode()
        z4 = z.permute(0, 2, 1, 3, 4).reshape(-1, z.shape[1], *z.shape[3:])
        assert torch.equal(m.decode(z4).sample, rec)


def test_forward_and_4d_paths():
    case = CASES["sd21_w32_image"]
    m, cfg, sd = _build(case, torch.float16)
    x = O.synthetic_video(case["shape"], MANIFEST["input_seed"]).half().cuda()
    out = m(x).sample
    assert out.shape == x.shape
    z = m.encode(x).latent_dist.mode()
    z4 = z.permute(0, 2, 1, 3, 4).reshape(-1, z.shape[1], *z.shape[3:])
    rec4 = m.decode(z4, num_frames=1).sample
    gold = np.load(os.path.join(GOLD, "sd21_w32_image.npz"))
    d = (rec4.float().cpu() - torch.from_numpy(gold["recon_4d"])).abs()
    assert d.max().item() < 5e-2 and d.mean().item() < 5e-3


@pytest.mark.parametrize("variant,shape", [("sd21", (1, 3, 5, 40, 56)), ("sd21", (2, 3, 9, 24, 72)), ("sd21", (1, 3, 1, 16, 16)),
                                           ("sd21", (1, 3, 13, 100, 44)), ("sd3", (1, 3, 5, 40, 56)), ("sd3", (2, 3, 1, 24, 24)),
                                           ("sd21", (1, 3, 1, 64, 96))])
def test_ragged_shapes_vs_oracle(variant, shape):
    """Edge shapes the reference accepts (single frame, sizes that are not multiples of the tile / of 16, batch > 1,
    odd down-sampled extents) against the fp32 oracle computed on the spot (width-32 models, no tiling)."""
    wrap = dict(tile_spatial_size=None, en_de_n_frames_a_time=None)
    case = dict(variant=variant, ch=32, wrap=wrap)
    m, cfg, sd = _build(case, torch.float16)
    x = O.synthetic_video(shape, 11)
    with torch.no_grad():
        opost = O.encode(x, sd, cfg)
        orec = O.decode(opost.mode(), sd, cfg)
    post = m.encode(x.half().cuda()).latent_dist
    rec = m.decode(post.mode()).sample
    assert post.parameters.shape == opost.parameters.shape and rec.shape == orec.shape
    em = (post.parameters.float().cpu() - opost.parameters).abs()
    er = (rec.float().cpu() - orec).abs()
    assert em.max().item() < 3e-2 and em.mean().item() < 3e-3, (em.max().item(), em.mean().item())
    assert er.max().item() < 8e-2 and er.mean().item() < 8e-3, (er.max().item(), er.mean().item())


@pytest.mark.parametrize("name", ["sd21_w32_tiled", "sd3_w32_plain"])
def test_cuda_graph_replay_is_bit_identical(name):
    """enable_cuda_graphs(): captured replay == eager launches, also for a second input through the same graphs."""
    case = CASES[name]
    m, cfg, sd = _build(case, torch.float16)
    xs = [O.synthetic_video(case["shape"], MANIFEST["input_seed"] + i).half().cuda() for i in range(2)]
    eager = []
    for x in xs:
        post = m.encode(x).latent_dist
        eager.append((post.parameters.clone(), m.decode(post.mode()).sample.clone()))
    m.enable_cuda_graphs(True)
    for rep in range(2):                      # first pass captures, second replays
        for x, (mom, rec) in zip(xs, eager):
            post = m.encode(x).latent_dist
            got = m.decode(post.mode()).sample
            assert torch.equal(post.parameters, mom) and torch.equal(got, rec)
    assert len(m._graph_cache) >= 2
    m.enable_cuda_graphs(False)
    assert not m._graph_cache


def test_compat_import_paths():
    """The reference scripts' import lines (cvvae_inference_video.py:1, pipelines/pipeline_stable_diffusion.py:41) resolve
    to this engine through compat/ and run: a tiny encode / decode(num_frames=1) on the GPU."""
    import importlib
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, os.path.join(root, "compat"))
    try:
        for n in [n for n in sys.modules if n == "models" or n.startswith("models.") or n.startswith("diffuser_engine")]:
            del sys.modules[n]
        A = importlib.import_module("models.modeling_vae").CVVAEModel
        Bm = importlib.import_module("diffuser_engine.models.modeling_vae").CVVAEModel
        import cvvae_b200
        assert A is cvvae_b200.CVVAEModel and Bm is cvvae_b200.CVVAEModel
        case = CASES["sd21_w32_image"]
        m, cfg, sd = _build(case, torch.float16)
        assert type(m) is A
        x = O.synthetic_video(case["shape"], MANIFEST["input_seed"]).half().cuda()
        lat = m.encode(x).latent_dist.sample(generator=torch.Generator().manual_seed(3))     # CPU generator, as pipelines pass
        z4 = lat.permute(0, 2, 1, 3, 4).reshape(-1, lat.shape[1], *lat.shape[3:]) * m.config.scaling_factor
        img = m.decode(z4 / m.config.scaling_factor, num_frames=1).sample                     # pipeline_stable_diffusion.py:1046
        assert img.shape == x.shape and torch.isfinite(img).all()
    finally:
        sys.path.remove(os.path.join(root, "compat"))
