"""Pin the CPU oracle against outputs of the reference itself (tests/golden/*.npz).

The fixtures were produced by tests/golden/make_golden.py from the unmodified
reference modules; here the oracle must reproduce them from the same seeds
(at the stored sample of positions for the larger outputs, tests/golden_data.py).
"""
import json
import os

import numpy as np
import pytest
import torch

from golden_data import stored
from oracle import cvvae_oracle as O

GOLD = os.path.join(os.path.dirname(__file__), "golden")
with open(os.path.join(GOLD, "manifest.json")) as f:
    MANIFEST = json.load(f)
CASES = {c["name"]: c for c in MANIFEST["cases"]}


def _cfg(case):
    extra = dict(z_channels=16) if case["variant"] == "sd3" else {}
    return O.VAEConfig(variant=case["variant"], ch=case["ch"], **extra, **case["wrap"])


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_matches_reference_outputs(name):
    case = CASES[name]
    cfg = _cfg(case)
    sd = O.make_state_dict(cfg, MANIFEST["weight_seed"])
    assert len(sd) == case["n_tensors"]
    assert sum(v.numel() for v in sd.values()) == case["n_params"]
    gold = np.load(os.path.join(GOLD, name + ".npz"))
    x = O.synthetic_video(case["shape"], MANIFEST["input_seed"])
    with torch.no_grad():
        post = O.encode(x, sd, cfg)
        rec = O.decode(post.mode(), sd, cfg)
    # same ATen kernels in the same order on CPU fp32 -> expected bit-exact; allow 1e-6 for
    # thread-count dependent reductions on a different host.
    assert list(rec.shape) == case["outputs"]["recon"]
    np.testing.assert_allclose(post.parameters.numpy(), gold["moments"], rtol=0, atol=2e-6)
    np.testing.assert_allclose(stored(gold, "recon", rec.numpy()), gold["recon"], rtol=0, atol=2e-6)
    if "recon_4d" in gold.files:
        z = post.mode()
        z4 = z.permute(0, 2, 1, 3, 4).reshape(-1, z.shape[1], *z.shape[3:])
        rec4 = O.decode(z4, sd, cfg, num_frames=1)
        np.testing.assert_allclose(rec4.numpy(), gold["recon_4d"], rtol=0, atol=2e-6)
    if "recon_4dlat" in gold.files:
        z = post.mode()
        z4 = z.permute(0, 2, 1, 3, 4).reshape(-1, z.shape[1], *z.shape[3:])
        np.testing.assert_allclose(O.decode(z4, sd, cfg).numpy(), gold["recon_4dlat"], rtol=0, atol=2e-6)


@pytest.mark.parametrize("variant", ["sd21", "sd3"])
def test_state_dict_schema_matches_reference(variant):
    """Key names + shapes of the default full-width models, as the reference modules expose them."""
    schema = MANIFEST[f"state_dict_schema_{variant}"]
    cfg = O.VAEConfig(variant=variant, z_channels=4 if variant == "sd21" else 16)
    mine = {k: list(v) for k, v in O.param_shapes(cfg).items()}
    assert mine == schema


def test_tile_geometry_rounding():
    g = O.TileGeometry.of(O.VAEConfig())
    assert (g.encode_chunk, g.decode_chunk, g.pixel_tile, g.latent_tile) == (16, 4, 576, 72)
    assert round(576 * (1 - 0.2222)) == 448 and round(72 * 0.2222) == 16 and round(576 * 0.2222) == 128
