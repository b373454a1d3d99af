"""Generate the committed golden fixtures by running the UNMODIFIED reference.

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden.py

The reference modules are imported verbatim from /root/reference through
``tests/ref_shim`` (stubs for the absent diffusers / xformers symbols).  Weights
come from ``oracle.cvvae_oracle.make_state_dict`` (per-key seeded, so they can
be regenerated anywhere) and are loaded into the reference with
``load_state_dict(strict=True)``; inputs from ``synthetic_video``.  Only the
reference OUTPUTS are stored (fp32 .npz, large outputs as a fixed sample, see
``tests/golden_data.py``) plus a manifest describing each case.
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import golden_data  # noqa: E402
import ref_shim  # noqa: E402

ref_shim.install()
from models.modeling_vae import CVVAEModel, CVVAESD3Model  # noqa: E402  (reference, verbatim)

from oracle import cvvae_oracle as O  # noqa: E402

CASES = [
    # name, variant, ch, wrapper kwargs, input shape, seeds
    dict(name="sd21_w32_plain", variant="sd21", ch=32, wrap=dict(tile_spatial_size=None, en_de_n_frames_a_time=None),
         shape=(1, 3, 9, 64, 64)),
    dict(name="sd21_w32_tiled", variant="sd21", ch=32, wrap=dict(tile_spatial_size=72, en_de_n_frames_a_time=4),
         shape=(1, 3, 9, 104, 120)),
    dict(name="sd21_w128_plain", variant="sd21", ch=128, wrap=dict(tile_spatial_size=None, en_de_n_frames_a_time=None),
         shape=(1, 3, 5, 32, 32)),
    dict(name="sd21_w32_image", variant="sd21", ch=32, wrap=dict(tile_spatial_size=None, en_de_n_frames_a_time=None),
         shape=(2, 3, 1, 32, 48)),
    # 4-D call convention of the wrappers: (b t) c h w in, num_video_frames / num_latent_frames regrouping, 4-D out
    dict(name="sd21_w32_frames4d", variant="sd21", ch=32,
         wrap=dict(tile_spatial_size=None, en_de_n_frames_a_time=4, num_video_frames=5, reshape_x_dim_to_4=True),
         shape=(10, 3, 32, 40)),
    dict(name="sd3_w32_plain", variant="sd3", ch=32, wrap=dict(tile_spatial_size=None, en_de_n_frames_a_time=None),
         shape=(1, 3, 9, 64, 64)),
    dict(name="sd3_w32_tiled", variant="sd3", ch=32, wrap=dict(tile_spatial_size=72, en_de_n_frames_a_time=4),
         shape=(1, 3, 9, 104, 120)),
    dict(name="sd3_w128_plain", variant="sd3", ch=128, wrap=dict(tile_spatial_size=None, en_de_n_frames_a_time=None),
         shape=(1, 3, 5, 32, 32)),
    # full-width models on inputs large enough for a non-trivial mid-block (attention over 8 x 8 = 64 tokens, 3 latent
    # frames) and, tiled + chunked, for the whole wrapper (2 chunks x 2 x 2 ragged tiles of <= 64 px, blends both ways)
    dict(name="sd21_w128_mid", variant="sd21", ch=128, wrap=dict(tile_spatial_size=None, en_de_n_frames_a_time=None),
         shape=(1, 3, 9, 64, 64)),
    dict(name="sd3_w128_mid", variant="sd3", ch=128, wrap=dict(tile_spatial_size=None, en_de_n_frames_a_time=None),
         shape=(1, 3, 9, 64, 64)),
    dict(name="sd21_w128_tiled", variant="sd21", ch=128, wrap=dict(tile_spatial_size=64, en_de_n_frames_a_time=4),
         shape=(1, 3, 9, 96, 112)),
]
WEIGHT_SEED = 1234
INPUT_SEED = 0


def build_reference(case):
    widths = [case["ch"] * m for m in (1, 2, 4, 4)]
    if case["variant"] == "sd21":
        m = CVVAEModel(ch=case["ch"], **case["wrap"])
        cfg = O.VAEConfig(variant="sd21", ch=case["ch"], **case["wrap"])
    else:
        m = CVVAESD3Model(block_out_channels=widths, **case["wrap"])
        cfg = O.VAEConfig(variant="sd3", ch=case["ch"], z_channels=16, **case["wrap"])
    sd = O.make_state_dict(cfg, WEIGHT_SEED)
    m.load_state_dict(sd, strict=True)
    return m.eval().requires_grad_(False), cfg, sd


def main():
    manifest = {"weight_seed": WEIGHT_SEED, "input_seed": INPUT_SEED, "cases": []}
    for i, case in enumerate(CASES):
        m, cfg, sd = build_reference(case)
        x = O.synthetic_video(case["shape"], INPUT_SEED)
        with torch.no_grad():
            post = m.encode(x).latent_dist
            moments = post.parameters
            z = post.mode()
            rec = m.decode(z).sample
            arrays = dict(moments=moments.numpy(), recon=rec.numpy())
            if case["name"].endswith("_image"):
                # 4-D path of the SD pipelines: decode(latents, num_frames=1) (pipeline_stable_diffusion.py:1046)
                z4 = z.permute(0, 2, 1, 3, 4).reshape(-1, *z.shape[1:2], *z.shape[3:])
                arrays["recon_4d"] = m.decode(z4, num_frames=1).sample.numpy()
            if case["name"].endswith("_frames4d"):
                # 4-D latents regrouped with the model's own num_latent_frames (modeling_vae.py:308-309)
                z4 = z.permute(0, 2, 1, 3, 4).reshape(-1, *z.shape[1:2], *z.shape[3:])
                arrays["recon_4dlat"] = m.decode(z4).sample.numpy()
        np.savez(os.path.join(HERE, case["name"] + ".npz"), **golden_data.shrink(arrays, seed=i))
        shapes = {k: list(v) for k, v in O.param_shapes(cfg).items()}
        entry = dict(case)
        entry["shape"] = list(case["shape"])
        entry["n_params"] = int(sum(np.prod(s) for s in shapes.values()))
        entry["n_tensors"] = len(shapes)
        entry["outputs"] = {k: list(v.shape) for k, v in arrays.items()}
        manifest["cases"].append(entry)
        print(case["name"], entry["outputs"], "params", entry["n_params"])
    # key schema of the default (full width) models, straight from the reference modules
    for variant, cls in (("sd21", CVVAEModel), ("sd3", CVVAESD3Model)):
        with torch.device("meta"):
            m = cls()
        manifest[f"state_dict_schema_{variant}"] = {k: list(v.shape) for k, v in m.state_dict().items()}
    with open(os.path.join(HERE, "manifest.json"), "w") as f:
        json.dump(manifest, f, indent=1)


if __name__ == "__main__":
    main()
