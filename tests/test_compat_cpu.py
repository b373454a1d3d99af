"""Zero-edit drop-in (north_star: "cvvae_inference_video.py and the SD pipelines call it unchanged").

With `compat/` in front on sys.path, the original project's `from models.modeling_vae import CVVAEModel` resolves to
this package.  The engine runs on the CPU test double of the operator set (tests/fake_ops.py); what is checked here is
the host-side contract the inference script relies on: from_pretrained(path, subfolder=, torch_dtype=), requires_grad_,
the fp16 input convention, encode(...).latent_dist.sample(), decode(...).sample, shapes and value range.
"""
import importlib
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture
def compat_path(monkeypatch):
    monkeypatch.syspath_prepend(os.path.join(ROOT, "compat"))
    for name in [n for n in sys.modules if n == "models" or n.startswith("models.") or n.startswith("diffuser_engine")]:
        monkeypatch.delitem(sys.modules, name)
    yield


def test_compat_paths_resolve_to_the_engine(compat_path):
    import cvvae_b200
    m1 = importlib.import_module("models.modeling_vae")
    m2 = importlib.import_module("diffuser_engine.models.modeling_vae")
    assert m1.CVVAEModel is cvvae_b200.CVVAEModel and m1.CVVAESD3Model is cvvae_b200.CVVAESD3Model
    assert m2.CVVAEModel is cvvae_b200.CVVAEModel


def test_video_inference_flow_through_compat(compat_path, monkeypatch, tmp_path):
    """What the video inference script of the original project does with the model, self-contained: load a checkpoint
    folder through the compat import path, encode a uint8 clip scaled to [-1, 1] in fp16, sample the posterior, decode,
    and map back to uint8 frames."""
    from fake_ops import FakeOps
    from oracle import cvvae_oracle as O
    import cvvae_b200
    wrap = dict(tile_spatial_size=72, en_de_n_frames_a_time=4)
    m = cvvae_b200.CVVAEModel(ch=32, **wrap)
    m.load_state_dict(O.make_state_dict(O.VAEConfig(variant="sd21", ch=32, **wrap), 1234))
    m.save_pretrained(str(tmp_path / "ckpt" / "vae3d"))
    monkeypatch.setattr(cvvae_b200.modeling_vae._CVVAEBase, "_ops_factory", FakeOps)
    CVVAEModel = importlib.import_module("models.modeling_vae").CVVAEModel
    vae = CVVAEModel.from_pretrained(str(tmp_path / "ckpt"), subfolder="vae3d", torch_dtype=torch.float16)
    vae.requires_grad_(False)
    assert type(vae) is cvvae_b200.CVVAEModel and vae.dtype == torch.float16
    assert all(not p.requires_grad for p in vae.parameters())
    for k, v in m.state_dict().items():
        assert torch.equal(vae.state_dict()[k], v.half()), k
    g = torch.Generator().manual_seed(3)
    frames = torch.randint(0, 256, (7, 80, 104, 3), generator=g, dtype=torch.uint8)    # t h w c, as a video reader gives
    n = 1 + (frames.shape[0] - 1) // 4 * 4                                              # whole latent frames only: 5
    video = frames[:n].permute(3, 0, 1, 2).unsqueeze(0).half() / 127.5 - 1.0           # 1 c t h w in [-1, 1]
    torch.manual_seed(0)
    latent = vae.encode(video).latent_dist.sample()
    assert latent.shape == (1, 4, 2, 10, 13) and latent.dtype == torch.float16
    rec = vae.decode(latent).sample
    assert rec.shape == video.shape and rec.dtype == torch.float16 and torch.isfinite(rec).all()
    out = ((rec[0].permute(1, 2, 3, 0).clamp(-1.0, 1.0) + 1.0) * 127.5).to(torch.uint8)
    assert tuple(out.shape) == (5, 80, 104, 3)
    assert 0 < out.float().mean().item() < 255

