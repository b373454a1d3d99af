"""GPU parity of every C-ABI entry point against its written-down semantics (tests/fake_ops.py, fp32 torch).

Tolerance for 16-bit outputs: the kernels accumulate in fp32 and round once, so |err| <= ~2^-11 |y| (fp16) /
2^-8 |y| (bf16) plus accumulation-order noise -> rtol 1e-3 / atol 1e-4 for fp16 as BASELINE.json's north_star
states (bf16: rtol 8e-3).  Integer/data-movement kernels are bit-exact.
"""
import json
import os

import pytest
import torch

from fake_ops import PAD_REPLICATE, PAD_ZERO, FakeOps

pytestmark = pytest.mark.gpu
DEV = "cuda"
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")


def _ops():
    from cvvae_b200.ops import CudaOps
    return CudaOps()


def _tol(dtype):
    return dict(rtol=1e-3, atol=1e-4) if dtype == torch.float16 else dict(rtol=8e-3, atol=1e-3)


def _rand(shape, dtype, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return ((torch.rand(shape, generator=g) * 2 - 1) * scale).to(dtype).to(DEV)


def _assert_close(got, want, rtol, atol, tag):
    """torch.testing.assert_close with a record of the worst offenders (gpurun_out/tol_<tag>.json) for diagnosis."""
    err = (got - want).abs()
    lim = atol + rtol * want.abs()
    bad = err > lim
    rec = {"rtol": rtol, "atol": atol, "max_abs_err": err.max().item(), "violations": int(bad.sum().item()), "numel": got.numel(),
           "max_err_over_limit": (err / lim).max().item()}
    if bad.any():
        idx = torch.nonzero(bad.flatten())[:8, 0]
        rec["worst"] = [{"i": int(i), "got": got.flatten()[i].item(), "want": want.flatten()[i].item()} for i in idx]
    _dump(f"tol_{tag}.json", rec)
    torch.testing.assert_close(got, want, rtol=rtol, atol=atol)


def _dump(name, obj):
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, name), "w") as f:
        json.dump(obj, f, indent=1)


# ----------------------------------------------------------------------------------------------------------
def test_library_loads_and_counts_launches():
    ops = _ops()
    n0 = ops.launch_count()
    x = _rand((1, 1, 4, 4, 8), torch.float16, 0)
    y = torch.empty_like(x)
    ops.copy(x, y)
    torch.cuda.synchronize()
    assert torch.equal(x, y) and ops.launch_count() == n0 + 1


def test_umma_descriptor_probe():
    """A 128xNx64 UMMA on a TMA-written SWIZZLE_128B slab.  Aligned starts (shift 0, 8) must be exact; what the
    hardware does for unaligned row shifts (with/without the base_offset field) is recorded for the next
    conv_tc revision (gpurun_out/probe_umma.json)."""
    import ctypes as C

    from cvvae_b200 import _lib as L
    lib = L.load()
    n = 64
    a = _rand((320, 64), torch.float16, 1)
    b = _rand((n, 64), torch.float16, 2)
    res = {}
    for sbo in (8, 16, 10, 12):
        for shift in (0, 8, 16, 1, 2, 3, 10, 17):
            for mode in (0, 1):
                out = torch.zeros((128, n), dtype=torch.float32, device=DEV)
                L.check(lib.cvvae_probe_umma_shift(a.data_ptr(), b.data_ptr(), out.data_ptr(), n, shift, mode, sbo,
                                                   torch.cuda.current_stream().cuda_stream), "probe")
                torch.cuda.synchronize()
                rows = torch.arange(128, device=DEV)
                src = (rows // 8) * sbo + rows % 8 + shift      # 8-row groups `sbo` slab rows apart
                want = a[src].float() @ b.float().t()
                err = (out - want).abs().max().item()
                res[f"sbo{sbo}_shift{shift}_mode{mode}"] = err
    _dump("probe_umma.json", res)
    print(res)
    # what conv_tc relies on: aligned starts with dense groups (all kernels), and - for the wide-slab persistent kernel -
    # groups 10 slab rows apart (8 + KW - 1 positions per image row) from starts shifted by kh * 10 + kw rows
    for sbo, shifts in ((8, (0, 8, 16)), (16, (0, 8, 16)), (10, (0, 1, 2, 10, 17)), (12, (0, 1, 2))):
        for shift in shifts:
            assert res[f"sbo{sbo}_shift{shift}_mode0"] < 1e-3, res


CONV_CASES = {
    # name: (x shape [B,T,H,W,Ci], Co, kernel, stride, pads, pad_t, pad_hw, up_time, extras)
    "gemm_flat": ((1, 1, 1, 300, 64), 128, (1, 1, 1), (1, 1, 1), ((0, 0), (0, 0), (0, 0)), PAD_ZERO, PAD_ZERO, 1, {}),
    "gemm_flat_big": ((1, 1, 1, 1500, 512), 512, (1, 1, 1), (1, 1, 1), ((0, 0), (0, 0), (0, 0)), PAD_ZERO, PAD_ZERO, 1, {}),
    "causal333": ((1, 5, 20, 24, 64), 128, (3, 3, 3), (1, 1, 1), ((2, 0), (1, 1), (1, 1)), PAD_REPLICATE, PAD_ZERO, 1, {}),
    "zero333_n256": ((2, 3, 16, 16, 128), 256, (3, 3, 3), (1, 1, 1), ((1, 1), (1, 1), (1, 1)), PAD_ZERO, PAD_ZERO, 1, {}),
    "frame133_odd": ((1, 2, 33, 17, 128), 128, (1, 3, 3), (1, 1, 1), ((0, 0), (1, 1), (1, 1)), PAD_ZERO, PAD_ZERO, 1, {}),
    "down222": ((1, 5, 32, 32, 128), 128, (3, 3, 3), (2, 2, 2), ((2, 0), (0, 1), (0, 1)), PAD_REPLICATE, PAD_ZERO, 1, {}),
    "down122": ((1, 3, 30, 26, 64), 64, (3, 3, 3), (1, 2, 2), ((2, 0), (0, 1), (0, 1)), PAD_REPLICATE, PAD_ZERO, 1, {}),
    "uptime": ((1, 3, 16, 16, 64), 128, (3, 3, 3), (1, 1, 1), ((1, 1), (1, 1), (1, 1)), PAD_REPLICATE, PAD_ZERO, 2, {}),
    "cout8_ncdhw": ((1, 2, 12, 12, 128), 8, (3, 3, 3), (1, 1, 1), ((2, 0), (1, 1), (1, 1)), PAD_REPLICATE, PAD_ZERO, 1,
                    {"ncdhw_out": True}),
    "cin32": ((1, 2, 16, 16, 32), 32, (3, 3, 3), (1, 1, 1), ((1, 1), (1, 1), (1, 1)), PAD_ZERO, PAD_ZERO, 1, {}),
    "res_bias_alpha": ((1, 2, 16, 24, 64), 128, (1, 3, 3), (1, 1, 1), ((0, 0), (1, 1), (1, 1)), PAD_ZERO, PAD_ZERO, 1,
                       {"residual": True, "alpha": 0.5}),
    "wide512": ((1, 2, 24, 24, 512), 512, (3, 3, 3), (1, 1, 1), ((1, 1), (1, 1), (1, 1)), PAD_ZERO, PAD_ZERO, 1, {}),
    "phase322_up": ((1, 3, 16, 24, 64), 128, (3, 2, 2), (1, 1, 1), ((1, 1), (1, 0), (0, 1)), PAD_REPLICATE, PAD_ZERO, 2,
                    {"lattice_out": (0, 1)}),
    "phase322": ((1, 2, 20, 16, 128), 256, (3, 2, 2), (1, 1, 1), ((1, 1), (0, 1), (1, 0)), PAD_REPLICATE, PAD_ZERO, 1,
                 {"lattice_out": (1, 0)}),
    # tall problems: pair_n256_odd / pair_n512 / pair_phase_up take CTA pairs (cta_group::2) along W with an odd tile count
    # (residual, interleaved); pair_n128 the persistent wide-slab kernel, pair_down the persistent kernel without wide slabs
    # (strided), pair_cout32 the single-CTA kernel.  Pairs along H: conv1x1_spatial
    "pair_n128": ((1, 3, 80, 48, 64), 128, (3, 3, 3), (1, 1, 1), ((2, 0), (1, 1), (1, 1)), PAD_REPLICATE, PAD_ZERO, 1, {}),
    "pair_n256_odd": ((1, 2, 72, 40, 128), 256, (3, 3, 3), (1, 1, 1), ((1, 1), (1, 1), (1, 1)), PAD_ZERO, PAD_ZERO, 1,
                      {"residual": True}),
    "pair_n512": ((1, 2, 50, 33, 256), 512, (1, 3, 3), (1, 1, 1), ((0, 0), (1, 1), (1, 1)), PAD_ZERO, PAD_ZERO, 1, {}),
    "pair_down": ((1, 5, 130, 66, 128), 128, (3, 3, 3), (2, 2, 2), ((2, 0), (0, 1), (0, 1)), PAD_REPLICATE, PAD_ZERO, 1, {}),
    "pair_phase_up": ((1, 3, 70, 24, 128), 256, (3, 2, 2), (1, 1, 1), ((1, 1), (1, 0), (0, 1)), PAD_REPLICATE, PAD_ZERO, 2,
                      {"lattice_out": (0, 1)}),
    "pair_cout32": ((1, 2, 90, 20, 64), 32, (3, 3, 3), (1, 1, 1), ((1, 1), (1, 1), (1, 1)), PAD_ZERO, PAD_ZERO, 1, {}),
    # fused 1x1 shortcut (K4): pair kernel (Cout 256 / 512), wide-slab persistent kernel (Cout 128), single-CTA kernel (Cout 64)
    "sc_pair_n256": ((2, 2, 40, 40, 256), 256, (1, 3, 3), (1, 1, 1), ((0, 0), (1, 1), (1, 1)), PAD_ZERO, PAD_ZERO, 1, {"shortcut": 128}),
    "sc_pair_n512_333": ((1, 3, 36, 24, 128), 512, (3, 3, 3), (1, 1, 1), ((2, 0), (1, 1), (1, 1)), PAD_REPLICATE, PAD_ZERO, 1,
                         {"shortcut": 256}),
    "sc_wide_n128": ((2, 3, 70, 44, 128), 128, (1, 3, 3), (1, 1, 1), ((0, 0), (1, 1), (1, 1)), PAD_ZERO, PAD_ZERO, 1, {"shortcut": 256}),
    "sc_wide_n128_333": ((1, 3, 33, 21, 64), 128, (3, 3, 3), (1, 1, 1), ((1, 1), (1, 1), (1, 1)), PAD_ZERO, PAD_ZERO, 1, {"shortcut": 72}),
    "sc_single_n64": ((1, 2, 20, 28, 64), 64, (1, 3, 3), (1, 1, 1), ((0, 0), (1, 1), (1, 1)), PAD_ZERO, PAD_ZERO, 1, {"shortcut": 32}),
    "conv1x1_spatial": ((1, 2, 20, 20, 128), 256, (1, 1, 1), (1, 1, 1), ((0, 0), (0, 0), (0, 0)), PAD_ZERO, PAD_ZERO, 1,
                        {"strided_in": True}),
}


def _run_conv(ops, fake, case, dtype, force):
    xs, Co, kernel, stride, pads, pad_t, pad_hw, up_time, ex = case
    B, T, H, W, Ci = xs
    taps = kernel[0] * kernel[1] * kernel[2]
    x = _rand(xs, dtype, 3)
    if ex.get("strided_in"):
        big = _rand((B, T, H + 2, W + 2, Ci), dtype, 33)
        big[:, :, 1:-1, 1:-1] = x
        x = big[:, :, 1:-1, 1:-1]
    w = _rand((taps, Co, Ci), dtype, 4, scale=(taps * Ci) ** -0.5 * 2)
    bias = _rand((Co,), torch.float32, 5, 0.3)
    (tl, th), (hl, hh), (wl, wh) = pads
    To = (T + tl + th - kernel[0]) // stride[0] + 1
    Ho = (H + hl + hh - kernel[1]) // stride[1] + 1
    Wo = (W + wl + wh - kernel[2]) // stride[2] + 1
    yshape = (B, 2 * To - 1, Ho, Wo, Co // 2) if up_time == 2 else (B, To, Ho, Wo, Co)

    def mk_out():
        if ex.get("lattice_out"):  # one (ph::2, pw::2) lattice of a 2x larger tensor (folded up-sample phases)
            ph, pw = ex["lattice_out"]
            big = torch.zeros((yshape[0], yshape[1], 2 * yshape[2], 2 * yshape[3], yshape[4]), dtype=dtype, device=DEV)
            return big[:, :, ph::2, pw::2, :]
        if ex.get("ncdhw_out"):
            return torch.zeros((yshape[0], yshape[4], yshape[1], yshape[2], yshape[3]), dtype=dtype, device=DEV).permute(0, 2, 3, 4, 1)
        return torch.zeros(yshape, dtype=dtype, device=DEV)

    residual = _rand(yshape, dtype, 6) if ex.get("residual") else None
    kw = dict(kernel=kernel, stride=stride, offset=(-tl, -hl, -wl), pad_t=pad_t, pad_hw=pad_hw, up_time=up_time,
              residual=residual, alpha=ex.get("alpha", 1.0))
    if ex.get("shortcut"):
        c2 = ex["shortcut"]
        kw["sc_x"] = _rand(yshape[:4] + (c2,), dtype, 7)
        kw["sc_w"] = _rand((Co, c2), dtype, 8, scale=c2 ** -0.5)
    got = ops.conv(x, w, bias, out=mk_out(), force=force, **kw)
    want = fake.conv(x, w, bias, out=torch.zeros(yshape, dtype=torch.float32, device=DEV),
                     **{**kw, "residual": residual})
    torch.cuda.synchronize()
    return got, want


@pytest.mark.parametrize("name", sorted(CONV_CASES))
def test_conv_tc_matches_spec(name):
    ops, fake = _ops(), FakeOps()
    got, want = _run_conv(ops, fake, CONV_CASES[name], torch.float16, "tc")
    torch.testing.assert_close(got.float(), want, **_tol(torch.float16))


@pytest.mark.parametrize("name", ["causal333", "down222", "uptime", "cout8_ncdhw", "res_bias_alpha"])
def test_conv_direct_matches_spec(name):
    ops, fake = _ops(), FakeOps()
    got, want = _run_conv(ops, fake, CONV_CASES[name], torch.float16, "direct")
    torch.testing.assert_close(got.float(), want, **_tol(torch.float16))


def test_conv_tc_bf16():
    ops, fake = _ops(), FakeOps()
    got, want = _run_conv(ops, fake, CONV_CASES["causal333"], torch.bfloat16, "tc")
    torch.testing.assert_close(got.float(), want, **_tol(torch.bfloat16))


def test_conv_direct_network_inputs():
    """3-channel NCDHW video read in place (conv_in) with zero and replicate H/W padding."""
    ops, fake = _ops(), FakeOps()
    x_ncdhw = _rand((1, 3, 5, 20, 24), torch.float16, 7)
    x = x_ncdhw.permute(0, 2, 3, 4, 1)
    w = _rand((27, 128, 3), torch.float16, 8, 0.2)
    b = _rand((128,), torch.float32, 9, 0.1)
    for pad_hw in (PAD_ZERO, PAD_REPLICATE):
        kw = dict(kernel=(3, 3, 3), offset=(-2, -1, -1), pad_t=PAD_REPLICATE, pad_hw=pad_hw)
        got = ops.conv(x, w, b, out=torch.zeros((1, 5, 20, 24, 128), dtype=torch.float16, device=DEV), **kw)
        want = fake.conv(x, w, b, out=torch.zeros((1, 5, 20, 24, 128), dtype=torch.float32, device=DEV), **kw)
        torch.testing.assert_close(got.float(), want, **_tol(torch.float16))


def test_conv_attention_style_gemms():
    """fp32 logits with a ragged token count, bias along rows, weight row stride (the three attention GEMMs)."""
    ops, fake = _ops(), FakeOps()
    N, Cc = 1000 + 8 * 3, 128  # multiple of 8 but not of 64/128
    ld = N
    q = _rand((1, 1, 1, N, Cc), torch.float16, 10)
    k = _rand((1, N, Cc), torch.float16, 11)
    S = torch.zeros((N, ld), dtype=torch.float32, device=DEV)
    Sw = torch.zeros((1, 1, 1, N, N), dtype=torch.float32, device=DEV)
    ops.conv(q, k, None, alpha=Cc ** -0.5, out_f32=True, out=S[:, :N][None, None, None], force="tc")
    fake.conv(q, k, None, alpha=Cc ** -0.5, out_f32=True, out=Sw)
    torch.testing.assert_close(S[:, :N], Sw[0, 0, 0], rtol=1e-4, atol=1e-4)
    # v^T = Wv x^T + bv (bias along M)
    wv = _rand((1, 1, 1, Cc, Cc), torch.float16, 12, Cc ** -0.5)
    hn = _rand((1, N, Cc), torch.float16, 13)
    bv = _rand((Cc,), torch.float32, 14, 0.2)
    vT = torch.zeros((Cc, ld), dtype=torch.float16, device=DEV)
    vTw = torch.zeros((1, 1, 1, Cc, N), dtype=torch.float32, device=DEV)
    ops.conv(wv, hn, bv, bias_along_m=True, out=vT[:, :N][None, None, None], force="tc")
    fake.conv(wv, hn, bv, bias_along_m=True, out=vTw)
    torch.testing.assert_close(vT[:, :N].float(), vTw[0, 0, 0], **_tol(torch.float16))
    # O = P v with K = N (ragged K: TMA zero-fill on both operands) and explicit weight row stride
    P = torch.softmax(S[:, :N], dim=-1).half()
    Pp = torch.zeros((N, ld), dtype=torch.float16, device=DEV)
    Pp[:, :N] = P
    out = torch.zeros((1, 1, 1, N, Cc), dtype=torch.float16, device=DEV)
    outw = torch.zeros((1, 1, 1, N, Cc), dtype=torch.float32, device=DEV)
    ops.conv(Pp[:, :N][None, None, None], vT[:, :N].unsqueeze(0), None, w_ld=ld, cout=Cc, out=out, force="tc")
    fake.conv(Pp[:, :N][None, None, None], vT[:, :N].unsqueeze(0), None, cout=Cc, out=outw)
    torch.testing.assert_close(out.float(), outw, **_tol(torch.float16))


@pytest.mark.parametrize("shape,per_frame,silu", [((1, 5, 24, 20, 128), False, True), ((2, 3, 9, 7, 512), True, False),
                                                  ((1, 2, 16, 16, 32), False, True), ((1, 9, 64, 64, 256), False, True)])
def test_groupnorm_matches_spec(shape, per_frame, silu):
    ops, fake = _ops(), FakeOps()
    x = _rand(shape, torch.float16, 20, 2.0) + 0.3
    g = _rand((shape[-1],), torch.float32, 21) * 0.5 + 1.0
    b = _rand((shape[-1],), torch.float32, 22, 0.2)
    got = ops.groupnorm(x, g, b, 32, 1e-5, per_frame=per_frame, silu=silu)
    want = fake.groupnorm(x, g, b, 32, 1e-5, per_frame=per_frame, silu=silu, out=torch.empty(shape, dtype=torch.float32, device=DEV))
    # north_star contract: rtol 1e-3 / atol 1e-4.  One rounding to fp16 costs <= 2^-11 |y| = 4.9e-4 |y| < rtol |y|.
    _assert_close(got.float(), want, 1e-3, 1e-4, f"groupnorm_{shape[-1]}_{int(per_frame)}{int(silu)}")
    # framed (sd3) output + border replicate
    pad, inner = ops.empty_padded(*shape, torch.float16, DEV)
    ops.groupnorm(x, g, b, 32, 1e-6, per_frame=per_frame, silu=silu, out=inner)
    ops.replicate_border(pad)
    ref = torch.nn.functional.pad(inner.permute(0, 4, 1, 2, 3).float(), (1, 1, 1, 1, 0, 0), mode="replicate").permute(0, 2, 3, 4, 1)
    assert torch.equal(pad.float(), ref)


def test_layernorm_softmax_temporal_attention():
    ops, fake = _ops(), FakeOps()
    x = _rand((1, 5, 6, 7, 512), torch.float16, 30, 2.0)
    g = _rand((512,), torch.float32, 31) * 0.5 + 1.0
    b = _rand((512,), torch.float32, 32, 0.2)
    _assert_close(ops.layernorm(x, g, b, 1e-5).float(), fake.layernorm(x.float(), g, b, 1e-5).float(), 1e-3, 1e-4, "layernorm")
    s = _rand((300, 1024), torch.float32, 33, 6.0)
    p = torch.zeros((300, 1024), dtype=torch.float16, device=DEV)
    ops.softmax_rows(s, 1000, p)
    torch.testing.assert_close(p[:, :1000].float(), torch.softmax(s[:, :1000], -1), rtol=1e-3, atol=1e-5)
    q, k, v = (_rand((2, 5, 6, 7, 512), torch.float16, 34 + i) for i in range(3))
    _assert_close(ops.attn_temporal(q, k, v).float(), fake.attn_temporal(q.float(), k.float(), v.float()).float(), 1e-3, 1e-4,
                  "attn_temporal")
    # more latent frames than the register-resident score array holds (en_de_n_frames_a_time=None on a long clip)
    q, k, v = (_rand((1, 40, 3, 4, 64), torch.float16, 37 + i) for i in range(3))
    _assert_close(ops.attn_temporal(q, k, v).float(), fake.attn_temporal(q.float(), k.float(), v.float()).float(), 1e-3, 1e-4,
                  "attn_temporal_T40")


def test_data_movement_is_bit_exact():
    ops, fake = _ops(), FakeOps()
    a = _rand((1, 8, 3, 20, 24), torch.float16, 41)  # NCDHW tiles as the wrapper holds them
    b1 = _rand((1, 8, 3, 20, 24), torch.float16, 42)
    b2 = b1.clone()
    for axis in (0, 1):
        ops.blend(a.permute(0, 2, 3, 4, 1), b1.permute(0, 2, 3, 4, 1), 6, axis)
        fake.blend(a.permute(0, 2, 3, 4, 1), b2.permute(0, 2, 3, 4, 1), 6, axis)
    assert torch.equal(b1, b2)
    w = _rand((128, 64, 3, 3, 3), torch.float16, 43)
    assert torch.equal(ops.pack_weight(w), fake.pack_weight(w))


@pytest.mark.parametrize("name", ["causal333", "frame133_odd", "uptime", "wide512", "res_bias_alpha", "phase322", "cin32",
                                  "pair_n128", "pair_n256_odd", "pair_phase_up", "sc_pair_n256", "sc_wide_n128"])
def test_conv_fused_groupnorm_stats(name):
    """The conv epilogue's (sum, sum^2) per (sample, group) equal those of the tensor it stored."""
    ops, fake = _ops(), FakeOps()
    xs, Co, kernel, stride, pads, pad_t, pad_hw, up_time, ex = CONV_CASES[name]
    yC = Co // 2 if up_time == 2 else Co
    stats = ops.new_stats(xs[0], 32, DEV)
    B, T, H, W, Ci = xs
    taps = kernel[0] * kernel[1] * kernel[2]
    x = _rand(xs, torch.float16, 3)
    w = _rand((taps, Co, Ci), torch.float16, 4, scale=(taps * Ci) ** -0.5 * 2)
    bias = _rand((Co,), torch.float32, 5, 0.3)
    (tl, th), (hl, hh), (wl, wh) = pads
    To = (T + tl + th - kernel[0]) // stride[0] + 1
    Ho = (H + hl + hh - kernel[1]) // stride[1] + 1
    Wo = (W + wl + wh - kernel[2]) // stride[2] + 1
    yshape = (B, 2 * To - 1, Ho, Wo, yC) if up_time == 2 else (B, To, Ho, Wo, Co)
    y = torch.zeros(yshape, dtype=torch.float16, device=DEV)
    skw = {}
    if ex.get("shortcut"):
        skw = dict(sc_x=_rand(yshape[:4] + (ex["shortcut"],), torch.float16, 7), sc_w=_rand((Co, ex["shortcut"]), torch.float16, 8, scale=0.1))
    ops.conv(x, w, bias, kernel=kernel, stride=stride, offset=(-tl, -hl, -wl), pad_t=pad_t, pad_hw=pad_hw, up_time=up_time,
             out=y, gn_stats=stats, gn_groups=32, **skw)
    torch.cuda.synchronize()
    v = y.double().reshape(B, -1, 32, yC // 32)
    want = torch.stack([v.sum(dim=(1, 3)), (v * v).sum(dim=(1, 3))], dim=-1)
    got = torch.stack([stats[..., 0].double() / 2.0 ** 20, stats[..., 1].double() / 2.0 ** 18], dim=-1)
    torch.testing.assert_close(got, want, rtol=1e-5, atol=2e-2)
    # and GroupNorm fed with them equals GroupNorm computing its own
    g = _rand((yC,), torch.float32, 21) * 0.5 + 1.0
    b = _rand((yC,), torch.float32, 22, 0.2)
    # the two statistics differ only by the accumulation order of fp32 partial sums (relative 1e-6): the normalised
    # outputs may differ by one fp16 rounding flip (2^-10 relative) on a few elements - inside the contract
    _assert_close(ops.groupnorm(y, g, b, 32, 1e-5, stats=stats).float(), ops.groupnorm(y, g, b, 32, 1e-5).float(), 1e-3, 1e-4,
                  f"gn_fused_stats_{name}")


@pytest.mark.parametrize("shape,cout,kt,off_t,pad_t", [((1, 3, 40, 50, 128), 3, 3, -1, PAD_ZERO), ((2, 5, 33, 61, 128), 3, 3, -2, PAD_REPLICATE),
                                                       ((1, 2, 16, 16, 64), 4, 3, -1, PAD_REPLICATE), ((1, 1, 70, 30, 128), 3, 1, 0, PAD_ZERO)])
def test_conv_stacked_matches_spec(shape, cout, kt, off_t, pad_t):
    """Tap-stacked tiny-Cout kernel (decoder conv_out) vs the conv spec, NCDHW scatter output."""
    ops, fake = _ops(), FakeOps()
    B, T, H, W, Ci = shape
    x = _rand(shape, torch.float16, 50)
    w = _rand((kt * 9, cout, Ci), torch.float16, 51, scale=(kt * 9 * Ci) ** -0.5 * 2)
    stk = torch.zeros((kt, 80, Ci), dtype=torch.float16, device=DEV)
    stk[:, :72].view(kt, 9, 8, Ci)[:, :, :cout] = w.view(kt, 9, cout, Ci)
    bias = _rand((cout,), torch.float32, 52, 0.3)
    got = torch.zeros((B, cout, T, H, W), dtype=torch.float16, device=DEV)
    want = torch.zeros((B, T, H, W, cout), dtype=torch.float32, device=DEV)
    ops.conv_stacked(x, stk, bias, kt=kt, cout=cout, offset=(off_t, -1, -1), pad_t=pad_t, out=got.permute(0, 2, 3, 4, 1))
    fake.conv(x, w, bias, kernel=(kt, 3, 3), offset=(off_t, -1, -1), pad_t=pad_t, out=want)
    torch.cuda.synchronize()
    torch.testing.assert_close(got.permute(0, 2, 3, 4, 1).float(), want, **_tol(torch.float16))


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_video_pre_post_processing_bit_exact(dtype):
    """Fused uint8<->16-bit pixel conversion equals the reference script's expressions bit for bit."""
    from cvvae_b200.video_io import frames_to_input, output_to_frames
    g = torch.Generator().manual_seed(60)
    frames = torch.randint(0, 256, (5, 36, 52, 3), generator=g, dtype=torch.uint8).to(DEV)
    frames[0, 0, 0] = torch.tensor([0, 255, 128], dtype=torch.uint8)
    got = frames_to_input(frames, dtype)
    # cvvae_inference_video.py:30-34 runs this on the CPU tensor (true division), before .cuda()
    want = frames.cpu().permute(3, 0, 1, 2).unsqueeze(0).to(dtype) / 127.5 - 1.0
    assert got.dtype == dtype and torch.equal(got.cpu(), want)
    x = (_rand((1, 3, 5, 36, 52), torch.float32, 61, 1.3)).to(dtype)             # includes values outside [-1, 1]
    got8 = output_to_frames(x)
    want8 = ((torch.clamp(x, -1.0, 1.0) + 1.0) * 127.5).to(torch.uint8).squeeze(0).permute(1, 2, 3, 0)  # :47-50
    assert torch.equal(got8, want8)


def test_batched_gemm_flags_match_per_item_calls():
    """CVVAE_CONV_W_PER_BATCH / CVVAE_CONV_X_SHARED (the batched attention products): one launch over F frames must equal
    F single-frame launches BIT FOR BIT (same tile plan per item) and the spec within tolerance."""
    ops, fake = _ops(), FakeOps()
    Fn, N, Cc = 3, 200, 128
    ld = N
    q = _rand((Fn, 1, 1, N, Cc), torch.float16, 70)
    k = _rand((Fn, N, Cc), torch.float16, 71)
    S = torch.zeros((Fn, N, ld), dtype=torch.float32, device=DEV)
    S1 = torch.zeros_like(S)
    ops.conv(q, k, None, alpha=Cc ** -0.5, out_f32=True, w_per_batch=True, cout=N, out=S[:, :, :N].unsqueeze(1).unsqueeze(1))
    for f in range(Fn):
        ops.conv(q[f:f + 1], k[f:f + 1], None, alpha=Cc ** -0.5, out_f32=True, cout=N, out=S1[f, :, :N][None, None, None])
    assert torch.equal(S, S1)
    Sw = torch.zeros((Fn, 1, 1, N, N), dtype=torch.float32, device=DEV)
    fake.conv(q, k, None, alpha=Cc ** -0.5, out_f32=True, w_per_batch=True, cout=N, out=Sw)
    torch.testing.assert_close(S.view(Fn, 1, 1, N, ld), Sw, rtol=1e-4, atol=1e-4)
    # v^T = Wv hn^T + bv with the left operand shared by the frames and the bias along rows
    wv = _rand((1, 1, 1, Cc, Cc), torch.float16, 72, Cc ** -0.5)
    hn = _rand((Fn, N, Cc), torch.float16, 73)
    bv = _rand((Cc,), torch.float32, 74, 0.2)
    vT = torch.zeros((Fn, Cc, ld), dtype=torch.float16, device=DEV)
    vT1 = torch.zeros_like(vT)
    ops.conv(wv, hn, bv, bias_along_m=True, x_shared=True, w_per_batch=True, cout=N, out=vT[:, :, :N].unsqueeze(1).unsqueeze(1))
    for f in range(Fn):
        ops.conv(wv, hn[f:f + 1], bv, bias_along_m=True, cout=N, out=vT1[f, :, :N][None, None, None])
    assert torch.equal(vT, vT1)
    want = torch.zeros((Fn, 1, 1, Cc, N), dtype=torch.float32, device=DEV)
    fake.conv(wv, hn, bv, bias_along_m=True, x_shared=True, w_per_batch=True, cout=N, out=want)
    torch.testing.assert_close(vT.view(Fn, 1, 1, Cc, ld).float(), want, **_tol(torch.float16))
    # O = P v, K = N with an explicit weight row stride
    P = torch.softmax(S, dim=-1).half()
    out = torch.zeros((Fn, 1, 1, N, Cc), dtype=torch.float16, device=DEV)
    out1 = torch.zeros_like(out)
    ops.conv(P[:, :, :N].unsqueeze(1).unsqueeze(1), vT, None, w_ld=ld, cout=Cc, w_per_batch=True, out=out)
    for f in range(Fn):
        ops.conv(P[f, :, :N][None, None, None], vT[f:f + 1], None, w_ld=ld, cout=Cc, out=out1[f:f + 1])
    assert torch.equal(out, out1)


def test_copy_rows_tile_assembly_is_bit_exact():
    """The wrapper's tile assembly copy: W-contiguous NCDHW crops, 128-bit path and the unaligned element path."""
    ops = _ops()
    for (W, w0, ww) in ((64, 0, 48), (64, 8, 56), (61, 3, 40)):
        src = _rand((2, 3, 5, 20, W), torch.float16, 80)
        dst = torch.zeros((2, 3, 7, 30, 96), dtype=torch.float16, device=DEV)
        win = dst[:, :, 2:7, 4:24, 16:16 + ww]
        ops.copy(src[:, :, :, :, w0:w0 + ww].permute(0, 2, 3, 4, 1), win.permute(0, 2, 3, 4, 1))
        want = torch.zeros_like(dst)
        want[:, :, 2:7, 4:24, 16:16 + ww] = src[:, :, :, :, w0:w0 + ww]
        assert torch.equal(dst, want)


def test_groupnorm_statistics_are_batch_invariant():
    """Per-frame statistics of a large frame (more positions than one CTA sweeps): the result for a sample must not depend
    on how many samples share the launch (tile batching and sharding rely on it)."""
    ops = _ops()
    x = _rand((2, 2, 288, 288, 128), torch.float16, 90, 2.0)
    g = _rand((128,), torch.float32, 91) * 0.5 + 1.0
    b = _rand((128,), torch.float32, 92, 0.2)
    for per_frame in (True, False):
        both = ops.groupnorm(x, g, b, 32, 1e-5, per_frame=per_frame)
        one = ops.groupnorm(x[1:2], g, b, 32, 1e-5, per_frame=per_frame)
        assert torch.equal(both[1:2], one)


def test_conv_pair_kernel_stress_is_deterministic():
    """compute-sanitizer racecheck reports hazards in the CTA-pair kernel that we read as remote mbarrier arrivals the
    tool does not model (profiles/r01_sanitizer.txt).  A real race would show up as run-to-run differences: 4000
    back-to-back launches of pair kernels (odd tile counts, residual, fused statistics) under SM contention must all be
    bit-identical to the first one and to the single-CTA kernel's result."""
    ops, fake = _ops(), FakeOps()
    mism = torch.zeros((), dtype=torch.int64, device=DEV)
    for name in ("pair_n256_odd", "pair_n512"):
        xs, Co, kernel, stride, pads, pad_t, pad_hw, up_time, ex = CONV_CASES[name]
        B, T, H, W, Ci = xs
        taps = kernel[0] * kernel[1] * kernel[2]
        x = _rand(xs, torch.float16, 3)
        w = _rand((taps, Co, Ci), torch.float16, 4, scale=(taps * Ci) ** -0.5 * 2)
        bias = _rand((Co,), torch.float32, 5, 0.3)
        (tl, th), (hl, hh), (wl, wh) = pads
        yshape = (B, T + tl + th - kernel[0] + 1, H + hl + hh - kernel[1] + 1, W + wl + wh - kernel[2] + 1, Co)
        res = _rand(yshape, torch.float16, 6) if ex.get("residual") else None
        kw = dict(kernel=kernel, offset=(-tl, -hl, -wl), pad_t=pad_t, pad_hw=pad_hw, residual=res)
        y0 = torch.zeros(yshape, dtype=torch.float16, device=DEV)
        st0 = ops.new_stats(B, 32, DEV)
        ops.conv(x, w, bias, out=y0, gn_stats=st0, gn_groups=32, **kw)
        y = torch.zeros_like(y0)
        st = ops.new_stats(B, 32, DEV)
        for it in range(2000):
            st.zero_()
            ops.conv(x, w, bias, out=y, gn_stats=st, gn_groups=32, **kw)
            mism += (y != y0).any().long() + (st != st0).any().long()
    torch.cuda.synchronize()
    assert mism.item() == 0, f"{mism.item()} of 4000 pair-kernel launches differed from the first"


def test_ops_follow_the_tensor_device():
    """A model on cuda:1 while cuda:0 is current (single-process multi-GPU, diffusers device placement)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ops, fake = _ops(), FakeOps()
    assert torch.cuda.current_device() == 0
    d1 = torch.device("cuda", 1)
    xs, Co = (1, 2, 40, 40, 128), 256
    x = _rand(xs, torch.float16, 3).to(d1)
    w = _rand((27, Co, 128), torch.float16, 4, scale=(27 * 128) ** -0.5 * 2).to(d1)
    bias = _rand((Co,), torch.float32, 5, 0.3).to(d1)
    y = torch.zeros((1, 2, 40, 40, Co), dtype=torch.float16, device=d1)
    kw = dict(kernel=(3, 3, 3), offset=(-1, -1, -1), pad_t=PAD_ZERO, pad_hw=PAD_ZERO)
    ops.conv(x, w, bias, out=y, **kw)
    want = fake.conv(x, w, bias, out=torch.zeros(y.shape, dtype=torch.float32, device=d1), **kw)
    torch.cuda.synchronize(d1)
    torch.testing.assert_close(y.float(), want, **_tol(torch.float16))
    assert torch.cuda.current_device() == 0


@pytest.mark.parametrize("cin,cp,pad_hw", [(3, 32, PAD_ZERO), (3, 32, PAD_REPLICATE), (4, 64, PAD_ZERO)])
def test_pack_taps_hw_is_bit_exact_and_conv_in_matches(cin, cp, pad_hw):
    """Spatial taps -> channels gather of the network-input convs (bit-exact data movement), and the KT x 1 x 1 conv over
    the packed tensor equals the 3x3x3 conv spec on the original NCDHW input."""
    ops, fake = _ops(), FakeOps()
    x_ncdhw = _rand((2, cin, 5, 21, 30), torch.float16, 100)
    x = x_ncdhw.permute(0, 2, 3, 4, 1)
    got = torch.full((2, 5, 21, 30, cp), float("nan"), dtype=torch.float16, device=DEV)
    want = torch.empty_like(got)
    ops.pack_taps_hw(x, got, 3, 3, offset=(-1, -1), pad_hw=pad_hw)
    fake.pack_taps_hw(x, want, 3, 3, offset=(-1, -1), pad_hw=pad_hw)
    assert torch.equal(got, want)
    co = 128
    w5 = _rand((co, cin, 3, 3, 3), torch.float16, 101, 0.2)
    b = _rand((co,), torch.float32, 102, 0.1)
    wp = torch.zeros((3, co, cp), dtype=torch.float16, device=DEV)
    wp[:, :, :9 * cin] = w5.permute(2, 0, 3, 4, 1).reshape(3, co, 9 * cin)
    y = torch.zeros((2, 5, 21, 30, co), dtype=torch.float16, device=DEV)
    ops.conv(got, wp, b, kernel=(3, 1, 1), offset=(-2, 0, 0), pad_t=PAD_REPLICATE, out=y, force="tc")
    ref = fake.conv(x, fake.pack_weight(w5), b, kernel=(3, 3, 3), offset=(-2, -1, -1), pad_t=PAD_REPLICATE, pad_hw=pad_hw,
                    out=torch.zeros(y.shape, dtype=torch.float32, device=DEV))
    torch.testing.assert_close(y.float(), ref, **_tol(torch.float16))


@pytest.mark.parametrize("src,dst", [((90, 120), (72, 96)), ((72, 128), (57, 101)), ((60, 80), (120, 160)), ((720, 1280), (576, 1024))])
def test_gpu_resize_matches_torchvision(src, dst):
    """GPU antialiased bilinear resize of the inference script (transforms.Resize on uint8 frames): within 1 LSB of
    torchvision's CPU result (its 16-bit fixed-point weights deviate from exact arithmetic on < 1 % of the pixels for
    generic ratios and on 3-4 % for exact 2x up-scaling, where a quarter of the exact results are .5 ties), and the fused
    resize+normalise pass equals normalising the resized frames bit for bit."""
    from torchvision import transforms
    from cvvae_b200.video_io import frames_to_input, resize_frames
    g = torch.Generator().manual_seed(70)
    T = 3 if src[0] < 700 else 2
    frames = torch.randint(0, 256, (T, src[0], src[1], 3), generator=g, dtype=torch.uint8)
    want = transforms.Resize(size=dst)(frames.permute(0, 3, 1, 2)).permute(0, 2, 3, 1)       # cvvae_inference_video.py:24-28
    got = resize_frames(frames.to(DEV), dst)
    d = (got.cpu().int() - want.int()).abs()
    assert got.shape == want.shape and d.max().item() <= 1, d.max().item()
    assert (d > 0).float().mean().item() < (0.06 if dst[0] == 2 * src[0] else 0.02)
    fused = frames_to_input(frames.to(DEV), torch.float16, size=dst)
    assert torch.equal(fused, frames_to_input(got, torch.float16))


def test_groupnorm_fixed_point_statistics_at_large_magnitudes():
    """The int64 fixed-point accumulators (sum * 2^20, sum of squares * 2^18; common.cuh) at the magnitudes a trained
    checkpoint could produce: activations of rms ~1.2e3 over a full-resolution chunk-tile (5.6 M positions per group: the
    documented range is |sum| < 8.8e12, sum^2 < 3.5e13) - no overflow, statistics exact to fp64, and the same through the
    convolution epilogue's fused sums."""
    ops = _ops()
    g = torch.Generator().manual_seed(110)
    x = ((torch.rand((1, 17, 576, 576, 32), generator=g) * 2 - 1) * 2000.0 + 300.0).to(torch.float16).to(DEV)
    gam = _rand((32,), torch.float32, 111) * 0.5 + 1.0
    bet = _rand((32,), torch.float32, 112, 0.2)
    got = ops.groupnorm(x, gam, bet, 32, 1e-5, silu=False)
    xd = x.double()
    mean = xd.mean(dim=(1, 2, 3), keepdim=True)
    var = xd.var(dim=(1, 2, 3), unbiased=False, keepdim=True)
    want = ((xd - mean) / torch.sqrt(var + 1e-5) * gam.double() + bet.double()).float()
    _assert_close(got.float(), want, 1e-3, 1e-4, "groupnorm_large_magnitude")
    del xd, want, got
    # conv epilogue: outputs of magnitude ~1e3 (weights scaled up), statistics vs fp64 sums of the stored tensor
    xs = _rand((1, 2, 64, 48, 128), torch.float16, 113)
    w = _rand((9, 128, 128), torch.float16, 114, scale=30.0)
    y = torch.zeros((1, 2, 64, 48, 128), dtype=torch.float16, device=DEV)
    st = ops.new_stats(1, 32, DEV)
    ops.conv(xs, w, None, kernel=(1, 3, 3), offset=(0, -1, -1), out=y, gn_stats=st, gn_groups=32)
    v = y.double().reshape(1, -1, 32, 4)
    assert torch.isfinite(y).all() and y.abs().max().item() > 500
    want_s = torch.stack([v.sum(dim=(1, 3)), (v * v).sum(dim=(1, 3))], dim=-1)
    got_s = torch.stack([st[..., 0].double() / 2.0 ** 20, st[..., 1].double() / 2.0 ** 18], dim=-1)
    torch.testing.assert_close(got_s, want_s, rtol=1e-5, atol=1.0)


def test_fused_shortcut_bf16_and_engine_equivalence():
    """K4 in bf16, and the engine's fused ResnetBlock (shortcut as extra K steps of conv2) against its own unfused form
    (separate 1x1 launch + residual add): same math up to one rounding of the shortcut tensor."""
    ops, fake = _ops(), FakeOps()
    got, want = _run_conv(ops, fake, CONV_CASES["sc_wide_n128"], torch.bfloat16, "tc")
    torch.testing.assert_close(got.float(), want, **_tol(torch.bfloat16))
    from cvvae_b200 import CVVAEModel
    from oracle import cvvae_oracle as O
    wrap = dict(tile_spatial_size=None, en_de_n_frames_a_time=None)
    m = CVVAEModel(ch=64, **wrap)
    m.load_state_dict(O.make_state_dict(O.VAEConfig(variant="sd21", ch=64, **wrap), 1234))
    m = m.half().cuda()
    x = O.synthetic_video((1, 3, 5, 64, 48), 3).half().cuda()
    fused = m.encode(x).latent_dist.parameters.float()
    n_fused = ops.launch_count()
    rec_f = m.decode(fused[:, :4].half()).sample.float()
    m._engine().fuse_shortcut = False
    plain = m.encode(x).latent_dist.parameters.float()
    rec_p = m.decode(plain[:, :4].half()).sample.float()
    assert not torch.equal(fused, plain)                      # different roundings: really two code paths
    assert (fused - plain).abs().max().item() < 2e-2 and (rec_f - rec_p).abs().max().item() < 5e-2
    assert (fused - plain).abs().mean().item() < 1e-3
