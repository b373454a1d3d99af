"""Encoder / Decoder graphs of CV-VAE executed on the hand-written sm_100a kernels.

This is the seam the reference crosses with ``self.encoder(tile)`` / ``self.decoder(tile)``
(models/modeling_vae.py:162,249).  The graphs follow

  sd21:  models/vae_models.py       Encoder.forward :790-823,   Decoder.forward :960-1002
  sd3 :  models/vae_models3d_sd3.py Encoder3D.forward :162-208, Decoder3D.forward :323-388
         with the blocks of models/vae_blocks3d_sd3.py

but nothing of their execution model survives: activations live channels-last ([B,T,H,W,C], 16-bit) from
the first convolution to the last, every padding is folded into convolution coordinates (TMA
out-of-bounds fill, time clamp, or - for the sd3 replicate mode - a 1-position frame kept around the
producer's output), GroupNorm+SiLU is one fused pass, the residual add, the 1x1 shortcut result and
the temporal interleave of the up-sampler are folded into convolution epilogues, and the caller's
NCDHW tensors are read / written in place through strided views (no layout copies).

All arithmetic goes through an ``ops`` backend (``cvvae_b200.ops.CudaOps`` in production).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, Optional, Tuple

import torch

from ._lib import PAD_REPLICATE, PAD_ZERO


@dataclass
class NetConfig:
    variant: str = "sd21"            # "sd21" | "sd3"
    in_channels: int = 3
    out_ch: int = 3
    z_channels: int = 4
    widths: Tuple[int, ...] = (128, 256, 512, 512)
    num_res_blocks: int = 2
    groups: int = 32
    double_z: bool = True
    causal_encoder: bool = True
    causal_decoder: bool = False
    half_3d: bool = True
    encoder_attn_type: str = "vanilla-xformers"
    decoder_attn_type: str = "spatial-temporal-xformer"
    mid_block_add_attention: bool = True

    @property
    def eps(self) -> float:
        return 1e-5 if self.variant == "sd21" else 1e-6

    @property
    def moments_channels(self) -> int:
        return 2 * self.z_channels if self.double_z else self.z_channels


class Act:
    """An activation: logical [B,T,H,W,C] tensor, plus (sd3) the framed buffer it is the interior of, plus - when
    the producing convolution computed them in its epilogue - the GroupNorm sums of its consumer."""
    __slots__ = ("t", "pad", "stats")

    def __init__(self, t: torch.Tensor, pad: Optional[torch.Tensor] = None, stats: Optional[torch.Tensor] = None):
        self.t = t
        self.pad = pad
        self.stats = stats


def prepack_params(state_dict: Dict[str, torch.Tensor], ops, dtype: torch.dtype) -> Dict[str, torch.Tensor]:
    """Weights -> [taps, Cout, Cin] in the compute dtype; biases and norm parameters -> fp32."""
    packed = {}
    for k, v in state_dict.items():
        if k.endswith(".weight") and v.dim() >= 2:
            v = v.detach().to(dtype)
            if k in ("encoder.conv_in.weight", "decoder.conv_in.weight") and v.shape[1] % 8:
                # network inputs have 3 / 4 channels: zero-pad Cin to 8 so the channel-padded channels-last copy of the
                # input (Engine.conv) runs on the tensor-core path; the MMA loop skips the all-zero K steps
                vp = torch.zeros((v.shape[0], (v.shape[1] + 7) // 8 * 8) + tuple(v.shape[2:]), dtype=dtype, device=v.device)
                vp[:, : v.shape[1]] = v
                v = vp
            if ".upsample.conv." in k or ".upsamplers.0.conv." in k:
                # nearest-x2 followed by a 3x3 (H,W) conv == four 2x2 phase convs on the NOT up-sampled input
                # (exact in real arithmetic): output (2i+ph, 2j+pw) reads input rows {i-1,i} (ph=0) or {i,i+1}
                # (ph=1) with the taps that land on the same input pixel pre-summed.  2.25x fewer MACs and no
                # materialised 4x tensor.  Sums are formed in fp32 and rounded once to the compute dtype.
                w32 = v.float()
                for ph in (0, 1):
                    rows = (w32[:, :, :, 0:1], w32[:, :, :, 1:2] + w32[:, :, :, 2:3]) if ph == 0 else \
                           (w32[:, :, :, 0:1] + w32[:, :, :, 1:2], w32[:, :, :, 2:3])
                    wr = torch.cat(rows, dim=3)  # [Co, Ci, 3, 2, 3]
                    for pw in (0, 1):
                        cols = (wr[..., 0:1], wr[..., 1:2] + wr[..., 2:3]) if pw == 0 else \
                               (wr[..., 0:1] + wr[..., 1:2], wr[..., 2:3])
                        wf = torch.cat(cols, dim=4).to(dtype).contiguous()  # [Co, Ci, 3, 2, 2]
                        packed[k[: -len("weight")] + f"phase{ph}{pw}.weight"] = ops.pack_weight(wf)
                continue
            packed[k] = ops.pack_weight(v)
            if k in ("encoder.conv_in.weight", "decoder.conv_in.weight") and v.dim() == 5 and tuple(v.shape[3:]) == (3, 3):
                # network-input convolutions (3 / 4 real channels): the nine spatial taps are packed into the channel axis
                # by cvvae_pack_taps_hw, so the conv runs as KT x 1 x 1 over 9*Cin (<= 64) channels instead of 27 taps
                # of a 95 %-empty 64-channel K block.  Weights [KT][Cout][(kh*3+kw)*Cin + ci], zero-padded to 32 / 64.
                ci_real = state_dict[k].shape[1]
                if 9 * ci_real <= 64:
                    cp = 32 if 9 * ci_real <= 32 else 64
                    w0 = state_dict[k].detach().to(dtype)
                    wp = torch.zeros((w0.shape[2], w0.shape[0], cp), dtype=dtype, device=v.device)
                    wp[:, :, : 9 * ci_real] = w0.permute(2, 0, 3, 4, 1).reshape(w0.shape[2], w0.shape[0], 9 * ci_real)
                    packed[k + ".hwpack"] = wp.contiguous()
            if k == "decoder.conv_out.weight" and v.dim() == 5 and v.shape[0] <= 4 and tuple(v.shape[3:]) == (3, 3):
                # tap-stacked form for the tiny-Cout kernel: [KT][80][Cin], row (kh*3+kw)*8 + c
                co, ci, kt = v.shape[0], v.shape[1], v.shape[2]
                stk = torch.zeros((kt, 80, ci), dtype=dtype, device=v.device)
                stk[:, :72].view(kt, 9, 8, ci)[:, :, :co] = v.permute(2, 3, 4, 0, 1).reshape(kt, 9, co, ci)
                packed[k + ".stk"] = stk
        else:
            packed[k] = v.detach().to(torch.float32).contiguous()
    return packed


def _out_len(n: int, k: int, s: int, lo: int, hi: int) -> int:
    return (n + lo + hi - k) // s + 1


class Engine:
    def __init__(self, cfg: NetConfig, params: Dict[str, torch.Tensor], ops, dtype: torch.dtype):
        self.cfg = cfg
        self.p = params
        self.ops = ops
        self.dtype = dtype
        self.sd3 = cfg.variant == "sd3"
        self.hw_mode = PAD_REPLICATE if self.sd3 else PAD_ZERO
        self._stats_arena = None   # [slots, B, groups, 2] int64, zeroed once per network pass
        self._stats_next = 0
        self.attn_scratch_bytes = 4 << 30  # cap of the fp32 logits buffer of the batched spatial attention
        # 1x1 shortcuts run as extra K steps of conv2 (resblock); inputs _tc_ok rejects take a separate launch + residual add
        self.fuse_shortcut = True

    # ------------------------------------------------------------------ shape arithmetic
    def encoded_frames(self, T: int) -> int:
        """Latent frames the encoder yields for T pixel frames (time stride 2 at the even levels, pads (2,0) / (1,1))."""
        for lvl in range(len(self.cfg.widths) - 1):
            if lvl % 2 == 0:
                T = (T - 1) // 2 + 1
        return T

    def decoded_frames(self, T: int) -> int:
        """Pixel frames the decoder yields for T latent frames (up_time 2 -> 2T-1 at the same levels, mirrored)."""
        L = len(self.cfg.widths)
        for i in range(L - 1):
            lvl = L - 1 - i
            if ((i % 2 == 0) if self.sd3 else (lvl % 2 == 1)):
                T = 2 * T - 1
        return T

    def encoded_hw(self, n: int) -> int:
        """Latent extent of a pixel extent: one stride-2 3-tap conv per level but the last, pads (0,1) (sd21) / (1,1) (sd3)."""
        for _ in range(len(self.cfg.widths) - 1):
            n = (n + (2 if self.sd3 else 1) - 3) // 2 + 1
        return n

    def decoded_hw(self, n: int) -> int:
        return n * 2 ** (len(self.cfg.widths) - 1)

    # ------------------------------------------------------------------ GroupNorm-sum accumulators
    _STATS_SLOTS = 96  # >= convolutions with fused statistics in one encoder / decoder pass (sd21 decoder: 49)

    def _begin_pass(self, B: int, device) -> None:
        """One zeroed accumulator arena per network pass (one fill kernel instead of one per convolution)."""
        self._stats_arena = self.ops.new_stats(self._STATS_SLOTS * B, self.cfg.groups, device).view(
            self._STATS_SLOTS, B, self.cfg.groups, 2)
        self._stats_next = 0

    def new_stats(self, B: int, device) -> torch.Tensor:
        a = self._stats_arena
        if a is None or a.shape[1] != B or a.device != device or self._stats_next >= a.shape[0]:
            return self.ops.new_stats(B, self.cfg.groups, device)
        self._stats_next += 1
        return a[self._stats_next - 1]

    # ------------------------------------------------------------------ primitives
    def _tc_ok(self, x: torch.Tensor) -> bool:
        return x.stride(4) == 1 and x.shape[4] % 8 == 0 and all(s % 8 == 0 for s in x.stride()[:4])

    def _framed(self, a: Act) -> Act:
        """Give `a` a replicate frame (copy into a framed buffer unless it already lives in one)."""
        if a.pad is not None:
            return a
        B, T, H, W, Cc = a.t.shape
        pad, inner = self.ops.empty_padded(B, T, H, W, Cc, a.t.dtype, a.t.device)
        self.ops.copy(a.t, inner)
        self.ops.replicate_border(pad)
        return Act(inner, pad)

    def conv(self, a: Act, name: str, *, kernel, stride=(1, 1, 1), pads, pad_t, pad_hw, up_time=1,
             residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
             weight_key: Optional[str] = None, ref_taps: Optional[int] = None,
             stats: Optional[torch.Tensor] = None, want_stats: bool = False, k_alg: Optional[int] = None,
             shortcut: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]] = None) -> Act:
        """Convolution with the reference's padding expressed as ((t_lo,t_hi),(h_lo,h_hi),(w_lo,w_hi)).

        want_stats: also produce the consumer GroupNorm's (sum, sum^2) per (sample, group) in the epilogue
        (`stats` continues an accumulator across the launches that fill one tensor)."""
        x = a.t
        wkey = weight_key or (name + ".weight")
        w = self.p[wkey]
        b = self.p.get(name + ".bias")
        if shortcut is not None:   # (input [B,T,H,W,C2], matrix [Cout, C2], summed bias): fused as extra K steps
            b = shortcut[2]
        B, T, H, W, _ = x.shape
        (tl, th), (hl, hh), (wl, wh) = pads
        kt, kh, kw = kernel
        hwp = self.p.get(name + ".weight.hwpack") if weight_key is None else None
        if (hwp is not None and not self._tc_ok(x) and (kh, kw) == (3, 3) and tuple(stride[1:]) == (1, 1) and up_time == 1
                and residual is None and hasattr(self.ops, "pack_taps_hw")):
            # network input (3 / 4 channels, NCDHW): spatial taps -> channels in one gather pass, then a KT x 1 x 1
            # convolution on the tensor cores (the single-frame fold below then applies to the time taps as usual)
            Ho, Wo = _out_len(H, kh, 1, hl, hh), _out_len(W, kw, 1, wl, wh)
            xp = self.ops.empty((B, T, Ho, Wo, hwp.shape[2]), x.dtype, x.device)
            self.ops.pack_taps_hw(x, xp, kh, kw, offset=(-hl, -wl), pad_hw=pad_hw)
            return self.conv(Act(xp), name, kernel=(kt, 1, 1), stride=(stride[0], 1, 1), pads=((tl, th), (0, 0), (0, 0)),
                             pad_t=pad_t, pad_hw=PAD_ZERO, out=out, weight_key=name + ".weight.hwpack", stats=stats,
                             want_stats=want_stats, k_alg=kt * kh * kw * x.shape[4])
        if T == 1 and kt > 1 and _out_len(1, kt, stride[0], tl, th) == 1:
            # single-frame input (image path, SURVEY 8f row 4): every time tap reads frame 0 (replicate padding) or
            # nothing (zero padding), so the conv is a per-frame one with pre-summed / selected time taps; of an
            # `up_time` conv only the channel half that lands on the kept frame is computed
            w, b = self._single_frame_weights(wkey, name, w, b, kt, kh * kw, tl, pad_t, up_time)
            if ref_taps is None:
                ref_taps = kt * kh * kw
            kernel, stride, pads = (1, kh, kw), (1, stride[1], stride[2]), ((0, 0), (hl, hh), (wl, wh))
            tl = th = 0
            kt, up_time, pad_t = 1, 1, PAD_ZERO
        Co = w.shape[1]
        To = _out_len(T, kt, stride[0], tl, th)
        Ho = _out_len(H, kh, stride[1], hl, hh)
        Wo = _out_len(W, kw, stride[2], wl, wh)
        if up_time == 2:
            yshape = (B, 2 * To - 1, Ho, Wo, Co // 2)
        else:
            yshape = (B, To, Ho, Wo, Co)
        if out is None:
            out = self.ops.empty(yshape, x.dtype, x.device)
        else:
            assert tuple(out.shape) == yshape, (tuple(out.shape), yshape)
        off = (-tl, -hl, -wl)
        needs_hw_pad = (kh > 1 or kw > 1) and (hl or hh or wl or wh)
        if not self._tc_ok(x):
            # the caller's NCDHW tensor (network input, 3 / 4 / 16 channels): one gather into a channels-last,
            # channel-padded buffer (framed when the conv wants replicate padding) feeds the tensor-core path
            Cp = w.shape[2]
            if pad_hw == PAD_REPLICATE and needs_hw_pad:
                pad, inner = self.ops.empty_padded(B, T, H, W, Cp, x.dtype, x.device)
                self.ops.copy(x, inner)
                self.ops.replicate_border(pad)
                a = Act(inner, pad)
            else:
                a = Act(self.ops.copy(x, self.ops.empty((B, T, H, W, Cp), x.dtype, x.device)))
            x = a.t
        if pad_hw == PAD_REPLICATE and needs_hw_pad and self._tc_ok(x):
            a = self._framed(a)
            x = a.pad
            off = (-tl, 1 - hl, 1 - wl)
            pad_hw = PAD_ZERO
        flat = (kernel == (1, 1, 1) and stride == (1, 1, 1) and x.is_contiguous() and out.is_contiguous()
                and (residual is None or residual.is_contiguous()) and up_time == 1)
        yC = yshape[4]
        cpg = yC // self.cfg.groups if yC % self.cfg.groups == 0 else 0
        stats_ok = (cpg >= 1 and (cpg & (cpg - 1)) == 0 and out.stride(4) == 1 and yC % 8 == 0
                    and all(st_ % 8 == 0 for st_ in out.stride()[:4]))
        if (want_stats or stats is not None) and stats_ok:
            if stats is None:
                stats = self.new_stats(B, x.device)
        else:
            stats = None
        skw = dict(gn_stats=stats, gn_groups=self.cfg.groups) if stats is not None else {}
        if flat:
            # a 1x1x1 convolution is a plain GEMM over the positions of each sample: [B, 1, 1, T*H*W, C] keeps the
            # samples on the batch axis, so the tile plan, every rounding and the epilogue's per-sample GroupNorm
            # sums are the same whether a clip runs alone or in a batch
            P = T * H * W
            self.ops.conv(x.view(B, 1, 1, P, x.shape[4]), w, b, kernel=kernel,
                          residual=residual.view(B, 1, 1, P, Co) if residual is not None else None,
                          out=out.view(B, 1, 1, P, Co), **skw)
        else:
            if k_alg is not None:
                skw["k_alg"] = k_alg
            if shortcut is not None:
                skw["sc_x"], skw["sc_w"] = shortcut[0], shortcut[1]
            self.ops.conv(x, w, b, kernel=kernel, stride=stride, offset=off, pad_t=pad_t, pad_hw=pad_hw,
                          up_time=up_time, residual=residual, out=out, ref_taps=ref_taps, **skw)
        return Act(out, stats=stats)

    def _single_frame_weights(self, wkey, name, w, b, kt, khw, tl, pad_t, up_time):
        """[kt*khw, Co, Ci] -> [khw, Co', Ci] for a one-frame input (cached in the parameter table)."""
        key = f"{wkey}.t1.{tl}.{pad_t}.{up_time}"
        if key not in self.p:
            w4 = w.view(kt, khw, w.shape[1], w.shape[2])
            if pad_t == PAD_REPLICATE:
                wf = w4.float().sum(0).to(w.dtype)      # one rounding of the fp32 sum
            elif 0 <= tl < kt:
                wf = w4[tl]
            else:
                wf = torch.zeros_like(w4[0])
            bf = b
            if up_time == 2:                            # "b (n c) t h w -> b c (t n) h w" then drop frame 0: keep n = 1
                half = w.shape[1] // 2
                wf = wf[:, half:]
                bf = b[half:].contiguous() if b is not None else None
            self.p[key] = wf.contiguous()
            if bf is not None:
                self.p[key + ".bias"] = bf
        return self.p[key], self.p.get(key + ".bias")

    def conv3(self, a: Act, name: str, causal: bool, **kw) -> Act:
        """3x3x3, stride 1, 'same': CausalConv3d / nn.Conv3d(padding=1) / Conv3d(replicate)."""
        if self.sd3:
            tp, pad_t = ((2, 0) if causal else (1, 1)), PAD_REPLICATE
        else:
            tp, pad_t = ((2, 0), PAD_REPLICATE) if causal else ((1, 1), PAD_ZERO)
        return self.conv(a, name, kernel=(3, 3, 3), pads=(tp, (1, 1), (1, 1)), pad_t=pad_t, pad_hw=self.hw_mode, **kw)

    def conv2(self, a: Act, name: str, **kw) -> Act:
        """Conv2dWithExtraDim 3x3 pad 1 (zeros in both families), per frame."""
        return self.conv(a, name, kernel=(1, 3, 3), pads=((0, 0), (1, 1), (1, 1)), pad_t=PAD_ZERO, pad_hw=PAD_ZERO, **kw)

    def conv1(self, a: Act, name: str, **kw) -> Act:
        """1x1(x1) convolution / Linear over channels."""
        return self.conv(a, name, kernel=(1, 1, 1), pads=((0, 0), (0, 0), (0, 0)), pad_t=PAD_ZERO, pad_hw=PAD_ZERO, **kw)

    def gn(self, a: Act, name: str, *, silu=True, per_frame=False, framed=False) -> Act:
        x = a.t
        g, b = self.p[name + ".weight"], self.p[name + ".bias"]
        skw = dict(stats=a.stats) if (a.stats is not None and not per_frame) else {}
        if framed:
            B, T, H, W, Cc = x.shape
            pad, inner = self.ops.empty_padded(B, T, H, W, Cc, x.dtype, x.device)
            self.ops.groupnorm(x, g, b, self.cfg.groups, self.cfg.eps, per_frame=per_frame, silu=silu, out=inner, **skw)
            self.ops.replicate_border(pad)
            return Act(inner, pad)
        return Act(self.ops.groupnorm(x, g, b, self.cfg.groups, self.cfg.eps, per_frame=per_frame, silu=silu, **skw))

    # ------------------------------------------------------------------ blocks
    def resblock(self, a: Act, p: str, causal: bool) -> Act:
        """ResnetBlock3D.forward: vae_models.py:390-410 / vae_blocks3d_sd3.py:518-569."""
        cfg = self.cfg
        h = self.gn(a, p + ".norm1", framed=self.sd3)
        h = self.conv3(h, p + ".conv1", causal, want_stats=True)
        # conv2 is a zero-padded per-frame 3x3 when half_3d, else another conv_cls 3x3x3
        h = self.gn(h, p + ".norm2", framed=(self.sd3 and not cfg.half_3d))
        sc_name = p + (".conv_shortcut" if self.sd3 else ".nin_shortcut")
        conv2 = self.conv2 if cfg.half_3d else (lambda hh, nn, **kw: self.conv3(hh, nn, causal, **kw))
        if (sc_name + ".weight") in self.p:
            if self.fuse_shortcut and self._tc_ok(a.t):
                # K4: the 1x1 shortcut runs as extra K steps of conv2 on the block input (never written, never re-read,
                # the sum rounded once); the two biases are pre-summed in fp32
                key = p + ".conv2.bias+shortcut"
                if key not in self.p:
                    self.p[key] = (self.p[p + ".conv2.bias"] + self.p[sc_name + ".bias"]).contiguous()
                wsc = self.p[sc_name + ".weight"]
                return conv2(h, p + ".conv2", want_stats=True, shortcut=(a.t, wsc.view(wsc.shape[1], wsc.shape[2]), self.p[key]))
            shortcut = self.conv1(Act(a.t), sc_name).t
        else:
            shortcut = a.t
            if not shortcut.is_contiguous():
                # residual operands share the (dense) output geometry
                shortcut = self.ops.copy(shortcut, self.ops.empty(shortcut.shape, shortcut.dtype, shortcut.device))
        # every block output feeds a GroupNorm (next block's norm1 / norm_out) or a conv that ignores the sums
        return conv2(h, p + ".conv2", residual=shortcut, want_stats=True)

    def spatial_attention(self, hn: torch.Tensor, q: torch.Tensor, k: torch.Tensor, v_name: str) -> torch.Tensor:
        """softmax(q k^T / sqrt(C)) v per frame, one head (vae_models.py:446-461,500-528; diffusers Attention).

        Three BATCHED tensor-core GEMMs (batch = the B*T frames, 1x1x1 'flat' problems of the convolution kernel with
        one right operand per frame) and one row softmax over all frames:
          v^T = W_v hn^T + b_v   (left operand W_v shared by the frames, bias along rows; gives the K-major operand of
                                  the last GEMM directly)
          S   = q k^T * C^-0.5   (fp32 logits) ; P = softmax(S) (16 bit)
          O   = P v
        Frames are processed in groups so that the fp32 logits stay below `attn_scratch_bytes`.
        """
        ops = self.ops
        B, T, H, W, Cc = hn.shape
        F, N = B * T, H * W
        ld = (N + 7) // 8 * 8
        wv, bv = self.p[v_name + ".weight"], self.p[v_name + ".bias"]
        out = ops.empty((B, T, H, W, Cc), hn.dtype, hn.device)
        wv_act = wv.view(1, 1, 1, Cc, Cc)
        scale = float(Cc) ** -0.5
        fg = max(1, min(F, self.attn_scratch_bytes // max(1, N * ld * 4)))
        vT = ops.empty((fg, Cc, ld), hn.dtype, hn.device)
        S = torch.empty((fg, N, ld), dtype=torch.float32, device=hn.device)
        P = ops.empty((fg, N, ld), hn.dtype, hn.device)
        hf, qf, kf, of = (t.reshape(F, N, Cc) for t in (hn, q, k, out))
        for f0 in range(0, F, fg):
            n = min(fg, F - f0)
            ops.conv(wv_act, hf[f0:f0 + n], bv, bias_along_m=True, x_shared=True, w_per_batch=True, cout=N,
                     out=vT[:n, :, :N].unsqueeze(1).unsqueeze(1))
            ops.conv(qf[f0:f0 + n].view(n, 1, 1, N, Cc), kf[f0:f0 + n], None, alpha=scale, out_f32=True, w_per_batch=True,
                     cout=N, out=S[:n, :, :N].unsqueeze(1).unsqueeze(1))
            ops.softmax_rows(S[:n].view(n * N, ld), N, P[:n].view(n * N, ld))
            ops.conv(P[:n, :, :N].unsqueeze(1).unsqueeze(1), vT[:n], None, w_ld=ld, cout=Cc, w_per_batch=True,
                     out=of[f0:f0 + n].view(n, 1, 1, N, Cc))
        return out

    def attn_sd21(self, a: Act, p: str, attn_type: str) -> Act:
        """AttnBlock / MemoryEfficientAttnBlock / MemoryEfficientAttnVideoBlock (vae_models.py:427-629)."""
        if attn_type == "none":
            return a
        if attn_type not in ("vanilla", "vanilla-xformers", "spatial-temporal-xformer"):
            raise NotImplementedError(f"attn_type {attn_type!r} is outside the CV-VAE hot path")
        x = a.t
        hn = self.gn(a, p + ".norm", silu=False, per_frame=True)
        q = self.conv1(hn, p + ".q").t
        k = self.conv1(hn, p + ".k").t
        o = Act(self.spatial_attention(hn.t, q, k, p + ".v"))
        if attn_type != "spatial-temporal-xformer":
            return self.conv1(o, p + ".proj_out", residual=x, want_stats=True)
        h1 = self.conv1(o, p + ".proj_out")
        hn2 = Act(self.ops.layernorm(h1.t, self.p[p + ".norm_t.weight"], self.p[p + ".norm_t.bias"], 1e-5))
        qt = self.conv1(hn2, p + ".q_t").t
        kt = self.conv1(hn2, p + ".k_t").t
        vt = self.conv1(hn2, p + ".v_t").t
        ot = Act(self.ops.attn_temporal(qt, kt, vt))
        return self.conv1(ot, p + ".proj_out_t", residual=x, want_stats=True)

    def attn_sd3(self, a: Act, p: str) -> Act:
        """AttentionWithExtraDim over diffusers Attention (vae_blocks3d_sd3.py:119-147,805-823)."""
        x = a.t
        if not x.is_contiguous():
            x = self.ops.copy(x, self.ops.empty(x.shape, x.dtype, x.device))
        hn = self.gn(Act(x), p + ".group_norm", silu=False, per_frame=True)
        q = self.conv1(hn, p + ".to_q").t
        k = self.conv1(hn, p + ".to_k").t
        o = Act(self.spatial_attention(hn.t, q, k, p + ".to_v"))
        return self.conv1(o, p + ".to_out.0", residual=x, want_stats=True)

    # ------------------------------------------------------------------ networks
    def encode(self, x: torch.Tensor) -> torch.Tensor:
        """x: [B, C, T, H, W] (any strides) -> moments [B, 2z, T', H/8, W/8] (contiguous NCDHW)."""
        cfg = self.cfg
        causal = cfg.causal_encoder
        L = len(cfg.widths)
        a = Act(x.permute(0, 2, 3, 4, 1))
        self._begin_pass(x.shape[0], x.device)
        E = "encoder."
        h = self.conv3(a, E + "conv_in", causal, want_stats=True)
        for lvl in range(L):
            for b in range(cfg.num_res_blocks):
                name = f"{E}down_blocks.{lvl}.resnets.{b}" if self.sd3 else f"{E}down.{lvl}.block.{b}"
                h = self.resblock(h, name, causal)
            if lvl != L - 1:
                h = self.downsample(h, lvl, causal)
        if self.sd3:
            h = self.resblock(h, E + "mid_block.resnets.0", causal)
            if cfg.mid_block_add_attention:
                h = self.attn_sd3(h, E + "mid_block.attentions.0")
            h = self.resblock(h, E + "mid_block.resnets.1", causal)
            h = self.gn(h, E + "conv_norm_out", framed=True)
        else:
            h = self.resblock(h, E + "mid.block_1", causal)
            h = self.attn_sd21(h, E + "mid.attn_1", cfg.encoder_attn_type)
            h = self.resblock(h, E + "mid.block_2", causal)
            h = self.gn(h, E + "norm_out")
        B, T, H, W, _ = h.t.shape
        out = torch.empty((B, cfg.moments_channels, T, H, W), dtype=x.dtype, device=x.device)
        self.conv3(h, E + "conv_out", causal, out=out.permute(0, 2, 3, 4, 1))
        return out

    def decode(self, z: torch.Tensor) -> torch.Tensor:
        """z: [B, zc, T', h, w] -> x [B, 3, 4(T'-1)+1, 8h, 8w] (contiguous NCDHW)."""
        cfg = self.cfg
        causal = cfg.causal_decoder
        L = len(cfg.widths)
        D = "decoder."
        a = Act(z.permute(0, 2, 3, 4, 1))
        self._begin_pass(z.shape[0], z.device)
        h = self.conv3(a, D + "conv_in", causal, want_stats=True)
        if self.sd3:
            h = self.resblock(h, D + "mid_block.resnets.0", causal)
            if cfg.mid_block_add_attention:
                h = self.attn_sd3(h, D + "mid_block.attentions.0")
            h = self.resblock(h, D + "mid_block.resnets.1", causal)
        else:
            h = self.resblock(h, D + "mid.block_1", causal)
            h = self.attn_sd21(h, D + "mid.attn_1", cfg.decoder_attn_type)
            h = self.resblock(h, D + "mid.block_2", causal)
        for i in range(L):
            lvl = L - 1 - i  # sd21 names levels bottom-up, sd3 names blocks in execution order
            for b in range(cfg.num_res_blocks + 1):
                name = f"{D}up_blocks.{i}.resnets.{b}" if self.sd3 else f"{D}up.{lvl}.block.{b}"
                h = self.resblock(h, name, causal)
            if i != L - 1:
                up_time = 2 if (lvl % 2 == 1) else 1  # == (i % 2 == 0) for L = 4
                if self.sd3:
                    up_time = 2 if (i % 2 == 0) else 1
                h = self.upsample(h, f"{D}up_blocks.{i}.upsamplers.0.conv" if self.sd3 else f"{D}up.{lvl}.upsample.conv",
                                  up_time, causal)
        h = self.gn(h, D + ("conv_norm_out" if self.sd3 else "norm_out"), framed=self.sd3)
        B, T, H, W, _ = h.t.shape
        out = torch.empty((B, cfg.out_ch, T, H, W), dtype=z.dtype, device=z.device)
        stk = self.p.get(D + "conv_out.weight.stk")
        if stk is not None and hasattr(self.ops, "conv_stacked"):
            # 128 -> 3 at full resolution: tap-stacked kernel (N = 16 MMAs are bound by A-operand reads)
            if self.sd3:
                tl, pad_t = (2 if causal else 1), PAD_REPLICATE
                x_in, off = h.pad, (-tl, 0, 0)        # framed input: replicate border already in place
            else:
                tl, pad_t = ((2, PAD_REPLICATE) if causal else (1, PAD_ZERO))
                x_in, off = h.t, (-tl, -1, -1)
            self.ops.conv_stacked(x_in, stk, self.p.get(D + "conv_out.bias"), kt=stk.shape[0], cout=cfg.out_ch, offset=off,
                                  pad_t=pad_t, pad_hw=PAD_ZERO, out=out.permute(0, 2, 3, 4, 1))
        else:
            self.conv3(h, D + "conv_out", causal, out=out.permute(0, 2, 3, 4, 1))
        return out

    def downsample(self, h: Act, lvl: int, causal: bool) -> Act:
        """Downsample3D.forward of encoder level `lvl` (time stride 2 at the even levels)."""
        st = 2 if lvl % 2 == 0 else 1
        if self.sd3:
            # Downsample3D -> conv_cls(k3, stride, padding=1): vae_blocks3d_sd3.py:200-210
            tp = (2, 0) if causal else (1, 1)
            return self.conv(h, f"encoder.down_blocks.{lvl}.downsamplers.0.conv", kernel=(3, 3, 3), stride=(st, 2, 2),
                             pads=(tp, (1, 1), (1, 1)), pad_t=PAD_REPLICATE, pad_hw=PAD_REPLICATE, want_stats=True)
        # Downsample3D.forward vae_models.py:251-263: zero pad right/bottom, replicate 2 frames in front
        return self.conv(h, f"encoder.down.{lvl}.downsample.conv", kernel=(3, 3, 3), stride=(st, 2, 2),
                         pads=((2, 0), (0, 1), (0, 1)), pad_t=PAD_REPLICATE, pad_hw=PAD_ZERO, want_stats=True)

    def upsample(self, a: Act, name: str, up_time: int, causal: bool) -> Act:
        """Upsample3D.forward (vae_models.py:214-235, vae_blocks3d_sd3.py:314-364): nearest x(1,2,2), 3x3x3 conv
        to C*up_time channels, channel->time interleave and drop of frame 0.

        Executed as four 3x2x2 phase convolutions on the NOT up-sampled input (weights folded in prepack_params),
        each writing its (ph::2, pw::2) lattice of the output through a strided view; the interleave/drop is the
        conv epilogue's store address.  The 4x tensor of the reference never exists."""
        x = a.t
        B, T, H, W, Cc = x.shape
        if self.sd3:
            tp = (2, 0) if causal else (1, 1)
            pad_t, pad_hw = PAD_REPLICATE, PAD_REPLICATE
            a = self._framed(a)  # one replicate frame around the (small) input serves all four phases
        else:
            # NB the sd21 Decoder never forwards `causal` to Upsample3D (vae_models.py:936): always replicate (1,1)
            tp = (1, 1)
            pad_t, pad_hw = PAD_REPLICATE, PAD_ZERO
        Co = self.p[name + ".phase00.weight"].shape[1]
        To = _out_len(T, 3, 1, tp[0], tp[1])
        yshape = (B, 2 * To - 1, 2 * H, 2 * W, Co // 2) if up_time == 2 else (B, To, 2 * H, 2 * W, Co)
        y = self.ops.empty(yshape, x.dtype, x.device)
        stats = None
        for ph in (0, 1):
            for pw in (0, 1):
                r = self.conv(a, name, kernel=(3, 2, 2), pads=(tp, (1, 0) if ph == 0 else (0, 1), (1, 0) if pw == 0 else (0, 1)),
                              pad_t=pad_t, pad_hw=pad_hw, up_time=up_time, out=y[:, :, ph::2, pw::2, :],
                              weight_key=f"{name}.phase{ph}{pw}.weight", ref_taps=27, stats=stats,
                              want_stats=(ph == 0 and pw == 0))
                stats = r.stats
        return Act(y, stats=stats)
