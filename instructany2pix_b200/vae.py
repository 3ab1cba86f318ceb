"""``B200VAE``: the SDXL ``AutoencoderKL`` decode / encode path on the sm_100a kernels (SURVEY.md 8f-1, row a22).

Reference call sites: ``vae.decode(latents / vae.config.scaling_factor)`` after the sampling loop
(ddim/sdxl_pipeline.py:859-871, fp32 upcast :523-540) and ``vae.encode(image).latent_dist.sample() * scaling_factor`` in
``prepare_latents`` of the inversion pipeline (ddim/pnp_pipeline.py:195-204).  The module itself is third-party
(diffusers==0.26.3 ``AutoencoderKL``, SDXL VAE config): parameter names below are the diffusers state-dict names, so a real
checkpoint loads with ``load_state_dict``.

Same kernels as the UNet: NHWC activations, fp32 residual stream with bf16 tensor-core operands, fused GroupNorm+SiLU,
tcgen05 implicit-GEMM 3x3 convs with the 1x1 shortcut and the residual add in the epilogue.  The single 512-wide attention
head of the mid block (L*L tokens, once per image) runs as GEMM (fp32 scores) -> row softmax -> GEMM; V is produced already
transposed by swapping the GEMM operands, and its bias is added after P.V (rows of P sum to one).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Tuple

import torch
import torch.nn as nn

from . import ops
from .packing import pack_conv3x3, pack_conv3x3_up2x, pack_conv_out
from .sampler import randn_per_request


@dataclass
class B200VAEConfig:
    in_channels: int = 3
    out_channels: int = 3
    latent_channels: int = 4
    block_out_channels: Tuple[int, ...] = (128, 256, 512, 512)
    layers_per_block: int = 2
    norm_num_groups: int = 32
    scaling_factor: float = 0.13025
    force_upcast: bool = True

    def get(self, k, default=None):
        return getattr(self, k, default)


class _Holder(nn.Module):
    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError("parameter holder: arithmetic runs in libia2p_sm100a.so via B200VAE.decode / encode")


class _Res(_Holder):
    def __init__(self, cin, cout, groups):
        super().__init__()
        self.norm1 = nn.GroupNorm(groups, cin, eps=1e-6)
        self.conv1 = nn.Conv2d(cin, cout, 3, padding=1)
        self.norm2 = nn.GroupNorm(groups, cout, eps=1e-6)
        self.conv2 = nn.Conv2d(cout, cout, 3, padding=1)
        if cin != cout:
            self.conv_shortcut = nn.Conv2d(cin, cout, 1)


class _Attn(_Holder):
    def __init__(self, c, groups):
        super().__init__()
        self.group_norm = nn.GroupNorm(groups, c, eps=1e-6)
        self.to_q, self.to_k, self.to_v = nn.Linear(c, c), nn.Linear(c, c), nn.Linear(c, c)
        self.to_out = nn.ModuleList([nn.Linear(c, c), nn.Dropout(0.0)])


class _Mid(_Holder):
    def __init__(self, c, groups):
        super().__init__()
        self.resnets = nn.ModuleList([_Res(c, c, groups), _Res(c, c, groups)])
        self.attentions = nn.ModuleList([_Attn(c, groups)])


class _ConvHolder(_Holder):
    def __init__(self, c, stride=1):
        super().__init__()
        self.conv = nn.Conv2d(c, c, 3, stride=stride, padding=1 if stride == 1 else 0)


class _UpBlock(_Holder):
    def __init__(self, cin, cout, n, groups, add_up):
        super().__init__()
        self.resnets = nn.ModuleList([_Res(cin if i == 0 else cout, cout, groups) for i in range(n)])
        if add_up:
            self.upsamplers = nn.ModuleList([_ConvHolder(cout)])


class _DownBlock(_Holder):
    def __init__(self, cin, cout, n, groups, add_down):
        super().__init__()
        self.resnets = nn.ModuleList([_Res(cin if i == 0 else cout, cout, groups) for i in range(n)])
        if add_down:
            self.downsamplers = nn.ModuleList([_ConvHolder(cout, stride=2)])


class _Decoder(_Holder):
    def __init__(self, cfg):
        super().__init__()
        ch, G = cfg.block_out_channels, cfg.norm_num_groups
        self.conv_in = nn.Conv2d(cfg.latent_channels, ch[-1], 3, padding=1)
        self.mid_block = _Mid(ch[-1], G)
        rch = list(reversed(ch))
        ups, prev = [], rch[0]
        for i, c in enumerate(rch):
            ups.append(_UpBlock(prev, c, cfg.layers_per_block + 1, G, add_up=i < len(rch) - 1))
            prev = c
        self.up_blocks = nn.ModuleList(ups)
        self.conv_norm_out = nn.GroupNorm(G, ch[0], eps=1e-6)
        self.conv_out = nn.Conv2d(ch[0], cfg.out_channels, 3, padding=1)


class _Encoder(_Holder):
    def __init__(self, cfg):
        super().__init__()
        ch, G = cfg.block_out_channels, cfg.norm_num_groups
        self.conv_in = nn.Conv2d(cfg.in_channels, ch[0], 3, padding=1)
        downs, prev = [], ch[0]
        for i, c in enumerate(ch):
            downs.append(_DownBlock(prev, c, cfg.layers_per_block, G, add_down=i < len(ch) - 1))
            prev = c
        self.down_blocks = nn.ModuleList(downs)
        self.mid_block = _Mid(ch[-1], G)
        self.conv_norm_out = nn.GroupNorm(G, ch[-1], eps=1e-6)
        self.conv_out = nn.Conv2d(ch[-1], 2 * cfg.latent_channels, 3, padding=1)


class B200VAE(nn.Module):
    """decode(latents) -> images, encode(images) -> latents, with the latent scaling of the reference call sites folded in."""

    def __init__(self, config=None, device="cuda", with_encoder=True):
        super().__init__()
        cfg = config if isinstance(config, B200VAEConfig) else B200VAEConfig(**(config or {}))
        self.config = cfg
        with torch.device("meta"):
            self.decoder = _Decoder(cfg)
            self.post_quant_conv = nn.Conv2d(cfg.latent_channels, cfg.latent_channels, 1)
            if with_encoder:
                self.encoder = _Encoder(cfg)
                self.quant_conv = nn.Conv2d(2 * cfg.latent_channels, 2 * cfg.latent_channels, 1)
        self.to_empty(device=device)
        for p in self.parameters():
            p.requires_grad_(False)
        self._packed = None

    @property
    def device(self):
        return next(self.parameters()).device

    @property
    def dtype(self):
        return torch.float32                        # callers upcast the VAE to fp32 (sdxl_pipeline.py:523-540)

    def invalidate(self):
        self._packed = None

    def load_state_dict(self, sd, strict=True, assign=False):
        r = super().load_state_dict(sd, strict=strict, assign=assign)
        self.invalidate()
        return r

    # ------------------------------------------------------------------ packing (once per load)
    def prepare(self):
        if self._packed is not None:
            return self._packed
        P = {}
        f32 = lambda t: t.detach().float().contiguous()
        bf = lambda t: t.detach().to(torch.bfloat16).contiguous()
        for name, m in self.named_modules():
            if isinstance(m, _Res):
                sc = getattr(m, "conv_shortcut", None)
                P[name] = dict(g1=f32(m.norm1.weight), b1=f32(m.norm1.bias), w1=pack_conv3x3(m.conv1.weight), cb1=f32(m.conv1.bias),
                               g2=f32(m.norm2.weight), b2=f32(m.norm2.bias),
                               w2=pack_conv3x3(m.conv2.weight, None if sc is None else sc.weight),
                               cb2=f32(m.conv2.bias if sc is None else m.conv2.bias.float() + sc.bias.float()), has_sc=sc is not None)
            elif isinstance(m, _Attn):
                P[name] = dict(g=f32(m.group_norm.weight), b=f32(m.group_norm.bias),
                               wq=bf(m.to_q.weight), bq=f32(m.to_q.bias), wk=bf(m.to_k.weight), bk=f32(m.to_k.bias),
                               wv=bf(m.to_v.weight), bv=f32(m.to_v.bias), wo=bf(m.to_out[0].weight), bo=f32(m.to_out[0].bias))
            elif isinstance(m, _ConvHolder):
                P[name] = dict(w=pack_conv3x3(m.conv.weight), b=f32(m.conv.bias))
                if ".upsamplers." in name:
                    P[name]["w4"] = pack_conv3x3_up2x(m.conv.weight)
        for side in ("decoder", "encoder"):
            if hasattr(self, side):
                mod = getattr(self, side)
                P[side + ".conv_in"] = (f32(mod.conv_in.weight), f32(mod.conv_in.bias))
                P[side + ".conv_out"] = pack_conv_out(mod.conv_out.weight, mod.conv_out.bias)
                P[side + ".norm_out"] = (f32(mod.conv_norm_out.weight), f32(mod.conv_norm_out.bias))
        self._packed = P
        return P

    # ------------------------------------------------------------------ shared blocks
    def _res(self, P, name, x):
        p, G = P[name], self.config.norm_num_groups
        raw = None
        if p["has_sc"]:
            h, raw = ops.groupnorm(x, None, p["g1"], p["b1"], G, 1e-6, True, want_raw=True)
        else:
            h = ops.groupnorm(x, None, p["g1"], p["b1"], G, 1e-6, True)
        h = ops.conv3x3(h, p["w1"], p["w1"].shape[0], bias=p["cb1"], out_dtype=torch.float32, want_colstats=True)
        h = ops.groupnorm(h, None, p["g2"], p["b2"], G, 1e-6, True)
        if p["has_sc"]:
            return ops.conv3x3(h, p["w2"], p["w2"].shape[0], sc_a=raw, bias=p["cb2"], out_dtype=torch.float32, want_colstats=True)
        return ops.conv3x3(h, p["w2"], p["w2"].shape[0], bias=p["cb2"], residual=x, out_dtype=torch.float32, want_colstats=True)

    def _attn(self, P, name, x):
        """single head, head_dim = C ([3P] Attention with heads=1): softmax(q k^T / sqrt C) v, residual add in to_out's epilogue."""
        p, G = P[name], self.config.norm_num_groups
        B, H, W, C = x.shape
        N = H * W
        t = ops.groupnorm(x, None, p["g"], p["b"], G, 1e-6, False).reshape(B * N, C)
        q = ops.gemm(t, p["wq"], bias=p["bq"])                                       # [B*N, C] bf16
        k = ops.gemm(t, p["wk"], bias=p["bk"])
        o = torch.empty(B * N, C, device=x.device, dtype=torch.bfloat16)
        for b in range(B):
            rows = slice(b * N, (b + 1) * N)
            s = ops.gemm(q[rows], k[rows], out_dtype=torch.float32)                 # scores [N, N] fp32
            pr = ops.softmax_rows(s, C ** -0.5)
            del s
            vt = ops.gemm(p["wv"], t[rows])                                         # V^T [C, N] (bias added after P.V)
            ops.gemm(pr, vt, bias=p["bv"], out=o[rows])
            del pr, vt
        xf = x.reshape(B * N, C)
        return ops.gemm(o, p["wo"], bias=p["bo"], residual=xf, out_dtype=torch.float32).reshape(B, H, W, C)

    def _mid(self, P, side, x):
        x = self._res(P, f"{side}.mid_block.resnets.0", x)
        x = self._attn(P, f"{side}.mid_block.attentions.0", x)
        return self._res(P, f"{side}.mid_block.resnets.1", x)

    # ------------------------------------------------------------------ decode (sdxl_pipeline.py:859-871)
    @torch.no_grad()
    def decode(self, latents, scaled=True):
        """latents (B,4,L,L) as the sampler returns them -> images (B,3,8L,8L) fp32, nominal range [-1, 1].
        ``scaled=True`` folds the reference's ``latents / scaling_factor`` into post_quant_conv."""
        P, cfg = self.prepare(), self.config
        G = cfg.norm_num_groups
        z = ops.conv1x1_nchw_small(latents.to(self.device, torch.float32), self.post_quant_conv.weight, self.post_quant_conv.bias,
                                   1.0 / cfg.scaling_factor if scaled else 1.0)
        x = ops.conv_in(z, *P["decoder.conv_in"], out_dtype=torch.float32)
        x = self._mid(P, "decoder", x)
        for i, blk in enumerate(self.decoder.up_blocks):
            for j in range(len(blk.resnets)):
                x = self._res(P, f"decoder.up_blocks.{i}.resnets.{j}", x)
            if hasattr(blk, "upsamplers"):
                q = P[f"decoder.up_blocks.{i}.upsamplers.0"]
                x = ops.conv_up2x(ops.to_bf16(x), q["w4"], q["w"].shape[0], bias=q["b"], want_colstats=True)   # Upsample2D folded
        h = ops.groupnorm(x, None, *P["decoder.norm_out"], G, 1e-6, True)
        return ops.conv_out_tc(h, *P["decoder.conv_out"], cfg.out_channels)

    # ------------------------------------------------------------------ encode (pnp_pipeline.py:195-204)
    @torch.no_grad()
    def encode(self, images, noise=None, generator=None, sample=True, scaled=True):
        """images (B,3,H,W) in [-1, 1] -> latents (B,4,H/8,W/8) fp32 = ``latent_dist.sample() * scaling_factor``
        (``sample=False``: the mode).  ``noise`` may be supplied for parity tests; ``generator`` may be one generator per image."""
        P, cfg = self.prepare(), self.config
        G = cfg.norm_num_groups
        x = ops.conv_in(images.to(self.device, torch.float32), *P["encoder.conv_in"], out_dtype=torch.float32)
        for i, blk in enumerate(self.encoder.down_blocks):
            for j in range(len(blk.resnets)):
                x = self._res(P, f"encoder.down_blocks.{i}.resnets.{j}", x)
            if hasattr(blk, "downsamplers"):
                q = P[f"encoder.down_blocks.{i}.downsamplers.0"]
                x = ops.conv3x3_down_padend(ops.to_bf16(x), q["w"], q["w"].shape[0], bias=q["b"], out_dtype=torch.float32)
        x = self._mid(P, "encoder", x)
        h = ops.groupnorm(x, None, *P["encoder.norm_out"], G, 1e-6, True)
        moments = ops.conv_out_tc(h, *P["encoder.conv_out"], 2 * cfg.latent_channels)               # (B, 8, h, w)
        moments = ops.conv1x1_nchw_small(moments, self.quant_conv.weight, self.quant_conv.bias, 1.0)
        sf = cfg.scaling_factor if scaled else 1.0
        if not sample:
            return ops.gaussian_sample(moments, None, sf)
        # DiagonalGaussianDistribution.sample ([3P]): mean + exp(0.5 * clamp(logvar, -30, 20)) * noise
        if noise is None:
            B, C2, h, w = moments.shape
            noise = randn_per_request((B, C2 // 2, h, w), moments.device, generator)
        return ops.gaussian_sample(moments, noise.to(moments.device, torch.float32), sf)
