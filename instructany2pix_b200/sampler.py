"""Fused sampling loops over ``B200UNet`` (the denoising hot path itself).

``generate`` replaces the loop body the reference runs through ``IPAdapterXL.generate`` ->
``StableDiffusionXLPipeline.__call__`` (in-tree text: diffusion/ip_adapter/custom_pipelines.py:324-363,
ddim/sdxl_pipeline.py:823-857); ``invert`` replaces ``SDXLDDIMPipeline.inverse``'s loop (ddim/pnp_pipeline.py:251-275).
Per step the device sees: one copy of the step's pre-computed time-embedding biases, ONE CUDA-graph replay of the whole
UNet forward (CFG duplication folded into conv_in), and ONE fused CFG+DDIM kernel.  No host<->device sync, no NCCL.
Everything step-invariant (cross-attention K/V of all layers, time-embedding MLPs for all timesteps) is done once.
"""
from __future__ import annotations

import math
import numbers

import torch

from . import ops
from .scheduler import B200DDIMScheduler


def per_request(v, B, name):
    """``v`` as B finite floats, one per request, or None when it is one number for the whole batch (a float, or a 0-d tensor)."""
    if isinstance(v, numbers.Real) or (isinstance(v, torch.Tensor) and v.ndim == 0):
        return None
    vals = [float(u) for u in (v.reshape(-1).tolist() if isinstance(v, torch.Tensor) else v)]
    if len(vals) != B:
        raise ValueError(f"{name}: {len(vals)} values for {B} requests")
    if not all(math.isfinite(u) for u in vals):
        raise ValueError(f"{name}: non-finite value in {vals}")
    return vals


def randn_per_request(shape, device, generator=None):
    """``torch.randn(shape)`` in fp32; a list of generators (diffusers' convention) gives row i its own draw from
    ``generator[i]``, the same draw a batch of one with that generator gets."""
    if not isinstance(generator, (list, tuple)):
        return torch.randn(shape, device=device, dtype=torch.float32, generator=generator)
    if len(generator) != shape[0]:
        raise ValueError(f"generator: {len(generator)} generators for {shape[0]} requests")
    return torch.cat([torch.randn((1,) + tuple(shape[1:]), device=device, dtype=torch.float32, generator=g) for g in generator])


class B200Sampler:
    def __init__(self, unet, scheduler=None, use_cuda_graph=True):
        self.unet = unet
        self.scheduler = scheduler or B200DDIMScheduler()
        self.use_cuda_graph = use_cuda_graph
        self.max_graphs = 2
        self._graphs = {}

    # ------------------------------------------------------------------ CUDA-graph plumbing
    def _static(self, key, sample_shape, unet_batch, kv, rb_width, dev, ip_rows=False):
        ent = self._graphs.get(key)
        if ent is not None:
            self._graphs[key] = self._graphs.pop(key)      # most recently used last
            return ent
        kv_t, kv_i, n_text, n_ip = kv
        ent = dict(
            x=torch.zeros(sample_shape, device=dev, dtype=torch.float32),
            rb=torch.zeros(rb_width, device=dev, dtype=torch.float32),       # one row of the blocked rowbias table
            kv_t=torch.empty_like(kv_t), kv_i=None if kv_i is None else torch.empty_like(kv_i),
            # per-request IP scales of the UNet rows: the captured cross-attentions read them at replay time
            ips=torch.zeros(unet_batch, device=dev, dtype=torch.float32) if ip_rows else None,
            g=None,                                                          # per-request guidance scales, made on first use
            graph=None, eps=None)
        # small LRU: an edit request alternates the inversion graph (batch B) and the CFG graph (batch 2B); each resident graph's
        # private pool holds a full set of activations, so older shapes are dropped (B200HotPath.edit never recaptures in steady state)
        while len(self._graphs) >= self.max_graphs:
            self._graphs.pop(next(iter(self._graphs)))
        self._graphs[key] = ent
        return ent

    def _forward(self, ent, unet_batch, n_text, n_ip):
        kv = (ent["kv_t"], ent["kv_i"], n_text, n_ip)
        ips = ent["ips"]
        if not self.use_cuda_graph:
            ent["eps"] = self.unet.forward_core(ent["x"], ent["rb"], kv, unet_batch, out_dtype=torch.float32, ip_scales=ips)
            return
        if ent["graph"] is None:
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):      # warm-up outside capture: first-use function attributes, workspaces
                self.unet.forward_core(ent["x"], ent["rb"], kv, unet_batch, out_dtype=torch.float32, ip_scales=ips)
            torch.cuda.current_stream().wait_stream(s)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                ent["eps"] = self.unet.forward_core(ent["x"], ent["rb"], kv, unet_batch, out_dtype=torch.float32, ip_scales=ips)
            ent["graph"] = g
        ent["graph"].replay()

    def _prepare(self, kind, latents, ctx, added, unet_batch, timesteps, ip_rows=None):
        """``ip_rows``: per-request IP scales (B floats, the CFG batch is [uncond; cond]) or None for the processors' scale"""
        unet = self.unet
        dev = unet.device
        kv = unet.context_kv(ctx)
        table = unet.time_rowbias_table(timesteps, added, unet_batch)      # [steps, unet_batch * sumC], blocked per ResnetBlock
        n_ip, ip_scale = unet._ip_state()
        if ip_rows is not None and n_ip == 0:
            raise ValueError("ip_scale given, but the UNet has no IP-adapter processors")
        # per-request scales are data of the entry, not part of the key: new values never re-capture the graph
        key = (kind, tuple(latents.shape), unet_batch, tuple(kv[0].shape), None if kv[1] is None else tuple(kv[1].shape),
               kv[2], kv[3], "per-row" if ip_rows is not None else ip_scale, unet._proc_version, id(unet._packed))
        cin = int(getattr(unet.config, "in_channels", 4))      # 9: inpainting UNet (latents + mask + masked-image latents)
        ent = self._static(key, (latents.shape[0], cin) + tuple(latents.shape[2:]), unet_batch, kv, table.shape[-1], dev,
                           ip_rows=ip_rows is not None)
        ent["kv_t"].copy_(kv[0])
        if kv[1] is not None:
            ent["kv_i"].copy_(kv[1])
        if ip_rows is not None:
            ent["ips"].copy_(torch.tensor(ip_rows * (unet_batch // len(ip_rows)), dtype=torch.float32))
        return ent, table, kv[2], kv[3]

    # ------------------------------------------------------------------ start latent (pipeline.py:330-336)
    @torch.no_grad()
    def start_latent(self, latent_inv, alpha=0.7, noise=None, generator=None):
        """``polar_intrtpolate(latent_inv, randn_like(latent_inv), alpha)`` (pipeline.py:295-300, :332-336): the inverted
        latent is blended with fresh noise and the blend is rescaled to the blended norm.  ``noise`` may be supplied (parity
        tests); otherwise it is drawn like the reference does (global RNG or ``generator``).  ``alpha`` may hold one value per
        request and ``generator`` one generator per request (diffusers' convention: request i draws its noise from
        ``generator[i]`` alone, exactly as it would in a batch of one)."""
        x = latent_inv.to(self.unet.device, torch.float32).contiguous()
        B = x.shape[0]
        alphas = per_request(alpha, B, "alpha") or [alpha] * B
        if noise is None:
            noise = randn_per_request(x.shape, x.device, generator)
        noise = noise.to(x.device, torch.float32).contiguous()
        if x.shape[0] == 1:
            return ops.polar_interpolate(x, noise, alphas[0])
        # the reference takes the norms over the whole tensor and only ever runs one image (pipeline.py:295-300, :332-336); a batch
        # here is a batch of independent requests, so every sample is blended with ITS OWN norms
        out = torch.empty_like(x)
        for b in range(x.shape[0]):
            ops.polar_interpolate(x[b], noise[b], alphas[b], out=out[b])
        return out

    # ------------------------------------------------------------------ generation (CFG, DDIM eta=0)
    @torch.no_grad()
    def generate(self, latents, ctx, added_cond_kwargs, num_inference_steps=50, guidance_scale=10.0, trace=None,
                 teacher=None, init_latents=None, strength=1.0, inpaint_mask=None, masked_image_latents=None, ip_scale=None):
        """latents: (B,4,L,L) initial noise; ctx: (2B,S,D) = cat([negative, positive]) incl. IP tokens
        (ip_adapter.py:341-342, custom_pipelines.py:296-302); added_cond_kwargs: text_embeds (2B,P), time_ids (2B,6).
        Returns final latents (B,4,L,L) fp32 on the device.

        Mixed requests in one batch: ``guidance_scale`` may be one float or B values (sequence or tensor), and ``ip_scale`` one
        float or B values applied to the IP branch of every cross-attention (None: the processors' ``scale``, as ``set_scale``
        left it).  Per-request values live in device buffers of the graph entry; changing them between calls never re-captures.

        img2img / refiner (pipeline.py:358-361, [3P] StableDiffusionXLImg2ImgPipeline): ``init_latents`` (the encoded image) and
        ``strength`` < 1 -> only the last int(N * strength) steps run, starting from ``add_noise(init_latents, latents, t_start)``.
        Inpainting (gdino/lib.py:85-102, [3P] StableDiffusionXLInpaintPipeline with a 4-channel UNet): additionally
        ``inpaint_mask`` (B,1,L,L), 1 = repaint: after every step the kept region is reset to the re-noised original.
        9-channel inpainting UNet (``unet.config.in_channels == 9``, the released SDXL-inpainting layout; the reference itself hands
        the 4-channel base UNet to the pipeline, pipeline.py:132-139): the model sees ``cat([latents, mask, masked_image_latents])``
        every step -- ``inpaint_mask`` and ``masked_image_latents`` (B,4,L,L) are required and nothing is blended."""
        nine = int(getattr(self.unet.config, "in_channels", 4)) == 9
        if nine and (inpaint_mask is None or masked_image_latents is None or init_latents is None):
            raise ValueError("a 9-channel inpainting UNet needs init_latents, inpaint_mask and masked_image_latents")
        if inpaint_mask is not None and init_latents is None:
            raise ValueError("generate(inpaint_mask=...) needs init_latents (the encoded original the kept region is reset to)")
        s = self.scheduler
        s.set_timesteps(num_inference_steps)
        B = latents.shape[0]
        assert ctx.shape[0] == 2 * B, "ctx must hold [uncond; cond] rows"
        g_rows = per_request(guidance_scale, B, "guidance_scale")
        ip_rows = None
        if ip_scale is not None:          # one value for all requests also takes the per-row path: no re-capture when it changes
            ip_rows = per_request(ip_scale, B, "ip_scale") or per_request([ip_scale] * B, B, "ip_scale")
        timesteps = s.timesteps
        if init_latents is not None:
            n_run = min(int(num_inference_steps * strength), num_inference_steps)
            timesteps = timesteps[max(num_inference_steps - n_run, 0):]
            assert len(timesteps) > 0, "strength too small: no denoising step left"
        ent, table, n_text, n_ip = self._prepare("gen", latents, ctx, added_cond_kwargs, 2 * B, timesteps, ip_rows=ip_rows)
        if g_rows is not None:
            if ent["g"] is None:
                ent["g"] = torch.empty(B, device=ent["x"].device, dtype=torch.float32)
            ent["g"].copy_(torch.tensor(g_rows, dtype=torch.float32))
            guidance_scale = ent["g"]
        scaled_input = hasattr(s, "input_scale")           # Euler: the UNet sees x / sqrt(sigma^2 + 1), DDIM: x itself
        x = torch.empty(latents.shape, device=ent["x"].device, dtype=torch.float32) if (scaled_input or nine) else ent["x"]
        if nine:                                           # channels 4..8 of the model input are constant over the trajectory
            ent["x"][:, 4:5].copy_(inpaint_mask.to(x.device, torch.float32))
            ent["x"][:, 5:9].copy_(masked_image_latents.to(x.device, torch.float32))
        noise = latents.to(x.device, torch.float32)
        if init_latents is None:
            x.copy_(noise * s.init_noise_sigma)
        else:
            orig = init_latents.to(x.device, torch.float32).contiguous()
            if strength >= 1.0 and inpaint_mask is not None:
                x.copy_(noise * s.init_noise_sigma)            # pure-noise start ([3P] inpaint pipeline, strength == 1)
            else:
                c_x, c_e = s.add_noise_coefficients(timesteps[0])
                ops.axpby(noise.contiguous(), orig, c_x, c_e, out=x)
        mask = None if inpaint_mask is None else inpaint_mask.to(x.device, torch.float32).contiguous()
        ts_list = timesteps.tolist()
        for i, t in enumerate(ts_list):
            if teacher is not None:
                x.copy_(teacher[i])
            if nine:
                ent["x"][:, :4].copy_(x * s.input_scale(t) if scaled_input else x)
            elif scaled_input:
                ops.axpby(x, x, s.input_scale(t), 0.0, out=ent["x"])
            ent["rb"].copy_(table[i])
            self._forward(ent, 2 * B, n_text, n_ip)
            if trace is not None:
                trace.append(dict(t=t, x=x.clone(), eps2=ent["eps"].clone()))
            s.cfg_step(ent["eps"], t, x, guidance_scale, out=x)
            if mask is not None and not nine:
                if i + 1 < len(ts_list):
                    c_x, c_e = s.add_noise_coefficients(ts_list[i + 1])
                    ops.inpaint_blend(x, orig, noise, mask, c_x, c_e, out=x)
                else:
                    ops.inpaint_blend(x, orig, None, mask, 1.0, 0.0, out=x)
        return x.clone()

    # ------------------------------------------------------------------ DDIM inversion (batch B, no CFG)
    @torch.no_grad()
    def invert(self, latents, ctx, added_cond_kwargs, num_inference_steps=50, trace=None):
        s = self.scheduler
        s.set_timesteps(num_inference_steps)
        B = latents.shape[0]
        ts = list(reversed(s.timesteps.tolist()))
        ent, table, n_text, n_ip = self._prepare("inv", latents, ctx, added_cond_kwargs, B, torch.tensor(ts))
        x = ent["x"]
        x.copy_(latents.to(torch.float32))
        prev = None
        for i, t in enumerate(ts):
            ent["rb"].copy_(table[i])
            self._forward(ent, B, n_text, n_ip)
            c_x, c_e = s.inverse_coefficients(t, prev)
            prev = t
            ops.axpby(ent["eps"], x, c_x, c_e, out=x)
            if trace is not None:
                trace.append(dict(t=t, eps=ent["eps"].clone(), x=x.clone()))
        return x.clone()
