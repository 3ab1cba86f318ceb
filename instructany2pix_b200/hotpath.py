"""``B200HotPath``: the denoising sequence of ``InstructAny2PixPipeline.__call__`` (pipeline.py:303-361) in one object.

What the reference does per edit request once the LLM / prompt encoders have produced their embeddings (those stay on the
reference code, SURVEY 8 "out of scope"), and which call below replaces it:

  pipeline.py:313-316   y = self.model.generate_diffusion(...)                      -> ``prior.generate_diffusion`` (B200Prior)
  pipeline.py:324-326   latent_la = mix(base, llm, y / |y| * 20); / |.| * norm       -> ``ip_context`` (caller arithmetic on 1024-vectors)
  ip_adapter.py:171-209 image_proj_model(embeds) / (zeros) -> 4 IP tokens            -> ``image_proj.get_image_embeds`` (B200ImageProj)
  ip_adapter.py:336-342 cat([text, ip_tokens], dim=1), [negative ; positive]         -> ``ip_context``
  pnp_pipeline.py:195   latents = vae.encode(image).latent_dist.sample() * sf       -> ``vae.encode``
  pnp_pipeline.py:251   DDIM inversion, N UNet forwards, no CFG                      -> ``sampler.invert``
  pipeline.py:332-336   polar_intrtpolate(latent_inv, randn_like(latent_inv), alpha) -> ``sampler.start_latent``
  ip_adapter.py:341-354 50-step (here N) CFG sampling with text + IP tokens          -> ``sampler.generate``
  sdxl_pipeline.py:859  vae.decode(latents / sf)                                     -> ``vae.decode``
  pipeline.py:358-361   piperf(image=<8-bit image>, strength=refinement)             -> ``refine`` (``edit(refinement=...)``)

Everything runs on the sm_100a kernels; tensors stay on the device between the stages.  Where the reference hands PIL images
from one pipeline to the next (the base output into the refiner), the hand-off here is the same 8-bit image as a uint8
(B, H, W, 3) tensor: the decoder writes it and the refiner's encoder reads it, bit for bit diffusers' postprocess / preprocess.
"""
from __future__ import annotations

import torch

from .sampler import B200Sampler, per_request, randn_per_request
from .scheduler import B200DDIMScheduler


class B200HotPath:
    """``refiner``: a ``B200Sampler`` over the SDXL-refiner UNet with its Euler scheduler (``piperf``, pipeline.py:128-131), needed
    by ``refine`` and ``edit(refinement=...)``; ``refiner_vae`` (default ``vae``) encodes and decodes around it."""

    def __init__(self, unet, vae, scheduler=None, prior=None, use_cuda_graph=True, image_proj=None, refiner=None, refiner_vae=None):
        self.unet, self.vae, self.prior, self.image_proj = unet, vae, prior, image_proj
        self.sampler = B200Sampler(unet, scheduler=scheduler, use_cuda_graph=use_cuda_graph)
        self.refiner = refiner
        self.refiner_vae = vae if refiner_vae is None else refiner_vae

    @torch.no_grad()
    def edit(self, image, ctx_inv, added_inv, ctx_cfg, added_cfg, alpha=0.7, num_inference_steps=25, guidance_scale=10.0,
             noise=None, encode_noise=None, generator=None, return_latents=False, ip_scale=None, refiner_ctx=None,
             refiner_added=None, refinement=None, refiner_steps=50, refiner_guidance_scale=5.0, output="float"):
        """image (B,3,H,W) in [-1,1]; ctx_inv (B,S,D) / added_inv: conditioning of the inversion pass (prompt '' in the
        reference, pipeline.py:330); ctx_cfg (2B,S',D) / added_cfg: [negative; positive] conditioning incl. the IP tokens.
        ``noise`` / ``encode_noise``: optional fixed draws (parity tests); otherwise drawn like the reference does.
        Each request may carry its own settings (pipeline.py:303-304): ``alpha``, ``guidance_scale`` and ``ip_scale`` take one
        value or B values, ``generator`` one generator or a list of B (request i draws its encode and start noise from
        ``generator[i]``).  ``ip_scale`` None keeps the processors' scale; the inversion always runs with it, as in the reference
        (pipeline.py:330 runs before ip_adapter.py:306 sets the request's scale).
        The inversion runs on a DDIM scheduler made from the generation scheduler's config (pnp_pipeline.py:133, pipeline.py:306-307);
        generation runs on the sampler's scheduler (DDIM, Euler or LCM).
        ``refinement``: one img2img strength for the whole call; when given, the refinement pass (pipeline.py:358-361) follows:
        the decoded 8-bit images go through ``refine`` with ``refiner_ctx`` (2B,77,1280) / ``refiner_added``, ``refiner_steps``
        and ``refiner_guidance_scale``, drawing from ``generator`` after the base pass.  Mixed strengths are served by
        ``B200ContinuousSampler``.
        Returns images -- fp32 (B,3,H,W) with ``output="float"``, uint8 (B,H,W,3) with ``output="u8"`` -- and, if asked, the
        final latents of the pass that made them (the refiner's when it runs)."""
        B = image.shape[0]
        per_request(alpha, B, "alpha")                        # argument errors before any GPU work
        per_request(guidance_scale, B, "guidance_scale")
        if ip_scale is not None:
            per_request(ip_scale, B, "ip_scale")
        if isinstance(generator, (list, tuple)) and len(generator) != B:
            raise ValueError(f"generator: {len(generator)} generators for {B} requests")
        _check_output(output)
        if refinement is not None:
            self._check_refine(B, refiner_ctx, refiner_added, refinement, refiner_steps, refiner_guidance_scale)
        z0 = self.vae.encode(image, noise=encode_noise, generator=generator)
        inversion = B200DDIMScheduler.from_config(self.sampler.scheduler.config)
        z_inv = self.sampler.invert(z0, ctx_inv, added_inv, num_inference_steps=num_inference_steps, scheduler=inversion)
        z_t = self.sampler.start_latent(z_inv, alpha=alpha, noise=noise, generator=generator)
        z = self.sampler.generate(z_t, ctx_cfg, added_cfg, num_inference_steps=num_inference_steps, guidance_scale=guidance_scale,
                                  ip_scale=ip_scale)
        if refinement is None:
            img = self.vae.decode(z, output=output)
            return (img, z) if return_latents else img
        return self.refine(self.vae.decode(z, output="u8"), refiner_ctx, refiner_added, refinement, refiner_steps,
                           refiner_guidance_scale, generator=generator, output=output, return_latents=return_latents)

    @torch.no_grad()
    def refine(self, images_u8, ctx_rf, added_rf, refinement, num_inference_steps=50, guidance_scale=5.0, generator=None,
               encode_noise=None, noise=None, output="float", return_latents=False):
        """The refinement pass (pipeline.py:358-361: ``piperf(image=..., strength=refinement)``, [3P]
        StableDiffusionXLImg2ImgPipeline): 8-bit images uint8 (B,H,W,3) -> ``refiner_vae.encode`` (sampled from the latent
        distribution, as diffusers 0.26's ``retrieve_latents(vae.encode(image), generator)`` does) -> the last
        int(num_inference_steps * refinement) steps of the refiner's Euler schedule from ``add_noise(z0, noise, t_start)`` with
        CFG on ctx_rf (2B,77,1280) / added_rf -> ``refiner_vae.decode``.  Draws: the encode noise first, then the start noise,
        request i from ``generator[i]`` when a list is given; ``encode_noise`` / ``noise`` inject them (parity tests).
        Returns images as ``output`` says (see ``edit``), and the final latents if asked."""
        B = images_u8.shape[0]
        if images_u8.dtype != torch.uint8 or images_u8.ndim != 4 or images_u8.shape[-1] != 3:
            raise ValueError(f"images_u8: expected uint8 (B, H, W, 3), got {images_u8.dtype} {tuple(images_u8.shape)}")
        if isinstance(generator, (list, tuple)) and len(generator) != B:
            raise ValueError(f"generator: {len(generator)} generators for {B} requests")
        _check_output(output)
        self._check_refine(B, ctx_rf, added_rf, refinement, num_inference_steps, guidance_scale)
        z0 = self.refiner_vae.encode(images_u8, noise=encode_noise, generator=generator)
        if noise is None:
            noise = randn_per_request(z0.shape, z0.device, generator)
        z = self.refiner.generate(noise, ctx_rf, added_rf, num_inference_steps=num_inference_steps, guidance_scale=guidance_scale,
                                  init_latents=z0, strength=float(refinement))
        img = self.refiner_vae.decode(z, output=output)
        return (img, z) if return_latents else img

    def _check_refine(self, B, ctx_rf, added_rf, refinement, num_inference_steps, guidance_scale):
        if self.refiner is None:
            raise ValueError("refinement needs B200HotPath(..., refiner=B200Sampler(refiner_unet, scheduler=<Euler>))")
        if not hasattr(self.refiner_vae, "encoder"):
            raise ValueError("refinement needs a VAE with its encoder (B200VAE(with_encoder=True))")
        if per_request(refinement, 1, "refinement") is not None or isinstance(refinement, bool):
            raise ValueError(f"refinement: one strength per call, got {refinement!r} (mixed strengths: B200ContinuousSampler)")
        r = float(refinement)
        if not 0.0 < r <= 1.0:
            raise ValueError(f"refinement: strength must be in (0, 1], got {r}")
        if int(num_inference_steps * r) < 1:
            raise ValueError(f"refinement {r} of {num_inference_steps} steps leaves no denoising step")
        if ctx_rf is None or added_rf is None:
            raise ValueError("refinement needs the refiner's conditioning (refiner_ctx, refiner_added)")
        if ctx_rf.shape[0] != 2 * B:
            raise ValueError(f"refiner_ctx: {ctx_rf.shape[0]} rows for {B} requests (expected [negative; positive] = {2 * B})")
        per_request(guidance_scale, B, "guidance_scale")

    @torch.no_grad()
    def ip_context(self, text_ctx_cfg, llm_embed, prior_embed=None, base_embed=None, h=(0.0, 0.4, 1.0), norm=20.0,
                   mode="global"):
        """The conditioning hand-over of an edit request: text_ctx_cfg (2B, 77, D) = [negative ; positive] prompt embeddings,
        llm_embed (B, 1024) = the LLM's image embedding, prior_embed (B, 1024) = ``generate_diffusion`` output (None: the
        LLM embedding is used as it is), base_embed (B, 1024) optional.  Mixes like pipeline.py:324-326
        (``base h0 + llm h1 + y/|y| 20 h2``, renormalised to ``norm``; plain torch on B x 1024 numbers, the caller's
        arithmetic in the reference), projects to IP tokens with ``B200ImageProj`` (uncond = projector(zeros)) and appends them:
        -> (2B, 77 + T, D) for ``B200Sampler.generate``.
        Per-request mixing: ``h`` of shape (B, 3) and ``norm`` of shape (B,) give request i the weights ``h[i]`` and ``norm[i]``."""
        B = llm_embed.shape[0]
        e = llm_embed.reshape(B, -1).float()
        h = _mix_weights(h, B, e.device)
        norm = norm if per_request(norm, B, "norm") is None else torch.as_tensor(norm, dtype=torch.float32).reshape(B, 1).to(e.device)
        if prior_embed is not None:
            y = prior_embed.reshape(B, -1).float().to(e.device)
            e = e * h[1] + y / y.norm(dim=-1, keepdim=True) * 20.0 * h[2]
            if base_embed is not None:
                e = e + base_embed.reshape(B, -1).float() * h[0]
        e = e / e.norm(dim=-1, keepdim=True) * norm
        cond, uncond = self.image_proj.get_image_embeds(clip_image_embeds=e, mode=mode)
        ip = torch.cat([uncond, cond], dim=0).to(text_ctx_cfg.dtype)
        return torch.cat([text_ctx_cfg, ip], dim=1).contiguous()

    @torch.no_grad()
    def generate(self, latents, ctx_cfg, added_cfg, num_inference_steps=50, guidance_scale=10.0, ip_scale=None):
        """text/IP-conditioned generation from given start latents (ip_adapter.py:341-354 + sdxl_pipeline.py:859-871).
        ``guidance_scale`` / ``ip_scale``: one value or one per request, as in ``edit``."""
        return self.vae.decode(self.sampler.generate(latents, ctx_cfg, added_cfg, num_inference_steps=num_inference_steps,
                                                     guidance_scale=guidance_scale, ip_scale=ip_scale))


def _check_output(output):
    if output not in ("float", "u8"):
        raise ValueError(f"output: 'float' or 'u8', got {output!r}")


def _mix_weights(h, B, device):
    """``h`` as (h0, h1, h2): three floats for the batch, or three (B, 1) columns when ``h`` has shape (B, 3)"""
    t = torch.as_tensor(h, dtype=torch.float32)
    if t.ndim == 1 and t.shape[0] == 3:
        return h
    if t.shape != (B, 3):
        raise ValueError(f"h: expected 3 weights or shape ({B}, 3), got {tuple(t.shape)}")
    if not bool(torch.isfinite(t).all()):
        raise ValueError("h: non-finite weight")
    t = t.to(device)
    return t[:, 0:1], t[:, 1:2], t[:, 2:3]
