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

Everything runs on the sm_100a kernels; tensors stay on the device between the stages.
"""
from __future__ import annotations

import torch

from .sampler import B200Sampler, per_request


class B200HotPath:
    def __init__(self, unet, vae, scheduler=None, prior=None, use_cuda_graph=True, image_proj=None):
        self.unet, self.vae, self.prior, self.image_proj = unet, vae, prior, image_proj
        self.sampler = B200Sampler(unet, scheduler=scheduler, use_cuda_graph=use_cuda_graph)

    @torch.no_grad()
    def edit(self, image, ctx_inv, added_inv, ctx_cfg, added_cfg, alpha=0.7, num_inference_steps=25, guidance_scale=10.0,
             noise=None, encode_noise=None, generator=None, return_latents=False, ip_scale=None):
        """image (B,3,H,W) in [-1,1]; ctx_inv (B,S,D) / added_inv: conditioning of the inversion pass (prompt '' in the
        reference, pipeline.py:330); ctx_cfg (2B,S',D) / added_cfg: [negative; positive] conditioning incl. the IP tokens.
        ``noise`` / ``encode_noise``: optional fixed draws (parity tests); otherwise drawn like the reference does.
        Each request may carry its own settings (pipeline.py:303-304): ``alpha``, ``guidance_scale`` and ``ip_scale`` take one
        value or B values, ``generator`` one generator or a list of B (request i draws its encode and start noise from
        ``generator[i]``).  ``ip_scale`` None keeps the processors' scale; the inversion always runs with it, as in the reference
        (pipeline.py:330 runs before ip_adapter.py:306 sets the request's scale).
        Returns images (B,3,H,W) fp32 (and the final latents if asked)."""
        B = image.shape[0]
        per_request(alpha, B, "alpha")                        # argument errors before any GPU work
        per_request(guidance_scale, B, "guidance_scale")
        if ip_scale is not None:
            per_request(ip_scale, B, "ip_scale")
        if isinstance(generator, (list, tuple)) and len(generator) != B:
            raise ValueError(f"generator: {len(generator)} generators for {B} requests")
        z0 = self.vae.encode(image, noise=encode_noise, generator=generator)
        z_inv = self.sampler.invert(z0, ctx_inv, added_inv, num_inference_steps=num_inference_steps)
        z_t = self.sampler.start_latent(z_inv, alpha=alpha, noise=noise, generator=generator)
        z = self.sampler.generate(z_t, ctx_cfg, added_cfg, num_inference_steps=num_inference_steps, guidance_scale=guidance_scale,
                                  ip_scale=ip_scale)
        img = self.vae.decode(z)
        return (img, z) if return_latents else img

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
