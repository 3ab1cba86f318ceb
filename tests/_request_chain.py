"""Shared pieces of the whole-request tests (``B200HotPath.edit`` / ``refine``): the models, the conditioning, the 8-bit image
formulas of diffusers 0.26 and the oracle chain an edit request is checked against."""
import numpy as np
import torch

from oracle import sampler as osampler
from oracle.schedulers import DDIMSchedulerOracle, EulerDiscreteSchedulerOracle, polar_interpolate
from oracle.synth import synth_input, synth_state_dict
from oracle.unet import TINY, OracleUNet, UNetConfig
from oracle.vae import OracleVAEDecoder, OracleVAEEncoder, to_diffusers_keys
from tests.test_host_unet_emu import make_inputs

# SDXL's VAE block structure at a quarter of the width
SMALL_VAE = dict(latent_channels=4, out_channels=3, block_out_channels=(64, 64, 128, 128), layers_per_block=2, norm_num_groups=32,
                 scaling_factor=0.13025)


def postprocess_u8(img):
    """diffusers 0.26 ``VaeImageProcessor.postprocess(output_type="pil")`` up to the PIL object: ``denormalize`` in torch, then
    ``numpy_to_pil``'s ``(images * 255).round().astype("uint8")``.  (B,3,H,W) fp32 -> uint8 (B,H,W,3)."""
    x = (img.float().cpu() / 2 + 0.5).clamp(0, 1).permute(0, 2, 3, 1).numpy()
    return torch.from_numpy((x * 255).round().astype("uint8"))


def preprocess_u8(u8):
    """diffusers 0.26 ``VaeImageProcessor.preprocess`` of a PIL image: ``np.float32(q) / 255`` (pil_to_numpy), then ``2 x - 1``
    (normalize) in torch.  uint8 (B,H,W,3) -> (B,3,H,W) fp32."""
    x = torch.from_numpy(u8.cpu().numpy().astype(np.float32) / 255.0).permute(0, 3, 1, 2).contiguous()
    return 2.0 * x - 1.0


def build_vae(device="cpu"):
    from instructany2pix_b200.vae import B200VAE
    dec, enc = OracleVAEDecoder(SMALL_VAE).eval(), OracleVAEEncoder(SMALL_VAE).eval()
    dec.load_state_dict(synth_state_dict(dec, seed=11))
    enc.load_state_dict(synth_state_dict(enc, seed=12))
    vae = B200VAE(dict(SMALL_VAE), device=device)
    sd = to_diffusers_keys(dec.state_dict(), "decoder")
    sd.update(to_diffusers_keys(enc.state_dict(), "encoder"))
    vae.load_state_dict(sd)
    return dec, enc, vae


def build_refiner(device="cpu"):
    """SDXL-refiner block layout (4 levels, attention on the middle two, text-only cross-attention, five time ids), narrow"""
    from instructany2pix_b200.unet import REFINER_CONFIG, B200UNet
    cfg = UNetConfig(**{**REFINER_CONFIG, "sample_size": 32, "block_out_channels": (64, 128, 256, 256), "attention_head_dim": (1, 2, 4, 4),
                        "transformer_layers_per_block": (2, 2, 2, 2), "cross_attention_dim": 128, "addition_time_embed_dim": 32,
                        "projection_class_embeddings_input_dim": 5 * 32 + 96})
    o = OracleUNet(cfg).eval()
    o.load_state_dict(synth_state_dict(o, 21))
    return o, B200UNet.from_module(o, device=device)


def request(B, L):
    """base conditioning (TINY: inversion rows = the positive prompt without IP tokens), refiner conditioning, input image"""
    _, ctx, added = make_inputs(TINY, B=B, L=L)
    ctx_inv, added_inv = ctx[B:, :77].contiguous(), {k: v[B:] for k, v in added.items()}
    ctx_rf = synth_input("req/rfctx", (2 * B, 77, 128))
    H = 8.0 * L
    added_rf = dict(text_embeds=synth_input("req/rfpooled", (2 * B, 96)),
                    time_ids=torch.tensor([[H, H, 0.0, 0.0, 2.5]] * B + [[H, H, 0.0, 0.0, 6.0]] * B))
    img = synth_input("req/img", (B, 3, 8 * L, 8 * L), seed=L).clamp(-1, 1)
    return img, ctx_inv, added_inv, ctx, added, ctx_rf, added_rf


def oracle_chain(o, enc, dec, img, ctx_inv, added_inv, ctx, added, draws, scheduler, steps=4, guidance_scale=7.5, alpha=0.7,
                 refiner=None):
    """One request on the fp32 oracles, drawing its noise from ``draws`` (a callable: shape -> tensor) in the reference's order:
    encode, start latent[, refiner encode, refiner start].  ``refiner``: (o_rf, ctx_rf, added_rf, strength, steps, guidance).
    -> (fp32 images, final latents)"""
    shape = (img.shape[0], 4, img.shape[2] // 8, img.shape[3] // 8)
    z0 = enc.encode(img, draws(shape))
    z_inv = osampler.invert(o, z0, ctx_inv, added_inv, num_inference_steps=steps, scheduler=DDIMSchedulerOracle())
    z_t = polar_interpolate(z_inv, draws(shape), alpha)
    z = osampler.generate(o, z_t, ctx, added, num_inference_steps=steps, guidance_scale=guidance_scale, scheduler=scheduler)
    img_out = dec.decode(z)
    if refiner is None:
        return img_out, z
    o_rf, ctx_rf, added_rf, strength, rf_steps, rf_g = refiner
    z0 = enc.encode(preprocess_u8(postprocess_u8(img_out)), draws(shape))
    z = osampler.generate(o_rf, draws(shape), ctx_rf, added_rf, num_inference_steps=rf_steps, guidance_scale=rf_g,
                          scheduler=EulerDiscreteSchedulerOracle(), init_latents=z0, strength=strength)
    return dec.decode(z), z

