"""A whole edit request through ``B200HotPath`` on the host: DDIM inversion beside the Euler / LCM sampler, the refinement pass with
its 8-bit image hand-off, the order of the noise draws and the argument checks -- against the oracle chain, with the kernel test
double extended by CPU doubles of the VAE-only ops and the two 8-bit image ops."""
import pytest
import torch
import torch.nn.functional as F

from instructany2pix_b200.hotpath import B200HotPath
from instructany2pix_b200.sampler import B200Sampler
from instructany2pix_b200.scheduler import B200EulerDiscreteScheduler, B200LCMScheduler
from oracle.schedulers import EulerDiscreteSchedulerOracle, LCMSchedulerOracle
from oracle.vae import psnr
from tests._request_chain import build_refiner, build_vae, oracle_chain, postprocess_u8, preprocess_u8, request
from tests.test_host_unet_emu import build_pair, rel

torch.set_grad_enabled(False)
BF = torch.bfloat16


@pytest.fixture
def req(emu, monkeypatch):
    """the test double plus the ops only the VAE and the 8-bit image paths use"""
    import instructany2pix_b200.ops as real

    def gaussian_sample(moments, noise, scale=1.0):
        mean, logvar = moments.float().chunk(2, 1)
        v = mean if noise is None else mean + torch.exp(0.5 * logvar.clamp(-30, 20)) * noise
        return (v * scale).contiguous()

    def conv1x1_nchw_small(x, w, bias, scale=1.0):
        y = F.conv2d(x.float(), w.reshape(w.shape[0], -1, 1, 1)) * scale
        return y if bias is None else y + bias.reshape(1, -1, 1, 1)

    def softmax_rows(scores, scale, out=None):
        return torch.softmax(scores.float() * scale, -1).to(BF)

    def conv3x3_down_padend(x, w, cout, bias=None, out_dtype=BF):
        cin = x.shape[-1]
        w3 = w.float().reshape(cout, 3, 3, cin).permute(0, 3, 1, 2)
        y = F.conv2d(F.pad(x.float().permute(0, 3, 1, 2), (0, 1, 0, 1)), w3, bias, stride=2)
        return y.permute(0, 2, 3, 1).to(out_dtype)

    def conv_in_u8(x, w, bias, out_dtype=BF):
        return emu.conv_in(preprocess_u8(x), w, bias, out_dtype=out_dtype)

    def image_u8(y):
        return postprocess_u8(y[..., :3].permute(0, 3, 1, 2))

    def conv_out_u8(x, w32, b32):
        return image_u8(emu.conv3x3(x, w32, 32, bias=b32, out_dtype=torch.float32))

    for f in (gaussian_sample, conv1x1_nchw_small, softmax_rows, conv3x3_down_padend, conv_in_u8, image_u8, conv_out_u8):
        monkeypatch.setattr(real, f.__name__, f)
    return emu


def _draws(seed):
    g = torch.Generator().manual_seed(seed)
    return lambda shape: torch.randn(shape, generator=g)


def _close(got, ref, what):
    db = psnr(got, ref, data_range=float(ref.max() - ref.min()))
    print(f"{what}: decoded image PSNR {db:.1f} dB")
    assert db >= 35.0


@pytest.mark.parametrize("sched", ["euler", "lcm"])
def test_edit_generates_with_euler_and_lcm(req, sched):
    """inversion on DDIM (made from the generation scheduler's config), generation on the sampler's Euler / LCM scheduler"""
    o, b = build_pair(True)
    dec, enc, vae = build_vae()
    img, ctx_inv, added_inv, ctx, added, _, _ = request(1, 8)
    if sched == "euler":
        so, sb = EulerDiscreteSchedulerOracle(), B200EulerDiscreteScheduler()
    else:
        so, sb = LCMSchedulerOracle(), B200LCMScheduler()
        so.generator, sb.generator = torch.Generator().manual_seed(9), torch.Generator().manual_seed(9)
    ref, z_ref = oracle_chain(o, enc, dec, img, ctx_inv, added_inv, ctx, added, _draws(3), so)
    hot = B200HotPath(b, vae, scheduler=sb, use_cuda_graph=False)
    out, z = hot.edit(img, ctx_inv, added_inv, ctx, added, alpha=0.7, num_inference_steps=4, guidance_scale=7.5,
                      generator=torch.Generator().manual_seed(3), return_latents=True)
    print(f"{sched}: final latent rel-L2 {rel(z, z_ref):.2e}")
    _close(out, ref, f"edit, {sched} generation")
    assert hot.sampler.scheduler is sb and len(hot.sampler._graphs) == 2


def test_edit_with_refiner_matches_the_oracle_chain(req):
    o, b = build_pair(True)
    o_rf, b_rf = build_refiner()
    dec, enc, vae = build_vae()
    img, ctx_inv, added_inv, ctx, added, ctx_rf, added_rf = request(1, 8)
    ref, _ = oracle_chain(o, enc, dec, img, ctx_inv, added_inv, ctx, added, _draws(4), EulerDiscreteSchedulerOracle(),
                          refiner=(o_rf, ctx_rf, added_rf, 0.5, 6, 5.0))
    hot = B200HotPath(b, vae, scheduler=B200EulerDiscreteScheduler(), use_cuda_graph=False,
                      refiner=B200Sampler(b_rf, scheduler=B200EulerDiscreteScheduler(), use_cuda_graph=False))
    kw = dict(alpha=0.7, num_inference_steps=4, guidance_scale=7.5, refiner_ctx=ctx_rf, refiner_added=added_rf, refinement=0.5,
              refiner_steps=6, refiner_guidance_scale=5.0)
    out = hot.edit(img, ctx_inv, added_inv, ctx, added, generator=torch.Generator().manual_seed(4), **kw)
    assert out.shape == img.shape and out.dtype == torch.float32
    _close(out, ref, "edit + refiner")
    u8 = hot.edit(img, ctx_inv, added_inv, ctx, added, generator=torch.Generator().manual_seed(4), output="u8", **kw)
    assert u8.dtype == torch.uint8 and u8.shape == (1, 64, 64, 3)
    assert torch.equal(u8, postprocess_u8(out))


def test_refine_draw_order(req):
    """request i draws its encode noise and then its start noise from generator[i], as a batch of one with that generator"""
    _, b_rf = build_refiner()
    _, _, vae = build_vae()
    img, _, _, _, _, ctx_rf, added_rf = request(2, 8)
    hot = B200HotPath(None, vae, refiner=B200Sampler(b_rf, scheduler=B200EulerDiscreteScheduler(), use_cuda_graph=False))
    u8 = postprocess_u8(img)
    seeds = [7, 2]
    got = hot.refine(u8, ctx_rf, added_rf, 0.5, num_inference_steps=4, generator=[torch.Generator().manual_seed(s) for s in seeds])
    gens = [torch.Generator().manual_seed(s) for s in seeds]
    enc_noise = [torch.randn((1, 4, 8, 8), generator=g) for g in gens]
    start_noise = [torch.randn((1, 4, 8, 8), generator=g) for g in gens]
    ref = hot.refine(u8, ctx_rf, added_rf, 0.5, num_inference_steps=4, encode_noise=torch.cat(enc_noise), noise=torch.cat(start_noise))
    assert torch.equal(got, ref)
    swapped = hot.refine(u8, ctx_rf, added_rf, 0.5, num_inference_steps=4, encode_noise=torch.cat(start_noise),
                         noise=torch.cat(enc_noise))
    assert not torch.equal(got, swapped)


def test_vae_8bit_paths(req):
    """decode(output="u8") is the formula applied to decode(); encode of the 8-bit image is encode of the formula's fp32 image"""
    _, _, vae = build_vae()
    z = torch.randn(2, 4, 8, 8) * 0.9
    u8 = vae.decode(z, output="u8")
    assert u8.dtype == torch.uint8 and u8.shape == (2, 64, 64, 3)
    assert torch.equal(u8, postprocess_u8(vae.decode(z)))
    assert torch.equal(vae.encode(u8, sample=False), vae.encode(preprocess_u8(u8), sample=False))
    with pytest.raises(ValueError, match="output"):
        vae.decode(z, output="pil")
    with pytest.raises(ValueError, match="8-bit"):
        vae.encode(u8.permute(0, 3, 1, 2).contiguous())


def test_ddim_edit_calls_the_ops_of_the_parent_sequence(req, monkeypatch):
    """with a DDIM generation scheduler ``edit`` makes exactly the op calls, with the same scalar arguments, that
    encode -> invert -> start_latent -> generate -> decode on one sampler make, and returns the same images and latents"""
    import instructany2pix_b200.ops as real
    o, b = build_pair(True)
    _, _, vae = build_vae()
    img, ctx_inv, added_inv, ctx, added, _, _ = request(1, 8)
    n_enc, n_pol = torch.randn(1, 4, 8, 8), torch.randn(1, 4, 8, 8)
    log = []
    for name in dir(real):
        f = getattr(real, name)
        if callable(f) and not name.startswith("_") and not isinstance(f, type) and getattr(f, "__module__", "").startswith("tests"):
            def rec(*a, _f=f, _n=name, **k):
                log.append((_n, tuple(v for v in list(a) + list(k.values()) if isinstance(v, (int, float)))))
                return _f(*a, **k)
            monkeypatch.setattr(real, name, rec)
    out, z = B200HotPath(b, vae, use_cuda_graph=False).edit(img, ctx_inv, added_inv, ctx, added, alpha=0.7, num_inference_steps=4,
                                                            guidance_scale=7.5, noise=n_pol, encode_noise=n_enc, return_latents=True)
    calls, log[:] = list(log), []
    s = B200Sampler(b, use_cuda_graph=False)
    z0 = vae.encode(img, noise=n_enc)
    z_inv = s.invert(z0, ctx_inv, added_inv, num_inference_steps=4)
    z_ref = s.generate(s.start_latent(z_inv, alpha=0.7, noise=n_pol), ctx, added, num_inference_steps=4, guidance_scale=7.5)
    ref = vae.decode(z_ref)
    assert len(calls) > 100 and calls == log
    assert torch.equal(z, z_ref) and torch.equal(out, ref)


class _NoDeviceWork:
    encoder = None

    def __getattr__(self, name):
        raise AssertionError(f"device work before the argument checks: vae.{name}")


def test_argument_errors_before_any_device_work(req):
    _, b_rf = build_refiner()
    img, ctx_inv, added_inv, ctx, added, ctx_rf, added_rf = request(2, 8)
    rf = B200Sampler(b_rf, scheduler=B200EulerDiscreteScheduler(), use_cuda_graph=False)
    hot = B200HotPath(None, _NoDeviceWork(), refiner=rf)
    base = dict(num_inference_steps=2, refiner_ctx=ctx_rf, refiner_added=added_rf)
    edit = lambda **k: hot.edit(img, ctx_inv, added_inv, ctx, added, **{**base, **k})
    with pytest.raises(ValueError, match="refinement"):
        edit(refinement=[0.5, 0.3])
    with pytest.raises(ValueError, match="refinement"):
        edit(refinement=[0.5])
    with pytest.raises(ValueError, match="refinement"):
        edit(refinement=torch.tensor([0.5, 0.5]))
    for bad in (0.0, 1.5, float("nan"), -0.2):
        with pytest.raises(ValueError, match="refinement"):
            edit(refinement=bad)
    with pytest.raises(ValueError, match="no denoising step"):
        edit(refinement=0.01, refiner_steps=50)
    with pytest.raises(ValueError, match="output"):
        edit(output="pil")
    with pytest.raises(ValueError, match="output"):
        edit(refinement=0.5, output="uint8")
    with pytest.raises(ValueError, match="refiner_ctx"):
        edit(refinement=0.5, refiner_ctx=ctx_rf[:2])
    with pytest.raises(ValueError, match="conditioning"):
        edit(refinement=0.5, refiner_added=None)
    with pytest.raises(ValueError, match="guidance_scale"):
        edit(refinement=0.5, refiner_guidance_scale=[5.0, 5.0, 5.0])
    with pytest.raises(ValueError, match="refiner="):
        B200HotPath(None, _NoDeviceWork()).edit(img, ctx_inv, added_inv, ctx, added, refinement=0.5, **base)
    u8 = torch.zeros(2, 64, 64, 3, dtype=torch.uint8)
    with pytest.raises(ValueError, match="images_u8"):
        hot.refine(u8.float(), ctx_rf, added_rf, 0.5)
    with pytest.raises(ValueError, match="images_u8"):
        hot.refine(u8.permute(0, 3, 1, 2), ctx_rf, added_rf, 0.5)
    with pytest.raises(ValueError, match="generator"):
        hot.refine(u8, ctx_rf, added_rf, 0.5, generator=[torch.Generator()])
    with pytest.raises(ValueError, match="refinement"):
        hot.refine(u8, ctx_rf, added_rf, [0.5, 0.5])
