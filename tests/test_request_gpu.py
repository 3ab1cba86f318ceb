"""A whole edit request on the B200: the two 8-bit image kernels bit for bit against diffusers' formulas, the VAE's 8-bit paths,
``edit`` with DDIM bitwise the sequence it replaces, Euler generation and the refinement pass against the oracle chains, and no
host synchronisation inside the sampling loops."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from instructany2pix_b200 import ops  # noqa: E402
from instructany2pix_b200.hotpath import B200HotPath  # noqa: E402
from instructany2pix_b200.sampler import B200Sampler  # noqa: E402
from instructany2pix_b200.scheduler import B200EulerDiscreteScheduler  # noqa: E402
from oracle.schedulers import EulerDiscreteSchedulerOracle  # noqa: E402
from oracle.vae import psnr  # noqa: E402
from tests._poison import is_poison, poisoned  # noqa: E402
from tests._request_chain import build_refiner, build_vae, oracle_chain, postprocess_u8, preprocess_u8, request  # noqa: E402
from tests.test_host_unet_emu import build_pair  # noqa: E402

torch.set_grad_enabled(False)
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False
SIZES = [(1, 128), (3, 128), (1, 1024), (3, 1024)]


def cu(t):
    return {k: v.cuda() for k, v in t.items()} if isinstance(t, dict) else t.cuda()


def _boundaries():
    """fp32 inputs v for which clamp(v / 2 + 0.5, 0, 1) * 255 is exactly k + 0.5 (ties of the rounding), and their neighbours"""
    out = []
    for k in range(255):
        c0 = np.float32((k + 0.5) / 255)
        for c in (c0 + np.arange(-4, 5, dtype=np.float32) * np.spacing(c0)).astype(np.float32):
            if np.float32(c * np.float32(255)) != np.float32(k + 0.5):
                continue
            v = np.float32(np.float32(2) * (c - np.float32(0.5)))
            out.extend(np.nextafter(v, np.float32(np.inf) * s) for s in (-1, 1))
            out.append(v)
    return torch.from_numpy(np.array(out, dtype=np.float32))


def _image_inputs(B, S, seed):
    """[B, S, S, 32] fp32 as the padded conv_out writes it: random values, +-1, values outside [-1, 1], +-inf, the rounding ties"""
    g = torch.Generator().manual_seed(seed)
    y = torch.randn(B, S, S, 32, generator=g) * 1.5
    flat = y[..., :3].reshape(-1)
    special = torch.cat([torch.tensor([1.0, -1.0, 3.0, -3.0, 1e30, -1e30, float("inf"), float("-inf"), 0.0, -0.0]), _boundaries()])
    pos = torch.randperm(flat.numel(), generator=g)[: 40 * special.numel()]
    vals = special.repeat(40)
    y3 = y[..., :3].reshape(-1).clone()
    y3[pos] = vals
    y[..., :3] = y3.reshape(B, S, S, 3)
    return y


@pytest.mark.parametrize("B,S", SIZES)
def test_image_u8_bitwise(B, S):
    y = _image_inputs(B, S, seed=S + B)
    assert int((y[..., :3] == 1.0).sum()) > 0
    ref = postprocess_u8(y[..., :3].permute(0, 3, 1, 2))
    with poisoned():
        out = ops.image_u8(y.cuda())
        again = ops.image_u8(y.cuda())
    assert out.dtype == torch.uint8 and out.shape == (B, S, S, 3)
    bad = (out.cpu() != ref).sum().item()
    print(f"image_u8 {B}x{S}^2: {bad} of {ref.numel()} bytes differ from the numpy formula")
    assert torch.equal(out.cpu(), ref) and torch.equal(again, out)
    nan = torch.full((1, 4, 4, 32), float("nan"))
    assert int(ops.image_u8(nan.cuda()).max()) == 0                       # NaN -> 0
    assert not is_poison(out[..., :1]).all()


@pytest.mark.parametrize("B,S", SIZES)
def test_conv_in_u8_bitwise(B, S):
    """an identity tap (weight 1 on the centre, bias 0) returns the kernel's fp32 input exactly: every one of the 256 values
    maps to np.float32(q) / 255 * 2 - 1; with real weights the conv equals ops.conv_in on the formula's fp32 image"""
    g = torch.Generator().manual_seed(S + B)
    u8 = torch.randint(0, 256, (B, S, S, 3), generator=g, dtype=torch.uint8)
    u8.view(-1)[:768] = torch.arange(256, dtype=torch.uint8).repeat_interleave(3)      # all 256 values in every channel
    ident = torch.zeros(8, 3, 3, 3)
    for c in range(3):
        ident[c, c, 1, 1] = 1.0
    f32 = preprocess_u8(u8)
    with poisoned():
        got = ops.conv_in_u8(u8.cuda(), ident.cuda(), torch.zeros(8).cuda(), out_dtype=torch.float32)
    assert torch.equal(got[..., :3].cpu(), f32.permute(0, 2, 3, 1))
    w, b = torch.randn(128, 3, 3, 3, generator=g) * 0.2, torch.randn(128, generator=g)
    for dt in (torch.float32, torch.bfloat16):
        with poisoned():
            out = ops.conv_in_u8(u8.cuda(), w.cuda(), b.cuda(), out_dtype=dt)
            again = ops.conv_in_u8(u8.cuda(), w.cuda(), b.cuda(), out_dtype=dt)
        ref = ops.conv_in(f32.cuda(), w.cuda(), b.cuda(), out_dtype=dt)
        assert torch.equal(out, ref) and torch.equal(again, out)


@pytest.mark.parametrize("B,S", SIZES)
def test_vae_8bit_paths(B, S):
    """decode(output="u8") == decode() then the formula; encode(u8) == encode(the formula's fp32 image)"""
    _, _, vae = build_vae(device="cuda")
    L = S // 8
    z = torch.randn(B, 4, L, L, generator=torch.Generator().manual_seed(L)) * 0.9
    with poisoned():
        u8 = vae.decode(z.cuda(), output="u8")
        again = vae.decode(z.cuda(), output="u8")
    ref = postprocess_u8(vae.decode(z.cuda()))
    assert u8.shape == (B, S, S, 3) and torch.equal(u8.cpu(), ref) and torch.equal(again, u8)
    with poisoned():
        lat = vae.encode(u8, sample=False)
        lat2 = vae.encode(u8, sample=False)
    assert torch.equal(lat, vae.encode(preprocess_u8(u8).cuda(), sample=False)) and torch.equal(lat2, lat)


def test_ddim_edit_is_the_parent_sequence():
    """DDIM generation: edit's images and latents are torch.equal to encode, invert, start_latent, generate, decode on one sampler"""
    o, b = build_pair(True, device="cuda")
    _, _, vae = build_vae(device="cuda")
    img, ctx_inv, added_inv, ctx, added, _, _ = request(2, 16)
    n_enc, n_pol = torch.randn(2, 4, 16, 16).cuda(), torch.randn(2, 4, 16, 16).cuda()
    out, z = B200HotPath(b, vae).edit(cu(img), cu(ctx_inv), cu(added_inv), cu(ctx), cu(added), alpha=0.7, num_inference_steps=4,
                                      guidance_scale=7.5, noise=n_pol, encode_noise=n_enc, return_latents=True)
    s = B200Sampler(b)
    z_inv = s.invert(vae.encode(cu(img), noise=n_enc), cu(ctx_inv), cu(added_inv), num_inference_steps=4)
    z_ref = s.generate(s.start_latent(z_inv, alpha=0.7, noise=n_pol), cu(ctx), cu(added), num_inference_steps=4, guidance_scale=7.5)
    assert torch.equal(z, z_ref) and torch.equal(out, vae.decode(z_ref))


def _models():
    o, b = build_pair(True, device="cuda")
    o_rf, b_rf = build_refiner(device="cuda")
    dec, enc, vae = build_vae(device="cuda")
    return o, b, o_rf, b_rf, dec, enc, vae


def _cuda_draws(seed):
    g = torch.Generator("cuda").manual_seed(seed)
    return lambda shape: torch.randn(shape, generator=g, device="cuda").cpu()


@pytest.mark.parametrize("refine", [False, True], ids=["euler", "euler+refiner"])
def test_edit_against_the_oracle_chain(refine):
    o, b, o_rf, b_rf, dec, enc, vae = _models()
    img, ctx_inv, added_inv, ctx, added, ctx_rf, added_rf = request(1, 16)
    rf = (o_rf, ctx_rf, added_rf, 0.5, 8, 5.0) if refine else None
    ref, _ = oracle_chain(o, enc, dec, img, ctx_inv, added_inv, ctx, added, _cuda_draws(5), EulerDiscreteSchedulerOracle(), refiner=rf)
    hot = B200HotPath(b, vae, scheduler=B200EulerDiscreteScheduler(), refiner=B200Sampler(b_rf, scheduler=B200EulerDiscreteScheduler()))
    kw = dict(refiner_ctx=cu(ctx_rf), refiner_added=cu(added_rf), refinement=0.5, refiner_steps=8, refiner_guidance_scale=5.0) if refine else {}
    out = hot.edit(cu(img), cu(ctx_inv), cu(added_inv), cu(ctx), cu(added), alpha=0.7, num_inference_steps=4, guidance_scale=7.5,
                   generator=torch.Generator("cuda").manual_seed(5), **kw).cpu()
    db = psnr(out, ref, data_range=float(ref.max() - ref.min()))
    print(f"edit ({'Euler + refiner' if refine else 'Euler'}) vs the oracle chain: decoded image PSNR {db:.1f} dB")
    assert db >= 35.0


def test_no_host_sync_inside_the_sampling_loops(monkeypatch):
    """Euler edit + refinement with CUDA graphs: from the first UNet forward of each loop until the loop returns (every step after
    the first entirely, and the first step's forward and update) no operation may synchronise with the host"""
    o, b, o_rf, b_rf, dec, enc, vae = _models()
    img, ctx_inv, added_inv, ctx, added, ctx_rf, added_rf = request(2, 16)
    hot = B200HotPath(b, vae, scheduler=B200EulerDiscreteScheduler(), refiner=B200Sampler(b_rf, scheduler=B200EulerDiscreteScheduler()))
    run = lambda: hot.edit(cu(img), cu(ctx_inv), cu(added_inv), cu(ctx), cu(added), num_inference_steps=4, refiner_ctx=cu(ctx_rf),
                           refiner_added=cu(added_rf), refinement=0.5, refiner_steps=8, generator=torch.Generator("cuda").manual_seed(1),
                           output="u8")
    first = run()                                              # captures the three graphs
    forward, seen = B200Sampler._forward, []

    def checked_forward(self, *a, **k):
        torch.cuda.set_sync_debug_mode("error")
        seen.append(1)
        return forward(self, *a, **k)
    monkeypatch.setattr(B200Sampler, "_forward", checked_forward)
    for name in ("generate", "invert"):
        def loop(self, *a, _f=getattr(B200Sampler, name), **k):
            try:
                return _f(self, *a, **k)
            finally:
                torch.cuda.set_sync_debug_mode(0)
        monkeypatch.setattr(B200Sampler, name, loop)
    out = run()
    torch.cuda.set_sync_debug_mode(0)
    assert len(seen) == 4 + 4 + 4 and torch.equal(out, first)
