"""Batches of requests with per-request settings on the B200: the per-row entry points (ia2p_cfg_ddim_step_rows,
ia2p_decoupled_cross_attn_rows_bf16) against fp32 torch and against the scalar entry points bit for bit, the sampler's per-row
path against the scalar path and the oracle, and ``B200HotPath.edit`` with mixed settings against the oracle chain per request."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from instructany2pix_b200 import ops  # noqa: E402
from instructany2pix_b200.attention_processor import B200IPAttnProcessor  # noqa: E402
from instructany2pix_b200.hotpath import B200HotPath  # noqa: E402
from instructany2pix_b200.sampler import B200Sampler  # noqa: E402
from oracle import sampler as osampler  # noqa: E402
from oracle.attention import IPAttnProcessor2_0  # noqa: E402
from oracle.unet import TINY  # noqa: E402
from tests.test_host_unet_emu import build_pair, make_inputs  # noqa: E402
from tests.test_unet_parity_gpu import sdxl_pair  # noqa: E402,F401  (module fixture: the SDXL-width oracle + B200 pair)

torch.set_grad_enabled(False)
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False
DEV = "cuda"
TOL = 4e-3          # kernel gate: bf16 output rounding over an fp32 reference


def rnd(*shape, seed, dtype=torch.bfloat16):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g).to(dtype).to(DEV)


def rel(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-12)).item()


def cu(t):
    return {k: v.cuda() for k, v in t.items()} if isinstance(t, dict) else t.cuda()


# ------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("n_text,n_ip,B,N,heads", [
    (77, 4, 4, 300, 3), (80, 4, 4, 300, 3), (100, 4, 3, 256, 2),        # tcgen05 kernel (T1 = 80, 80, 112)
    (77, 4, 8, 1024, 20),                                               # c3 level-2 shape, several items per CTA
    (120, 4, 4, 300, 3), (120, 16, 3, 200, 2),                          # > 128 key columns: the mma.sync kernel
])
def test_cross_attn_rows(n_text, n_ip, B, N, heads):
    C = heads * 64
    q, kvt, kvi = rnd(B * N, C, seed=1), rnd(B * n_text, 2 * C, seed=2), rnd(B * n_ip, 2 * C, seed=3)
    s = torch.linspace(0.0, 1.2, B, device=DEV, dtype=torch.float32)          # distinct per row, row 0 text only
    out = ops.cross_attn(q, kvt, n_text, kvi, n_ip, s, B, N, heads)
    hq = q.float().reshape(B, N, heads, 64).transpose(1, 2)
    sp = lambda t, n: t.float().reshape(B, n, heads, 64).transpose(1, 2)
    ref = F.scaled_dot_product_attention(hq, sp(kvt[:, :C], n_text), sp(kvt[:, C:], n_text)) + \
        s.reshape(B, 1, 1, 1) * F.scaled_dot_product_attention(hq, sp(kvi[:, :C], n_ip), sp(kvi[:, C:], n_ip))
    assert rel(out, ref.transpose(1, 2).reshape(B * N, C)) < TOL
    rows = out.reshape(B, N, C)
    for b in range(B):             # row b is the scalar kernel's row b at that row's scale, bit for bit
        one = ops.cross_attn(q, kvt, n_text, kvi, n_ip, float(s[b]), B, N, heads).reshape(B, N, C)
        assert torch.equal(rows[b], one[b]), b
    if n_text + 16 <= 128:           # the text-only call runs the same tcgen05 kernel: scale 0 is exactly the text-only result
        text_only = ops.cross_attn(q, kvt, n_text, None, 0, 0.0, B, N, heads).reshape(B, N, C)
        assert torch.equal(rows[0], text_only[0])
    for v in (0.0, 0.6, 1.0):        # all rows equal: the scalar call
        same = ops.cross_attn(q, kvt, n_text, kvi, n_ip, torch.full((B,), v, device=DEV), B, N, heads)
        assert torch.equal(same, ops.cross_attn(q, kvt, n_text, kvi, n_ip, v, B, N, heads))


@pytest.mark.parametrize("shape,dt", [((4, 4, 16, 16), torch.float32), ((3, 4, 5, 5), torch.float32),
                                      ((4, 4, 128, 128), torch.float32), ((2, 4, 16, 16), torch.bfloat16)])
def test_cfg_ddim_step_rows(shape, dt):
    """vectorised (n % 8 == 0) and scalar (n = 100) kernels, fp32 and bf16 latents, with the duplicated next input"""
    B = shape[0]
    eps2 = rnd(2 * B, *shape[1:], seed=4, dtype=dt)
    x = rnd(*shape, seed=5, dtype=dt)
    g = torch.tensor([5.0, 7.5, 10.0, 12.0][:B], device=DEV)
    nxt = torch.empty((2 * B,) + shape[1:], device=DEV, dtype=torch.bfloat16)
    out = ops.cfg_ddim_step(eps2, x, g, 0.98, -0.11, x_in_next2=nxt)
    eu, ec = eps2.float().chunk(2)
    ref = 0.98 * x.float() + -0.11 * (eu + g.reshape(B, 1, 1, 1) * (ec - eu))
    assert rel(out, ref) < (1e-6 if dt == torch.float32 else TOL)
    assert torch.equal(nxt, torch.cat([out, out]).to(torch.bfloat16))
    for b in range(B):
        assert torch.equal(out[b], ops.cfg_ddim_step(eps2, x, float(g[b]), 0.98, -0.11)[b]), b
    assert torch.equal(ops.cfg_ddim_step(eps2, x, torch.full((B,), 7.5, device=DEV), 0.98, -0.11),
                       ops.cfg_ddim_step(eps2, x, 7.5, 0.98, -0.11))


def test_per_row_argument_checks():
    eps2, x = rnd(4, 4, 8, 8, seed=6, dtype=torch.float32), rnd(2, 4, 8, 8, seed=7, dtype=torch.float32)
    with pytest.raises(ValueError):
        ops.cfg_ddim_step(eps2, x, torch.ones(3, device=DEV), 1.0, 0.1)
    with pytest.raises(ops.IA2PError):
        ops.cfg_ddim_step(eps2, x, torch.ones(2, device=DEV, dtype=torch.float64), 1.0, 0.1)
    with pytest.raises(ops.IA2PError):
        ops.cfg_ddim_step(eps2, x, torch.ones(2), 1.0, 0.1)
    q, kvt, kvi = rnd(2 * 128, 64, seed=8), rnd(2 * 77, 128, seed=9), rnd(2 * 4, 128, seed=10)
    with pytest.raises(ValueError):
        ops.cross_attn(q, kvt, 77, kvi, 4, torch.ones(3, device=DEV), 2, 128, 1)
    with pytest.raises(ops.IA2PError):
        ops.cross_attn(q, kvt, 77, kvi, 4, torch.ones(2, device=DEV, dtype=torch.bfloat16), 2, 128, 1)
    with pytest.raises(ops.IA2PError):
        ops.cross_attn(q, kvt, 77, kvi, 4, torch.ones(2), 2, 128, 1)


# ------------------------------------------------------------------------------------------------ sampler
G = [5.0, 7.5, 12.0]
S = [0.3, 0.0, 1.0]


def _set_scale(unet, s):
    for p in unet.attn_processors.values():
        if isinstance(p, (B200IPAttnProcessor, IPAttnProcessor2_0)):
            p.scale = s


def test_equal_values_match_the_scalar_path():
    o, b = build_pair(True, device=DEV)
    lat, ctx, added = [cu(t) for t in make_inputs(TINY, B=3, L=32)]
    s0 = b._ip_state()[1]
    ref = B200Sampler(b).generate(lat, ctx, added, num_inference_steps=4, guidance_scale=7.5)
    out = B200Sampler(b).generate(lat, ctx, added, num_inference_steps=4, guidance_scale=[7.5] * 3, ip_scale=[s0] * 3)
    assert torch.equal(out, ref)


def test_mixed_rows_match_uniform_batches():
    """64x64 latent: every level's map (4096 / 1024 / 256 tokens) is a whole number of 128-row tiles per image, so no kernel
    tile spans two requests and each row of the mixed batch is bitwise the row of a uniform batch with its settings"""
    o, b = build_pair(True, device=DEV)
    lat, ctx, added = [cu(t) for t in make_inputs(TINY, B=3, L=64)]
    s0 = b._ip_state()[1]
    mixed = B200Sampler(b).generate(lat, ctx, added, num_inference_steps=3, guidance_scale=G, ip_scale=S)
    for i in range(3):
        _set_scale(b, S[i])
        uni = B200Sampler(b).generate(lat, ctx, added, num_inference_steps=3, guidance_scale=G[i])
        assert torch.equal(mixed[i], uni[i]), i
    _set_scale(b, s0)


def test_graph_replay_with_new_scales_does_not_recapture():
    o, b = build_pair(True, device=DEV)
    lat, ctx, added = [cu(t) for t in make_inputs(TINY, B=3, L=32)]
    s = B200Sampler(b)
    s.generate(lat, ctx, added, num_inference_steps=3, guidance_scale=G, ip_scale=S)
    (key, ent), = s._graphs.items()
    graph = ent["graph"]
    g2, s2 = [9.0, 4.0, 6.5], [1.0, 0.5, 0.0]
    out = s.generate(lat, ctx, added, num_inference_steps=3, guidance_scale=g2, ip_scale=s2)
    assert list(s._graphs) == [key] and s._graphs[key] is ent and ent["graph"] is graph
    fresh = B200Sampler(b).generate(lat, ctx, added, num_inference_steps=3, guidance_scale=g2, ip_scale=s2)
    assert torch.equal(out, fresh)


def test_sdxl_width_mixed_pair_against_oracle(sdxl_pair):
    """the real SDXL-base configuration at a 32x32 latent, two requests with different guidance and IP scales in one CFG batch:
    teacher-forced per-step eps of each request against the fp32 oracle running that request alone"""
    from oracle.synth import synth_input
    o, b = sdxl_pair
    B, g, sc = 2, [5.0, 12.0], [0.3, 1.0]
    lat = synth_input("mix/lat", (B, 4, 32, 32))
    ctx = synth_input("mix/ctx", (2 * B, 81, 2048))
    added = dict(text_embeds=synth_input("mix/pooled", (2 * B, 1280)),
                 time_ids=torch.tensor([[256.0, 256.0, 0.0, 0.0, 256.0, 256.0]] * 2 * B))
    traces = []
    for i in range(B):
        _set_scale(o, sc[i])
        rows = [i, B + i]
        tr = []
        osampler.generate(o, lat[i:i + 1], ctx[rows], {k: v[rows] for k, v in added.items()}, num_inference_steps=2,
                          guidance_scale=g[i], trace=tr)
        traces.append(tr)
    _set_scale(o, 1.0)
    teacher = [cu(torch.cat([traces[i][k]["x"] for i in range(B)])) for k in range(2)]
    tr_b = []
    B200Sampler(b).generate(cu(lat), cu(ctx), cu(added), num_inference_steps=2, guidance_scale=g, ip_scale=sc, trace=tr_b,
                            teacher=teacher)
    for k in range(2):
        for i in range(B):
            e = rel(tr_b[k]["eps2"][[i, B + i]], traces[i][k]["eps2"])
            print(f"SDXL width, step {k}, request {i} (g {g[i]}, scale {sc[i]}): eps rel-L2 {e:.2e}")
            assert e < 1e-2


# ------------------------------------------------------------------------------------------------ hot path
def _polar(x, y, a):
    """polar_intrtpolate (pipeline.py:295-300) for one request"""
    ll = a * x + (1 - a) * y
    return ll / ll.norm() * (a * x.norm() + (1 - a) * y.norm())


def test_edit_with_mixed_settings_and_generators():
    from oracle.vae import psnr
    from tests.test_vae_parity_gpu import SMALL, build
    dec, enc, vae = build(SMALL)
    o, b = build_pair(True, device=DEV)
    B, steps, L = 3, 4, 16
    lat, ctx, added = make_inputs(TINY, B=B, L=L)
    from oracle.synth import synth_input
    img = synth_input("mix/img", (B, 3, 8 * L, 8 * L)).clamp(-1, 1)
    ctx_inv, added_inv = ctx[B:, :77].contiguous(), {k: v[B:] for k, v in added.items()}
    alphas, seeds = [0.7, 0.4, 0.9], [21, 5, 13]
    s0 = b._ip_state()[1]
    hot = B200HotPath(b, vae)
    _, z_out = hot.edit(img.cuda(), cu(ctx_inv), cu(added_inv), cu(ctx), cu(added), alpha=alphas, num_inference_steps=steps,
                        guidance_scale=G, ip_scale=S, generator=[torch.Generator(DEV).manual_seed(k) for k in seeds],
                        return_latents=True)
    z_out = z_out.cpu()
    for i in range(B):
        gen = torch.Generator(DEV).manual_seed(seeds[i])
        n_enc = torch.randn((1, 4, L, L), generator=gen, device=DEV).cpu()          # vae.encode's draw, then start_latent's
        n_start = torch.randn((1, 4, L, L), generator=gen, device=DEV).cpu()
        z0 = enc.encode(img[i:i + 1], noise=n_enc)
        _set_scale(o, s0)                                                         # inversion: the processors' scale
        z_inv = osampler.invert(o, z0, ctx_inv[i:i + 1], {k: v[i:i + 1] for k, v in added_inv.items()}, num_inference_steps=steps)
        _set_scale(o, S[i])
        rows = [i, B + i]
        z = osampler.generate(o, _polar(z_inv, n_start, alphas[i]), ctx[rows], {k: v[rows] for k, v in added.items()},
                              num_inference_steps=steps, guidance_scale=G[i])
        ref, got = dec.decode(z), dec.decode(z_out[i:i + 1])       # both final latents through the same fp32 decoder
        db = psnr(got, ref, data_range=float(ref.max() - ref.min()))
        print(f"edit request {i} (alpha {alphas[i]}, g {G[i]}, scale {S[i]}): latent rel-L2 {rel(z_out[i:i + 1], z):.2e}, "
              f"decoded PSNR {db:.1f} dB")
        assert db >= 35.0
    _set_scale(o, s0)
