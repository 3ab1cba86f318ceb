"""Batches of requests with per-request settings (guidance scale, IP scale, alpha, mixing weights, seeds): the host logic of
``B200Sampler`` / ``B200HotPath`` against the oracle run one request at a time, with the kernel test double."""
import pytest
import torch

from instructany2pix_b200.hotpath import B200HotPath
from instructany2pix_b200.image_proj import B200ImageProj
from instructany2pix_b200.sampler import B200Sampler, randn_per_request
from oracle import sampler as osampler
from oracle.attention import ImageProjModel, IPAttnProcessor2_0
from oracle.synth import synth_input, synth_state_dict
from oracle.unet import TINY
from tests.test_host_unet_emu import build_pair, make_inputs, rel

torch.set_grad_enabled(False)

G = [5.0, 7.5, 12.0]
S = [0.3, 0.0, 1.0]


@pytest.fixture
def mixed(emu, monkeypatch):
    """the test double, extended to the per-row forms: a tensor ``g`` / ``ip_scale`` holds one value per batch row"""
    import instructany2pix_b200.ops as real

    def cfg_ddim_step(eps2, x, g, c_x, c_e, x_out=None, x_in_next2=None):
        if isinstance(g, torch.Tensor):
            assert g.dtype == torch.float32 and g.shape == (x.shape[0],)
            g = g.reshape(-1, *([1] * (x.ndim - 1)))
        return emu.cfg_ddim_step(eps2, x, g, c_x, c_e, x_out=x_out, x_in_next2=x_in_next2)

    def cross_attn(q, kv_text, n_text, kv_ip, n_ip, ip_scale, batch, n_q, heads, out=None):
        if isinstance(ip_scale, torch.Tensor):
            assert ip_scale.dtype == torch.float32 and ip_scale.shape == (batch,)
            ip_scale = ip_scale.reshape(batch, 1, 1, 1)                    # [batch, heads, n_q, 64] attention output
        return emu.cross_attn(q, kv_text, n_text, kv_ip, n_ip, ip_scale, batch, n_q, heads, out=out)

    monkeypatch.setattr(real, "cfg_ddim_step", cfg_ddim_step)
    monkeypatch.setattr(real, "cross_attn", cross_attn)
    return emu


def _one(lat, ctx, added, i, B):
    rows = [i, B + i]
    return lat[i:i + 1], ctx[rows], {k: v[rows] for k, v in added.items()}


def _set_oracle_scale(o, s):
    for p in o.attn_processors.values():
        if isinstance(p, IPAttnProcessor2_0):
            p.scale = s


def test_mixed_batch_matches_each_request_alone(mixed):
    o, b = build_pair(True)
    B = 3
    lat, ctx, added = make_inputs(TINY, B=B, L=8)
    refs, traces = [], []
    for i in range(B):
        _set_oracle_scale(o, S[i])
        tr = []
        l1, c1, a1 = _one(lat, ctx, added, i, B)
        refs.append(osampler.generate(o, l1, c1, a1, num_inference_steps=4, guidance_scale=G[i], trace=tr))
        traces.append(tr)
    teacher = [torch.cat([traces[i][k]["x"] for i in range(B)]) for k in range(4)]
    s = B200Sampler(b, use_cuda_graph=False)
    tr_b = []
    s.generate(lat, ctx, added, num_inference_steps=4, guidance_scale=G, ip_scale=S, trace=tr_b, teacher=teacher)
    for k in range(4):
        for i in range(B):
            eps2 = tr_b[k]["eps2"][[i, B + i]]
            assert rel(eps2, traces[i][k]["eps2"]) < 1.5e-2, (k, i)
    out = B200Sampler(b, use_cuda_graph=False).generate(lat, ctx, added, num_inference_steps=4, guidance_scale=torch.tensor(G),
                                                         ip_scale=S)
    for i in range(B):
        assert rel(out[i:i + 1], refs[i]) < 1.5e-2, i


def test_per_request_ip_scale_keeps_the_graph_entry(mixed):
    o, b = build_pair(True)
    lat, ctx, added = make_inputs(TINY, B=2, L=8)
    s = B200Sampler(b, use_cuda_graph=False)
    s.generate(lat, ctx, added, num_inference_steps=2, guidance_scale=[5.0, 9.0], ip_scale=[0.2, 0.9])
    (key, ent), = s._graphs.items()
    assert "per-row" in key
    assert ent["ips"].tolist() == pytest.approx([0.2, 0.9, 0.2, 0.9])          # [uncond; cond] rows
    s.generate(lat, ctx, added, num_inference_steps=2, guidance_scale=7.0, ip_scale=[1.0, 0.0])
    assert list(s._graphs) == [key] and s._graphs[key] is ent
    assert ent["ips"].tolist() == [1.0, 0.0, 1.0, 0.0]
    s.generate(lat, ctx, added, num_inference_steps=2, guidance_scale=7.0, ip_scale=0.5)   # one value: same per-row entry
    assert list(s._graphs) == [key] and ent["ips"].tolist() == [0.5] * 4


def test_scalar_settings_keep_the_processor_scale_key(mixed):
    """plain floats keep today's graph key (the processors' scale value) and no per-row buffer"""
    o, b = build_pair(True)
    lat, ctx, added = make_inputs(TINY, B=2, L=8)
    s = B200Sampler(b, use_cuda_graph=False)
    s.generate(lat, ctx, added, num_inference_steps=2, guidance_scale=7.5)
    (key, ent), = s._graphs.items()
    assert key[7] == b._ip_state()[1] and ent["ips"] is None and ent["g"] is None


def _hot(monkeypatch):
    o = ImageProjModel(cross_attention_dim=128, clip_embeddings_dim=64, clip_extra_context_tokens=4)
    o.load_state_dict(synth_state_dict(o, 7))
    import instructany2pix_b200.hotpath as hp
    monkeypatch.setattr(hp, "B200Sampler", lambda *a, **k: None)
    return B200HotPath(None, None, image_proj=B200ImageProj.from_module(o.eval(), device="cpu"))


def test_ip_context_per_request_h_and_norm(mixed, monkeypatch):
    hot = _hot(monkeypatch)
    B = 3
    text = synth_input("mix/text", (2 * B, 77, 128))
    llm, y, base = synth_input("mix/llm", (B, 64)), synth_input("mix/y", (B, 1, 64)), synth_input("mix/base", (B, 64))
    h = [(0.2, 0.4, 1.0), (0.0, 1.0, 0.5), (0.5, 0.1, 2.0)]
    norm = [20.0, 10.0, 35.0]
    ctx = hot.ip_context(text, llm, prior_embed=y, base_embed=base, h=torch.tensor(h), norm=torch.tensor(norm))
    for i in range(B):
        one = hot.ip_context(text[[i, B + i]], llm[i:i + 1], prior_embed=y[i:i + 1], base_embed=base[i:i + 1], h=h[i], norm=norm[i])
        torch.testing.assert_close(ctx[[i, B + i]], one, rtol=1e-6, atol=1e-6)
    with pytest.raises(ValueError, match="h"):
        hot.ip_context(text, llm, prior_embed=y, h=torch.ones(2, 3))
    with pytest.raises(ValueError, match="h"):
        hot.ip_context(text, llm, prior_embed=y, h=torch.tensor([[0.1, 0.2, float("nan")]] * B))
    with pytest.raises(ValueError, match="norm"):
        hot.ip_context(text, llm, prior_embed=y, norm=[20.0, 20.0])
    with pytest.raises(ValueError, match="norm"):
        hot.ip_context(text, llm, prior_embed=y, norm=[20.0, float("inf"), 20.0])


def test_generator_list_gives_each_request_its_own_draws(mixed):
    o, b = build_pair(True)
    s = B200Sampler(b, use_cuda_graph=False)
    seeds, alphas = [3, 11, 7], [0.7, 0.2, 0.95]
    x = torch.randn(3, 4, 8, 8)
    gens = [torch.Generator().manual_seed(k) for k in seeds]
    noise = randn_per_request((3, 4, 8, 8), "cpu", gens)
    out = s.start_latent(x, alpha=alphas, generator=[torch.Generator().manual_seed(k) for k in seeds])
    for i, k in enumerate(seeds):
        assert torch.equal(noise[i:i + 1], torch.randn((1, 4, 8, 8), generator=torch.Generator().manual_seed(k)))
        alone = s.start_latent(x[i:i + 1], alpha=alphas[i], generator=torch.Generator().manual_seed(k))
        assert torch.equal(out[i:i + 1], alone)
    with pytest.raises(ValueError, match="generator"):
        randn_per_request((3, 4, 8, 8), "cpu", gens[:2])


def test_argument_errors(mixed):
    o, b = build_pair(True)
    lat, ctx, added = make_inputs(TINY, B=2, L=8)
    s = B200Sampler(b, use_cuda_graph=False)
    gen = lambda **k: s.generate(lat, ctx, added, num_inference_steps=2, **k)
    with pytest.raises(ValueError, match="guidance_scale"):
        gen(guidance_scale=[5.0, 6.0, 7.0])
    with pytest.raises(ValueError, match="guidance_scale"):
        gen(guidance_scale=torch.tensor([5.0]))
    with pytest.raises(ValueError, match="guidance_scale"):
        gen(guidance_scale=[5.0, float("nan")])
    with pytest.raises(ValueError, match="ip_scale"):
        gen(ip_scale=[0.5])
    with pytest.raises(ValueError, match="ip_scale"):
        gen(ip_scale=[0.5, float("inf")])
    with pytest.raises(ValueError, match="ip_scale"):
        gen(ip_scale=float("nan"))
    with pytest.raises(ValueError, match="alpha"):
        s.start_latent(lat, alpha=[0.5, 0.6, 0.7])
    # plain processors on attn2 (IPAdapter.disable()): no IP branch to scale
    o0, b0 = build_pair(False)
    ctx77 = ctx[:, :77].contiguous()
    with pytest.raises(ValueError, match="IP-adapter"):
        B200Sampler(b0, use_cuda_graph=False).generate(lat, ctx77, added, num_inference_steps=2, ip_scale=[0.5, 0.5])
    # B200HotPath.edit rejects before any device work (the VAE is never reached)
    hot = B200HotPath(b, None)
    img = torch.zeros(2, 3, 64, 64)
    kw = dict(ctx_inv=ctx[2:, :77], added_inv=added, ctx_cfg=ctx, added_cfg=added, num_inference_steps=2)
    with pytest.raises(ValueError, match="generator"):
        hot.edit(img, generator=[torch.Generator()], **kw)
    with pytest.raises(ValueError, match="alpha"):
        hot.edit(img, alpha=[0.7], **kw)
    with pytest.raises(ValueError, match="guidance_scale"):
        hot.edit(img, guidance_scale=[7.0, float("nan")], **kw)
    with pytest.raises(ValueError, match="ip_scale"):
        hot.edit(img, ip_scale=[0.1, 0.2, 0.3], **kw)
