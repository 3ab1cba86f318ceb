"""SDXL prompt encoders on the B200: causal attention and the GELU / quick-GELU GEMM epilogues against fp32 torch, the full-width
CLIP-L and OpenCLIP-bigG towers (synthetic weights) against the fp32 restatement (oracle/clip_text.py), and encode_prompt feeding
B200Sampler.generate against the oracle chain."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from instructany2pix_b200 import ops
from oracle import clip_text as O
from oracle.synth import synth_state_dict

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)
DEV = "cuda"


def rel(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm()).item()


@pytest.mark.parametrize("T", [2, 7, 77, 128])
@pytest.mark.parametrize("heads", [12, 16, 20])
@pytest.mark.parametrize("n", [1, 2, 16])
def test_causal_self_attn(T, heads, n):
    g = torch.Generator().manual_seed(T * 1000 + heads * 10 + n)
    C = heads * 64
    qkv = torch.randn(n * T, 3 * C, generator=g).to(torch.bfloat16)
    q, k, v = [t.float().reshape(n, T, heads, 64).transpose(1, 2) for t in qkv.split(C, dim=1)]
    ref = F.scaled_dot_product_attention(q, k, v, is_causal=True).transpose(1, 2).reshape(n * T, C)
    out = ops.causal_self_attn(qkv.to(DEV), n, T, heads)
    assert rel(out.cpu(), ref) <= 4e-3


@pytest.mark.parametrize("M", [154, 1232])
@pytest.mark.parametrize("act", ["gelu", "quick_gelu"])
@pytest.mark.parametrize("fold", [False, True])
def test_gemm_activation_epilogues(M, act, fold):
    from instructany2pix_b200.unet import _fold_ln
    g = torch.Generator().manual_seed(M + 7 * fold)
    K, N = 768, 3072
    a = (torch.randn(M, K, generator=g) * 2 + 0.3).to(torch.bfloat16)
    w = ((torch.rand(N, K, generator=g) * 2 - 1) * K ** -0.5).to(torch.bfloat16)
    b = torch.randn(N, generator=g) * 0.1
    fn = (lambda x: x * torch.sigmoid(1.702 * x)) if act == "quick_gelu" else F.gelu
    if fold:
        ln = nn.LayerNorm(K)
        ln.weight.data = 1 + 0.1 * torch.randn(K, generator=g)
        ln.bias.data = 0.1 * torch.randn(K, generator=g)
        ref = fn(ln(a.float()) @ w.float().t() + b)
        wp, c1, c2, eps = _fold_ln(w, b, ln)
        af = a.float()
        stats = torch.stack([af.sum(1), (af * af).sum(1)], -1)[:, None]          # producer format, one part per row
        out = ops.gemm(a.to(DEV), wp.to(DEV), bias=c2.to(DEV), ln=(stats.to(DEV), c1.to(DEV), eps), act=act)
    else:
        ref = fn(a.float() @ w.float().t() + b)
        out = ops.gemm(a.to(DEV), w.to(DEV), bias=b.to(DEV), act=act)
    assert out.dtype == torch.bfloat16 and rel(out.cpu(), ref) <= 4e-3
    with pytest.raises(ops.IA2PError):
        ops.gemm(a.to(DEV), w.to(DEV), bias=b.to(DEV), act=act, out_dtype=torch.float32)


def test_embedding_out_of_range_id_gives_nan_row():
    tok = (torch.randn(100, 128) * 0.02).to(torch.bfloat16).to(DEV)
    pos = (torch.randn(77, 128) * 0.02).to(DEV)
    ids = torch.randint(0, 100, (2, 77)).to(DEV)
    ids[1, 5], ids[0, 9] = 100, -3
    x, xb, st = ops.clip_embed(ids, tok, pos, want_ln=True)
    torch.cuda.synchronize()
    bad = torch.zeros(2 * 77, dtype=torch.bool)
    bad[77 + 5] = bad[9] = True
    assert x[bad.to(DEV)].isnan().all() and xb[bad.to(DEV)].float().isnan().all() and st[bad.to(DEV)].isnan().all()
    ref = tok.float()[ids.clamp(0, 99)] + pos[None]
    good = ~bad.to(DEV)
    assert torch.equal(x[good], ref.reshape(-1, 128)[good])
    assert rel(st[good, 0, 0], x[good].sum(1)) < 1e-5
    with pytest.raises(ops.IA2PError):
        ops.clip_embed(ids.cpu(), tok, pos)                               # host ids are range-checked up front


# ------------------------------------------------------------------------------------------------ full-width towers
def _tower(cfg, proj, seed):
    from instructany2pix_b200.text_encoder import B200CLIPTextModel, B200CLIPTextModelWithProjection
    sd = synth_state_dict(O.state_dict_shapes(cfg, proj), seed=seed)
    m = (B200CLIPTextModelWithProjection if proj else B200CLIPTextModel)(cfg.hf_kwargs(), device=DEV)
    m.load_state_dict(sd)
    return m, {k: v.to(DEV) for k, v in sd.items()}


@pytest.fixture(scope="module")
def full_towers():
    tl, sl = _tower(O.CLIP_L, False, seed=21)
    tg, sg = _tower(O.BIGG, True, seed=22)
    ids = [O.make_ids("full/l", 2, 77, O.PAD_CLIP_L), O.make_ids("full/g", 2, 77, O.PAD_BIGG)]
    return dict(l=(tl, sl, O.CLIP_L, False), g=(tg, sg, O.BIGG, True), ids=ids)


@pytest.mark.parametrize("which", ["l", "g"])
def test_full_width_tower_vs_restatement(full_towers, which):
    m, sd, cfg, proj = full_towers[which]
    ids = full_towers["ids"][0 if which == "l" else 1].to(DEV)
    ref = O.forward(sd, cfg, ids, with_projection=proj)
    out = m(ids, output_hidden_states=True)
    assert len(out.hidden_states) == cfg.num_hidden_layers + 1
    e_hs, e_last = rel(out.hidden_states[-2], ref["hidden_states"][-2]), rel(out.last_hidden_state, ref["last_hidden_state"])
    print(f"[clip {which}] hidden_states[-2] rel-L2 {e_hs:.2e}, last_hidden_state {e_last:.2e}")
    assert e_hs <= 1e-2 and e_last <= 1e-2
    if proj:
        cos = F.cosine_similarity(out.text_embeds.float(), ref["text_embeds"], dim=-1)
        print(f"[clip {which}] text_embeds cosine min {cos.min().item():.6f}")
        assert cos.min().item() >= 0.999
    again = m(ids, output_hidden_states=True)
    assert all(torch.equal(a, b) for a, b in zip(out.to_tuple()[:2], again.to_tuple()[:2]))


def test_full_width_encode_prompt_graph_equals_eager(full_towers):
    from instructany2pix_b200.text_encoder import encode_prompt
    tl, tg = full_towers["l"][0], full_towers["g"][0]
    pos = [i.to(DEV) for i in full_towers["ids"]]
    neg = [O.make_ids("full/nl", 2, 77, O.PAD_CLIP_L).to(DEV), O.make_ids("full/ng", 2, 77, O.PAD_BIGG).to(DEV)]
    eager = encode_prompt([tl, tg], pos, neg, use_cuda_graph=False)
    g1 = encode_prompt([tl, tg], pos, neg)
    g2 = encode_prompt([tl, tg], pos, neg)
    for a, b, c in zip(eager, g1, g2):
        assert torch.equal(a, b) and torch.equal(b, c)
    assert g1[0].shape == (2, 77, 768 + 1280) and g1[2].shape == (2, 1280)
    towers = [full_towers["l"][1:4], full_towers["g"][1:4]]
    ref = O.encode_prompt(towers, pos, neg)
    assert rel(g1[0], ref[0]) <= 1e-2 and rel(g1[1], ref[1]) <= 1e-2
    assert F.cosine_similarity(g1[2], ref[2], dim=-1).min() >= 0.999


# ------------------------------------------------------------------------------------------------ end to end
def test_encode_prompt_into_sampler_vs_oracle_chain():
    """encode_prompt -> B200Sampler.generate on the tiny SDXL-topology UNet (cross_attention_dim 256 = 128 + 128, pooled width 128)
    against O.encode_prompt -> the oracle sampler, per-step eps with teacher forcing."""
    from instructany2pix_b200.sampler import B200Sampler
    from instructany2pix_b200.text_encoder import encode_prompt
    from oracle import sampler as osampler
    from oracle.synth import synth_input
    from tests.test_host_unet_emu import build_pair
    cl = O.CLIPTextCfg(hidden_size=128, intermediate_size=512, num_hidden_layers=2, num_attention_heads=2, hidden_act="quick_gelu")
    cg = O.CLIPTextCfg(hidden_size=128, intermediate_size=512, num_hidden_layers=3, num_attention_heads=2, hidden_act="gelu",
                       projection_dim=128)
    tl, sl = _tower(cl, False, seed=31)
    tg, sg = _tower(cg, True, seed=32)
    o, b = build_pair(False, device=DEV)
    pos = [O.make_ids("e2e/pl", 1, 77, O.PAD_CLIP_L), O.make_ids("e2e/pg", 1, 77, O.PAD_BIGG)]
    neg = [O.make_ids("e2e/nl", 1, 77, O.PAD_CLIP_L), O.make_ids("e2e/ng", 1, 77, O.PAD_BIGG)]
    tid = torch.tensor([[128.0, 128.0, 0.0, 0.0, 128.0, 128.0]]).repeat(2, 1)
    lat = synth_input("e2e/lat", (1, 4, 16, 16))

    pe, ne, pp, npool = O.encode_prompt([(sl, cl, False), (sg, cg, True)], pos, neg)
    ctx_o, added_o = torch.cat([ne, pe]).cpu(), dict(text_embeds=torch.cat([npool, pp]).cpu(), time_ids=tid)
    tr_o = []
    osampler.generate(o, lat, ctx_o, added_o, num_inference_steps=3, guidance_scale=7.5, trace=tr_o)

    pe, ne, pp, npool = encode_prompt([tl, tg], pos, neg)
    ctx_b, added_b = torch.cat([ne, pe]), dict(text_embeds=torch.cat([npool, pp]), time_ids=tid.to(DEV))
    assert rel(ctx_b.cpu(), ctx_o) < 1e-2
    tr_b = []
    B200Sampler(b).generate(lat.to(DEV), ctx_b, added_b, num_inference_steps=3, guidance_scale=7.5, trace=tr_b,
                            teacher=[t["x"].to(DEV) for t in tr_o])
    worst = max(rel(x["eps2"].cpu(), r["eps2"]) for x, r in zip(tr_b, tr_o))
    print(f"[clip e2e] per-step eps rel-L2 vs oracle chain: {worst:.3e}")
    assert worst <= 1e-2
