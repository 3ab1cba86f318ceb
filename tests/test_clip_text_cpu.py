"""SDXL prompt encoders without a GPU: the fp32 restatement (oracle/clip_text.py) against transformers' own outputs
(tests/golden/clip_text.npz, and live when transformers is importable), the host logic of B200CLIPTextModel(WithProjection) /
encode_prompt under CPU doubles of the ops, and the argument checks of the new C entry points."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import clip_text as O
from oracle import gen_golden_clip_text as G
from oracle.synth import synth_state_dict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "clip_text.npz")
BF = torch.bfloat16


def rel(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm()).item()


# ------------------------------------------------------------------------------------------------ restatement vs transformers
@pytest.mark.parametrize("name", [c[0] for c in G.CLIP_TEXT_CASES])
def test_restatement_matches_golden(name):
    z = np.load(GOLDEN)
    sd, cfg, proj, ids = G.clip_text_case(name)
    assert (z[name + "/ids"] == ids.numpy()).all()
    o = O.forward(sd, cfg, ids, with_projection=proj)
    assert len(o["hidden_states"]) == int(z[name + "/n_hidden"]) == cfg.num_hidden_layers + 1
    for key, got in (("hs_m2", o["hidden_states"][-2]), ("last", o["last_hidden_state"]),
                     ("pooled", o["text_embeds"] if proj else o["pooler_output"])):
        assert (got - torch.from_numpy(z[name + "/" + key])).abs().max().item() <= 1e-5, key


def _hf(cfg, proj, seed=7):
    transformers = pytest.importorskip("transformers")
    cls = transformers.CLIPTextModelWithProjection if proj else transformers.CLIPTextModel
    m = cls(transformers.CLIPTextConfig(**cfg.hf_kwargs())).eval()
    sd = synth_state_dict(O.state_dict_shapes(cfg, proj), seed=seed)
    m.load_state_dict(sd, strict=False)
    return m, sd


@pytest.mark.parametrize("act,eos,pad", [("quick_gelu", 2, O.PAD_CLIP_L), ("gelu", 2, O.PAD_BIGG), ("gelu", 49407, O.PAD_BIGG)])
def test_restatement_matches_transformers_live(act, eos, pad):
    cfg = O.CLIPTextCfg(hidden_size=128, intermediate_size=192, num_hidden_layers=2, num_attention_heads=4, hidden_act=act,
                        projection_dim=32, eos_token_id=eos, max_position_embeddings=40)
    m, sd = _hf(cfg, True, seed=11)
    ids = O.make_ids(f"live/{act}/{eos}", 3, 33, pad)
    with torch.no_grad():
        ref = m(ids, output_hidden_states=True)
    o = O.forward(sd, cfg, ids, with_projection=True)
    for a, b in zip(o["hidden_states"], ref.hidden_states):
        assert (a - b).abs().max() < 1e-5
    assert (o["text_embeds"] - ref.text_embeds).abs().max() < 1e-5
    assert (o["last_hidden_state"] - ref.last_hidden_state).abs().max() < 1e-5


# ------------------------------------------------------------------------------------------------ host logic under CPU doubles
def _clip_embed(ids, tok, pos, want_ln=False):
    n, T = ids.shape
    V = tok.shape[0]
    bad = (ids < 0) | (ids >= V)
    x = tok[ids.clamp(0, V - 1)].float() + pos[:T][None].float()
    x[bad] = float("nan")
    x = x.reshape(n * T, -1)
    if want_ln:
        return x, x.to(BF), torch.stack([x.sum(1), (x * x).sum(1)], -1)[:, None]
    return x


def _causal(qkv, n, T, heads, out=None):
    Cw = heads * 64
    q, k, v = [t.float().reshape(n, T, heads, 64).transpose(1, 2) for t in qkv.split(Cw, dim=1)]
    return F.scaled_dot_product_attention(q, k, v, is_causal=True).transpose(1, 2).reshape(n * T, Cw).to(BF)


@pytest.fixture
def clip_emu(emu, monkeypatch):
    """the ``emu`` doubles plus the prompt-encoder ops: embedding, causal attention, GEMM activation epilogues"""
    import instructany2pix_b200.ops as real

    calls = {"clip_embed": 0}

    def embed(*a, **k):
        calls["clip_embed"] += 1
        return _clip_embed(*a, **k)

    def gemm(*a, act=None, **k):
        if act is None:
            return emu.gemm(*a, **k)
        h = emu.gemm(*a, **dict(k, out_dtype=torch.float32))
        return (h * torch.sigmoid(1.702 * h) if act == "quick_gelu" else F.gelu(h)).to(BF)

    monkeypatch.setattr(real, "clip_embed", embed)
    monkeypatch.setattr(real, "causal_self_attn", _causal)
    monkeypatch.setattr(real, "gemm", gemm)
    return calls


def _tower(cfg, proj, seed):
    from instructany2pix_b200.text_encoder import B200CLIPTextModel, B200CLIPTextModelWithProjection
    sd = synth_state_dict(O.state_dict_shapes(cfg, proj), seed=seed)
    m = (B200CLIPTextModelWithProjection if proj else B200CLIPTextModel)(cfg.hf_kwargs(), device="cpu")
    m.load_state_dict(dict(sd, **{"text_model.embeddings.position_ids": torch.arange(cfg.max_position_embeddings)[None]}))
    return m, sd


L_CFG = O.CLIPTextCfg(hidden_size=128, intermediate_size=256, num_hidden_layers=3, num_attention_heads=2, hidden_act="quick_gelu")
G_CFG = O.CLIPTextCfg(hidden_size=192, intermediate_size=384, num_hidden_layers=3, num_attention_heads=3, hidden_act="gelu",
                      projection_dim=64)


@pytest.mark.parametrize("proj,eos", [(False, 2), (True, 2), (True, 49405)])
def test_forward_host_logic(clip_emu, proj, eos):
    cfg = O.CLIPTextCfg(**dict(G_CFG.hf_kwargs(), eos_token_id=eos))
    m, sd = _tower(cfg, proj, seed=3)
    ids = O.make_ids("host", 2, 77, O.PAD_BIGG, eos_id=49405 if eos != 2 else 49407)
    ref = O.forward(sd, cfg, ids, with_projection=proj)
    out = m(ids, output_hidden_states=True)
    assert len(out.hidden_states) == cfg.num_hidden_layers + 1
    assert rel(out.hidden_states[-1], ref["hidden_states"][-1]) < 2e-2             # before final_layer_norm, as transformers
    assert rel(out.hidden_states[-2], ref["hidden_states"][-2]) < 2e-2
    assert rel(out.last_hidden_state, ref["last_hidden_state"]) < 2e-2
    if proj:
        assert out[0] is out.text_embeds and rel(out.text_embeds, ref["text_embeds"]) < 2e-2
        assert "pooler_output" not in out
    else:
        assert out[0] is out.last_hidden_state and rel(out.pooler_output, ref["pooler_output"]) < 2e-2
    assert m(ids).get("hidden_states") is None and isinstance(m(ids, return_dict=False), tuple)
    with pytest.raises(NotImplementedError):
        m(ids, attention_mask=torch.ones_like(ids))


def test_eos_selection_rules(clip_emu):
    from instructany2pix_b200.text_encoder import B200CLIPTextModelWithProjection
    ids = torch.tensor([[49406, 5, 7, 49407, 0, 0], [49406, 320, 49405, 9, 49407, 49407]])
    m = B200CLIPTextModelWithProjection(dict(G_CFG.hf_kwargs(), eos_token_id=2), device="cpu")
    assert m._eos_rows(ids).tolist() == [3, 6 + 4]                      # legacy rule: first arg-max id
    m.config.eos_token_id = 49405
    assert m._eos_rows(ids).tolist() == [0, 6 + 2]                      # first id equal to eos_token_id (row 0 has none: 0)


def test_encode_prompt_combination(clip_emu):
    from instructany2pix_b200.text_encoder import encode_prompt
    tl, sl = _tower(L_CFG, False, seed=5)
    tg, sg = _tower(G_CFG, True, seed=6)
    B, T = 2, 77
    pos = [O.make_ids("p/l", B, T, O.PAD_CLIP_L), O.make_ids("p/g", B, T, O.PAD_BIGG)]
    neg = [O.make_ids("n/l", B, T, O.PAD_CLIP_L), O.make_ids("n/g", B, T, O.PAD_BIGG)]
    towers = [(sl, L_CFG, False), (sg, G_CFG, True)]
    for clip_skip in (None, 1):
        got = encode_prompt([tl, tg], pos, neg, clip_skip=clip_skip)
        ref = O.encode_prompt(towers, pos, neg, clip_skip=clip_skip)
        assert got[0].shape == (B, T, 128 + 192) and got[2].shape == (B, 64)
        for a, b in zip(got, ref):
            assert a.shape == b.shape and rel(a, b) < 2e-2
    clip_emu["clip_embed"] = 0
    pe, ne, pp, npool = encode_prompt([tl, tg], pos)                    # no negative prompt: zeros
    assert clip_emu["clip_embed"] == 2                                  # one pass per tower
    assert not ne.any() and not npool.any() and rel(pe, O.encode_prompt(towers, pos)[0]) < 2e-2
    clip_emu["clip_embed"] = 0
    both = encode_prompt([tl, tg], pos, neg)
    assert clip_emu["clip_embed"] == 2                                  # negatives and positives in ONE pass of 2B sequences
    sep_n = encode_prompt([tl, tg], neg)
    assert torch.equal(both[1], sep_n[0]) and torch.equal(both[3], sep_n[2])      # [negative; positive] split back correctly
    # refiner: the bigG tower alone
    r = encode_prompt([tg], pos[1:], neg[1:])
    rr = O.encode_prompt(towers[1:], pos[1:], neg[1:])
    assert r[0].shape == (B, T, 192) and all(rel(a, b) < 2e-2 for a, b in zip(r, rr))
    with pytest.raises(ValueError):
        encode_prompt([tl, tg], pos, force_zeros_for_empty_prompt=False)
    with pytest.raises(ValueError):
        encode_prompt([tg, tl], pos[::-1])                              # pooled output must come from a projection tower


def test_host_ids_are_range_checked(clip_emu):
    m, _ = _tower(G_CFG, True, seed=6)
    ids = O.make_ids("bad", 1, 10, 0)
    ids[0, 3] = 49408
    with pytest.raises(ValueError):
        m(ids)


def test_from_transformers_module_keys():
    cfg = O.CLIPTextCfg(hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=2, hidden_act="gelu",
                        projection_dim=64, max_position_embeddings=77)
    hf, sd = _hf(cfg, True)
    from instructany2pix_b200.text_encoder import B200CLIPTextModelWithProjection
    m = B200CLIPTextModelWithProjection.from_module(hf, device="cpu")
    assert m.config.hidden_act == "gelu" and m.config.projection_dim == 64 and m.config.num_hidden_layers == 2
    assert m.dtype == torch.float32 and m.device.type == "cpu"
    mine = m.state_dict()
    assert set(mine) == {k for k in hf.state_dict() if not k.endswith("position_ids")}
    for k, v in sd.items():
        assert torch.equal(mine[k].float(), v), k                       # bf16-representable weights: exact


# ------------------------------------------------------------------------------------------------ C entry points
def test_new_entry_points_exported_and_reject_bad_args():
    from instructany2pix_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        subprocess.run(["make", "-C", os.path.join(ROOT, "instructany2pix_b200", "csrc"), "-j8"], check=True)
    lib = _lib.load()
    for name in ("ia2p_causal_self_attn_bf16", "ia2p_clip_embed"):
        assert hasattr(lib, name)
    assert (_lib.EPI_GELU, _lib.EPI_QUICK_GELU) == (2, 3)
    buf = C.create_string_buffer(4096 + 256)
    p = (C.addressof(buf) + 255) // 256 * 256
    attn = lambda q, n, T, heads, ld=192: lib.ia2p_causal_self_attn_bf16(q, q, q, ld, q, 64, n, T, heads, 0.125, None)
    assert attn(p, 1, 0, 1) == -3 and attn(p, 1, 129, 1) == -3           # IA2P_E_SHAPE: T outside [1, 128]
    assert attn(None, 1, 8, 1) == -1 and attn(p, 0, 8, 1) == -1         # IA2P_E_ARG
    assert attn(p, 1, 8, 1, ld=100) == -4                               # IA2P_E_ALIGN
    emb = lambda T, P, Cw, o2=None, st=None: lib.ia2p_clip_embed(p, 1, T, p, 10, p, P, Cw, p, o2, st, None)
    assert emb(78, 77, 64) == -3 and emb(4, 77, 60) == -3               # more positions than the table, C % 8
    assert emb(4, 77, 64, o2=p) == -1                                   # out_bf16 without stats
    assert lib.ia2p_clip_embed(None, 1, 4, p, 10, p, 77, 64, p, None, None, None) == -1
    gemm = lambda epi, res: lib.ia2p_gemm_bf16(p, 64, 64, None, 0, 0, p, p, 64, 128, 64, None, None, 0, res, 64, _lib.BF16,
                                               _lib.BF16, epi, None)
    assert gemm(_lib.EPI_GELU, p) < 0 and gemm(_lib.EPI_QUICK_GELU, p) < 0   # activation with a residual
