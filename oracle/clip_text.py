"""Oracle (test infrastructure): plain fp32 restatement of transformers' ``CLIPTextModel`` / ``CLIPTextModelWithProjection``
forward -- the SDXL prompt encoders (``text_encoder`` = CLIP-L, ``text_encoder_2`` = OpenCLIP-bigG with projection).

Call sites in the reference: ``IPAdapterXL.generate`` -> ``pipe.encode_prompt(prompt, ..., negative_prompt)`` (ip_adapter.py:320-342)
runs both towers for the positive and the negative prompt; the refinement pass (pipeline.py:358-361) runs the refiner's bigG
tower.  diffusers 0.26.3's ``encode_prompt`` reads ``out[0]`` (the projected pooled row of the last tower) and
``out.hidden_states[-(clip_skip or 0) - 2]``.

Works on a transformers-keyed state dict (``text_model.embeddings.token_embedding.weight``, ...), so the same name-seeded weights
(oracle/synth.py) drive transformers itself (tests/golden/clip_text.npz), this restatement and the B200 modules.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch
import torch.nn.functional as F

PAD_CLIP_L = 49407     # CLIP-L tokenizer: pads with its end-of-text id
PAD_BIGG = 0           # OpenCLIP-bigG tokenizer (SDXL tokenizer_2): pads with "!" = 0


@dataclass
class CLIPTextCfg:
    vocab_size: int = 49408
    hidden_size: int = 768
    intermediate_size: int = 3072
    num_hidden_layers: int = 12
    num_attention_heads: int = 12
    max_position_embeddings: int = 77
    hidden_act: str = "quick_gelu"
    layer_norm_eps: float = 1e-5
    projection_dim: int = 768
    eos_token_id: int = 2

    def hf_kwargs(self):
        return dict(self.__dict__)


CLIP_L = CLIPTextCfg()
BIGG = CLIPTextCfg(hidden_size=1280, intermediate_size=5120, num_hidden_layers=32, num_attention_heads=20, hidden_act="gelu",
                   projection_dim=1280)


def state_dict_shapes(cfg: CLIPTextCfg, with_projection: bool):
    C, F_ = cfg.hidden_size, cfg.intermediate_size
    s = {"text_model.embeddings.token_embedding.weight": (cfg.vocab_size, C),
         "text_model.embeddings.position_embedding.weight": (cfg.max_position_embeddings, C)}
    for i in range(cfg.num_hidden_layers):
        p = f"text_model.encoder.layers.{i}."
        for n in ("q_proj", "k_proj", "v_proj", "out_proj"):
            s[p + f"self_attn.{n}.weight"] = (C, C)
            s[p + f"self_attn.{n}.bias"] = (C,)
        for n in ("layer_norm1", "layer_norm2"):
            s[p + n + ".weight"] = (C,)
            s[p + n + ".bias"] = (C,)
        s[p + "mlp.fc1.weight"], s[p + "mlp.fc1.bias"] = (F_, C), (F_,)
        s[p + "mlp.fc2.weight"], s[p + "mlp.fc2.bias"] = (C, F_), (C,)
    s["text_model.final_layer_norm.weight"] = (C,)
    s["text_model.final_layer_norm.bias"] = (C,)
    if with_projection:
        s["text_projection.weight"] = (cfg.projection_dim, C)
    return s


def _act(x, name):
    if name == "quick_gelu":
        return x * torch.sigmoid(1.702 * x)
    if name == "gelu":
        return F.gelu(x)
    raise NotImplementedError(name)


def eos_positions(input_ids, eos_token_id):
    """transformers' pooling rule: eos_token_id == 2 (the legacy configs SDXL ships) -> first arg-max id, else the first id equal
    to eos_token_id."""
    if eos_token_id == 2:
        return input_ids.to(torch.int64).argmax(dim=-1)
    return (input_ids.to(torch.int64) == eos_token_id).int().argmax(dim=-1)


@torch.no_grad()
def forward(sd, cfg: CLIPTextCfg, input_ids, with_projection=False, dtype=torch.float32):
    """-> dict(last_hidden_state [n,T,C], pooler_output [n,C], hidden_states (num_hidden_layers + 1) x [n,T,C],
    text_embeds [n,P] when ``with_projection``), computed in ``dtype`` (fp32: the reference for the tests; bf16 on a GPU: the
    eager comparator of tools/bench_text_encoders.py)."""
    w = lambda k: sd[k].to(dtype)
    n, T = input_ids.shape
    C, H = cfg.hidden_size, cfg.num_attention_heads
    d = C // H
    dev = sd["text_model.embeddings.token_embedding.weight"].device
    ids = input_ids.to(dev, torch.int64)
    x = w("text_model.embeddings.token_embedding.weight")[ids] + w("text_model.embeddings.position_embedding.weight")[:T][None]
    hs = [x]
    causal = torch.full((T, T), float("-inf"), device=dev, dtype=dtype).triu(1)
    for i in range(cfg.num_hidden_layers):
        p = f"text_model.encoder.layers.{i}."
        lin = lambda t, name: t @ w(p + name + ".weight").t() + w(p + name + ".bias")
        h = F.layer_norm(x, (C,), w(p + "layer_norm1.weight"), w(p + "layer_norm1.bias"), cfg.layer_norm_eps)
        q, k, v = [lin(h, f"self_attn.{m}").reshape(n, T, H, d).transpose(1, 2) for m in ("q_proj", "k_proj", "v_proj")]
        a = torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(d) + causal, dim=-1) @ v
        x = x + lin(a.transpose(1, 2).reshape(n, T, C), "self_attn.out_proj")
        h = F.layer_norm(x, (C,), w(p + "layer_norm2.weight"), w(p + "layer_norm2.bias"), cfg.layer_norm_eps)
        x = x + lin(_act(lin(h, "mlp.fc1"), cfg.hidden_act), "mlp.fc2")
        hs.append(x)
    last = F.layer_norm(x, (C,), w("text_model.final_layer_norm.weight"), w("text_model.final_layer_norm.bias"), cfg.layer_norm_eps)
    pooled = last[torch.arange(n, device=dev), eos_positions(ids, cfg.eos_token_id)]
    out = dict(last_hidden_state=last, pooler_output=pooled, hidden_states=tuple(hs))
    if with_projection:
        out["text_embeds"] = pooled @ w("text_projection.weight").t()
    return out


def encode_prompt(towers, prompt_ids, negative_ids=None, force_zeros_for_empty_prompt=True, clip_skip=None, dtype=torch.float32):
    """diffusers 0.26.3 ``StableDiffusionXLPipeline.encode_prompt`` on token ids: ``towers`` = [(sd, cfg, with_projection), ...]
    (base: CLIP-L then bigG; refiner: bigG only).  -> (prompt_embeds, negative_prompt_embeds, pooled, negative_pooled)."""
    def run(ids_list):
        embeds, pooled = [], None
        for (sd, cfg, proj), ids in zip(towers, ids_list):
            o = forward(sd, cfg, ids, with_projection=proj, dtype=dtype)
            pooled = o["text_embeds"] if proj else o["last_hidden_state"]
            embeds.append(o["hidden_states"][-(clip_skip or 0) - 2])
        return torch.cat(embeds, dim=-1), pooled

    pe, pp = run(prompt_ids)
    if negative_ids is None and force_zeros_for_empty_prompt:
        return pe, torch.zeros_like(pe), pp, torch.zeros_like(pp)
    ne, npool = run(negative_ids)
    return pe, ne, pp, npool


def make_ids(tag, n, T, pad, eos_id=PAD_CLIP_L, seed=0):
    """token ids as a CLIP tokenizer emits them: BOS 49406, words, end-of-text ``eos_id``, then ``pad`` up to T."""
    from .synth import _gen
    g = _gen("clip_ids/" + tag, seed)
    ids = torch.full((n, T), pad, dtype=torch.int64)
    for i in range(n):
        L = int(torch.randint(1, T - 1, (1,), generator=g))
        ids[i, 0] = 49406
        ids[i, 1:L + 1] = torch.randint(300, 49000, (L,), generator=g)
        ids[i, L + 1] = eos_id
    return ids
