"""SDXL prompt encoders on the sm_100a kernels: ``B200CLIPTextModel`` (CLIP-L, the pipelines' ``text_encoder``) and
``B200CLIPTextModelWithProjection`` (OpenCLIP-bigG, ``text_encoder_2``; the refiner holds only this one), drop-ins for the
transformers classes, plus ``encode_prompt``: diffusers 0.26.3's SDXL combination rule on token ids.

Reference call sites: ``IPAdapterXL.generate`` -> ``pipe.encode_prompt(prompt, ..., negative_prompt)`` (ip_adapter.py:320-342,
both towers, positive and negative prompt) and the refinement pass (pipeline.py:358-361, the refiner's bigG tower).

Per layer the device runs four GEMMs and one attention kernel: LayerNorm 1 folded into the fused QKV GEMM, causal attention
(``ia2p_causal_self_attn_bf16``), the out-projection adding into the fp32 residual stream while emitting LayerNorm 2's row
statistics, fc1 with LayerNorm 2 folded in and the activation in its epilogue, fc2 adding into the stream.  The embedding kernel
emits layer 0's LayerNorm statistics the same way.  Tokenizers stay on the host: ids come in.
"""
from __future__ import annotations

from collections import OrderedDict
from types import SimpleNamespace

import torch
import torch.nn as nn

from . import ops
from .unet import _fold_ln

_CONFIG_FIELDS = ("vocab_size", "hidden_size", "intermediate_size", "num_hidden_layers", "num_attention_heads",
                  "max_position_embeddings", "hidden_act", "layer_norm_eps", "projection_dim", "eos_token_id")
_DEFAULTS = dict(vocab_size=49408, hidden_size=768, intermediate_size=3072, num_hidden_layers=12, num_attention_heads=12,
                 max_position_embeddings=77, hidden_act="quick_gelu", layer_norm_eps=1e-5, projection_dim=768, eos_token_id=2)


class CLIPTextOutput(OrderedDict):
    """What transformers' BaseModelOutputWithPooling / CLIPTextModelOutput offer diffusers: attribute access, and integer indexing
    over the fields that are set (``out[0]`` = last_hidden_state, or text_embeds for the projection model)."""

    def __getattr__(self, name):
        try:
            return self[name]
        except KeyError:
            raise AttributeError(name) from None

    def __getitem__(self, k):
        if isinstance(k, int):
            return self.to_tuple()[k]
        return super().__getitem__(k)

    def to_tuple(self):
        return tuple(v for v in self.values() if v is not None)


class _Attn(nn.Module):
    def __init__(self, C):
        super().__init__()
        self.q_proj, self.k_proj, self.v_proj, self.out_proj = (nn.Linear(C, C) for _ in range(4))


class _MLP(nn.Module):
    def __init__(self, C, F):
        super().__init__()
        self.fc1, self.fc2 = nn.Linear(C, F), nn.Linear(F, C)


class _Layer(nn.Module):
    def __init__(self, C, F, eps):
        super().__init__()
        self.self_attn = _Attn(C)
        self.layer_norm1 = nn.LayerNorm(C, eps=eps)
        self.mlp = _MLP(C, F)
        self.layer_norm2 = nn.LayerNorm(C, eps=eps)


class B200CLIPTextModel(nn.Module):
    """Drop-in for transformers' ``CLIPTextModel`` (same state-dict keys, ``.config``, ``.dtype``, ``.device``).  Weights are
    uninitialised until ``load_state_dict`` / ``from_module``.  Matrices are stored bf16 (tensor-core operands), norm scales,
    biases and the position table fp32; outputs are fp32."""

    with_projection = False

    def __init__(self, config=None, device="cuda"):
        super().__init__()
        src = config if isinstance(config, dict) else ({} if config is None else
                                                        {k: getattr(config, k) for k in _CONFIG_FIELDS if hasattr(config, k)})
        cfg = self.config = SimpleNamespace(**{k: src.get(k, v) for k, v in _DEFAULTS.items()})
        C, F, H = cfg.hidden_size, cfg.intermediate_size, cfg.num_attention_heads
        if C != 64 * H or C % 64 or F % 64:
            raise NotImplementedError(f"B200CLIPTextModel needs head_dim 64 and widths that are multiples of 64 (hidden {C}, "
                                      f"heads {H}, intermediate {F})")
        if cfg.hidden_act not in ("gelu", "quick_gelu"):
            raise NotImplementedError(f"hidden_act {cfg.hidden_act!r} (supported: gelu, quick_gelu)")
        with torch.device("meta"):
            tm = self.text_model = nn.Module()
            tm.embeddings = nn.Module()
            tm.embeddings.token_embedding = nn.Embedding(cfg.vocab_size, C)
            tm.embeddings.position_embedding = nn.Embedding(cfg.max_position_embeddings, C)
            tm.encoder = nn.Module()
            tm.encoder.layers = nn.ModuleList([_Layer(C, F, cfg.layer_norm_eps) for _ in range(cfg.num_hidden_layers)])
            tm.final_layer_norm = nn.LayerNorm(C, eps=cfg.layer_norm_eps)
            if self.with_projection:
                self.text_projection = nn.Linear(C, cfg.projection_dim, bias=False)
        for name, p in self.named_parameters():
            p.requires_grad_(False)
            if p.ndim >= 2 and "position_embedding" not in name:
                p.data = p.data.to(torch.bfloat16)
        self.to_empty(device=device)
        self._packed = None
        self._graphs = OrderedDict()
        self.max_graphs = 4

    @classmethod
    def from_module(cls, hf_module, device=None):
        """Adopt a transformers CLIPTextModel / CLIPTextModelWithProjection (config and weights)."""
        device = device or getattr(hf_module, "device", "cuda")
        new = cls(hf_module.config, device=device)
        new.load_state_dict(hf_module.state_dict())
        return new

    def load_state_dict(self, state_dict, strict=True, **kw):
        sd = {k: v for k, v in state_dict.items() if not k.endswith("embeddings.position_ids")}    # stale buffer of older versions
        r = super().load_state_dict(sd, strict=strict, **kw)
        self.invalidate()
        return r

    def invalidate(self):
        self._packed = None
        self._graphs.clear()

    @property
    def dtype(self):
        return torch.float32

    @property
    def device(self):
        return self.text_model.final_layer_norm.weight.device

    # ------------------------------------------------------------------ weight packing (once per load)
    def prepare(self):
        if self._packed is not None:
            return self._packed
        f32 = lambda t: t.detach().float().contiguous()
        bf = lambda t: t.detach().to(torch.bfloat16).contiguous()
        tm = self.text_model
        layers = []
        for L in tm.encoder.layers:
            a = L.self_attn
            wqkv = torch.cat([a.q_proj.weight, a.k_proj.weight, a.v_proj.weight], 0)
            bqkv = torch.cat([a.q_proj.bias, a.k_proj.bias, a.v_proj.bias], 0)
            layers.append(dict(qkv=_fold_ln(wqkv, bqkv, L.layer_norm1), wo=bf(a.out_proj.weight), bo=f32(a.out_proj.bias),
                               fc1=_fold_ln(L.mlp.fc1.weight, L.mlp.fc1.bias, L.layer_norm2), w2=bf(L.mlp.fc2.weight),
                               b2=f32(L.mlp.fc2.bias)))
        fl = tm.final_layer_norm
        self._packed = dict(tok=bf(tm.embeddings.token_embedding.weight), pos=f32(tm.embeddings.position_embedding.weight),
                            layers=layers, lnf=(f32(fl.weight), f32(fl.bias), float(fl.eps)),
                            proj=bf(self.text_projection.weight) if self.with_projection else None)
        return self._packed

    # ------------------------------------------------------------------ the tower
    def _ids(self, input_ids):
        """int64 ids on the device; host ids are range-checked first (a device id outside the vocabulary yields NaN rows)"""
        ids = input_ids.to(torch.int64)
        V = self.config.vocab_size
        if ids.device.type == "cpu" and ids.numel() and (int(ids.min()) < 0 or int(ids.max()) >= V):
            raise ValueError(f"token ids outside [0, {V})")
        if ids.device != self.device:
            if self.device.type == "cuda" and ids.device.type == "cpu":
                ids = ids.pin_memory()
            ids = ids.to(self.device, non_blocking=True)
        return ids.contiguous()

    def _eos_rows(self, ids):
        """flat row index of each sequence's pooled token: transformers' rule for config.eos_token_id (== 2: first arg-max id,
        the legacy rule SDXL's configs hit; else the first id equal to eos_token_id)"""
        n, T = ids.shape
        eos = self.config.eos_token_id
        pos = ids.argmax(-1) if eos == 2 else (ids == eos).int().argmax(-1)
        return torch.arange(n, device=ids.device) * T + pos

    def _run(self, ids, n_layers, pooled):
        """hidden states 0..n_layers (fp32 [n*T, C]) and, if ``pooled``, the final-LN rows at the EOS positions (and their
        projection for the projection model)"""
        P = self.prepare()
        cfg = self.config
        n, T = ids.shape
        heads = cfg.num_attention_heads
        x, xb, st = ops.clip_embed(ids, P["tok"], P["pos"], want_ln=True)
        hs = [x]
        for L in P["layers"][:n_layers]:
            w, c1, c2, eps = L["qkv"]
            qkv = ops.gemm(xb, w, bias=c2, ln=(st, c1, eps))
            a = ops.causal_self_attn(qkv, n, T, heads)
            x, xb, st = ops.gemm(a, L["wo"], bias=L["bo"], residual=x, out_dtype=torch.float32, want_ln=True)
            w, c1, c2, eps = L["fc1"]
            h = ops.gemm(xb, w, bias=c2, ln=(st, c1, eps), act=cfg.hidden_act)
            x, xb, st = ops.gemm(h, L["w2"], bias=L["b2"], residual=x, out_dtype=torch.float32, want_ln=True)
            hs.append(x)
        pool = emb = None
        if pooled:
            g, b, eps = P["lnf"]
            pool = ops.layernorm(x.index_select(0, self._eos_rows(ids)), g, b, eps, out_dtype=torch.float32)
            if self.with_projection:
                emb = ops.gemm_smallm(pool, P["proj"])
        return hs, pool, emb

    @torch.no_grad()
    def forward(self, input_ids, attention_mask=None, position_ids=None, output_hidden_states=None, return_dict=True):
        if attention_mask is not None:
            raise NotImplementedError("attention_mask: the SDXL pipelines never pass one; CLIP attends over pad tokens causally")
        if position_ids is not None:
            raise NotImplementedError("position_ids: only the default positions 0..T-1 are supported")
        ids = self._ids(input_ids)
        n, T = ids.shape
        cfg = self.config
        hs, pool, emb = self._run(ids, cfg.num_hidden_layers, pooled=True)
        g, b, eps = self.prepare()["lnf"]
        last = ops.layernorm(hs[-1], g, b, eps, out_dtype=torch.float32).reshape(n, T, -1)
        hidden = tuple(h.reshape(n, T, -1) for h in hs) if output_hidden_states else None
        if self.with_projection:
            out = CLIPTextOutput(text_embeds=emb, last_hidden_state=last, hidden_states=hidden)
        else:
            out = CLIPTextOutput(last_hidden_state=last, pooler_output=pool, hidden_states=hidden)
        return out if return_dict else out.to_tuple()

    # ------------------------------------------------------------------ encode_prompt's per-tower pass (CUDA graph)
    def _embeds(self, ids, hs_index, pooled, use_cuda_graph=True):
        """(hidden_states[hs_index] [n, T, C], text_embeds [n, P] | None) for ids on the device.  Layers past the selected hidden
        state run only when the pooled output is wanted.  One CUDA graph per (n, T, hs_index, pooled), small LRU."""
        n, T = ids.shape
        L = self.config.num_hidden_layers
        k = hs_index % (L + 1)
        n_layers = L if pooled else k

        def body(i):
            hs, _, emb = self._run(i, n_layers, pooled)
            return hs[k].reshape(n, T, -1), emb

        if not (use_cuda_graph and ids.is_cuda):
            return body(ids)
        key = (n, T, k, pooled)
        ent = self._graphs.get(key)
        if ent is None:
            while len(self._graphs) >= self.max_graphs:
                self._graphs.pop(next(iter(self._graphs)))
            ent = dict(ids=torch.empty_like(ids))
            ent["ids"].copy_(ids)
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):          # warm-up outside capture: first-use function attributes, packing
                body(ent["ids"])
            torch.cuda.current_stream().wait_stream(s)
            ent["graph"] = torch.cuda.CUDAGraph()
            with torch.cuda.graph(ent["graph"]):
                ent["out"] = body(ent["ids"])
            self._graphs[key] = ent
        else:
            self._graphs.move_to_end(key)
        ent["ids"].copy_(ids)
        ent["graph"].replay()
        return ent["out"]


class B200CLIPTextModelWithProjection(B200CLIPTextModel):
    """Drop-in for transformers' ``CLIPTextModelWithProjection`` (SDXL ``text_encoder_2``: ``out[0]`` = text_embeds)."""

    with_projection = True


@torch.no_grad()
def encode_prompt(text_encoders, prompt_ids, negative_ids=None, force_zeros_for_empty_prompt=True, clip_skip=None,
                  use_cuda_graph=True):
    """diffusers 0.26.3 ``StableDiffusionXLPipeline.encode_prompt`` on token ids (ip_adapter.py:320-342; refiner
    pipeline.py:358-361).  ``text_encoders``: the towers in pipeline order (base: [CLIP-L, bigG], refiner: [bigG]);
    ``prompt_ids`` / ``negative_ids``: one int64 [B, T] tensor per tower, from that tower's tokenizer.

    Per tower ``hidden_states[-(clip_skip or 0) - 2]``, concatenated over the towers on the last dim; the pooled output is the last
    tower's ``text_embeds``.  No negative ids with ``force_zeros_for_empty_prompt``: the negatives are zeros.  Negative and positive
    prompts go through each tower in ONE pass of 2B sequences.  Returns (prompt_embeds, negative_prompt_embeds,
    pooled_prompt_embeds, negative_pooled_prompt_embeds), fp32 on the device -- ``cat([negative, positive])`` is the ``ctx`` /
    ``text_embeds`` order of ``B200Sampler.generate``."""
    if len(prompt_ids) != len(text_encoders) or (negative_ids is not None and len(negative_ids) != len(text_encoders)):
        raise ValueError("one ids tensor per text encoder is needed")
    if not text_encoders[-1].with_projection:
        raise ValueError("the last text encoder must be a B200CLIPTextModelWithProjection (it supplies the pooled embedding)")
    if negative_ids is None and not force_zeros_for_empty_prompt:
        raise ValueError("negative_ids are required unless force_zeros_for_empty_prompt (tokenizers are not part of this library)")
    hs_index = -(clip_skip or 0) - 2
    B = prompt_ids[0].shape[0]
    embeds, pooled = [], None
    for i, enc in enumerate(text_encoders):
        ids = enc._ids(prompt_ids[i] if negative_ids is None else torch.cat([enc._ids(negative_ids[i]), enc._ids(prompt_ids[i])]))
        h, emb = enc._embeds(ids, hs_index, pooled=i == len(text_encoders) - 1, use_cuda_graph=use_cuda_graph)
        embeds.append(h)
        pooled = emb
    pe = torch.cat(embeds, dim=-1)
    if negative_ids is None:
        return pe, torch.zeros_like(pe), pooled.clone(), torch.zeros_like(pooled)
    return pe[B:], pe[:B], pooled[B:].clone(), pooled[:B].clone()
