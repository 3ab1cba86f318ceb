"""Oracle (test infrastructure): generate tests/golden/clip_text.npz by running transformers' OWN ``CLIPTextModel`` /
``CLIPTextModelWithProjection`` -- the SDXL prompt encoders -- at small widths: both activations (``quick_gelu`` CLIP-L, ``gelu``
bigG), both pooling (EOS) rules, ids padded like the CLIP-L tokenizer (49407) and like the bigG tokenizer (0).

Needs only transformers (no reference checkout):  ``python -m oracle.gen_golden_clip_text``.  Weights are name-seeded
(oracle/synth.py), so the fixture stores ids and outputs only; the GPU tests compare against the restatement
(oracle/clip_text.py), which tests/test_clip_text_cpu.py pins to this fixture.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from .clip_text import CLIPTextCfg, make_ids, state_dict_shapes
from .synth import synth_state_dict

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

CLIP_TEXT_CASES = [  # name, config overrides, with_projection, T, pad id, end-of-text id written into the ids
    ("l_quick", dict(hidden_size=64, intermediate_size=128, num_hidden_layers=2, num_attention_heads=1, hidden_act="quick_gelu"),
     False, 77, 49407, 49407),
    ("g_gelu", dict(hidden_size=128, intermediate_size=256, num_hidden_layers=3, num_attention_heads=2, hidden_act="gelu",
                    projection_dim=64), True, 77, 0, 49407),
    ("g_eosid", dict(hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=2, hidden_act="gelu",
                     projection_dim=64, eos_token_id=49405), True, 20, 0, 49405),
]


def clip_text_case(name):
    """(state dict, oracle config, with_projection, ids) of a CLIP_TEXT_CASES entry (name-seeded weights, seed 7)"""
    _, kw, proj, T, pad, eos_id = next(c for c in CLIP_TEXT_CASES if c[0] == name)
    cfg = CLIPTextCfg(**kw)
    sd = synth_state_dict(state_dict_shapes(cfg, proj), seed=7)
    return sd, cfg, proj, make_ids(name, 2, T, pad, eos_id)


def gen_clip_text():
    from transformers import CLIPTextConfig, CLIPTextModel, CLIPTextModelWithProjection
    out = {}
    for name, *_ in CLIP_TEXT_CASES:
        sd, cfg, proj, ids = clip_text_case(name)
        m = (CLIPTextModelWithProjection if proj else CLIPTextModel)(CLIPTextConfig(**cfg.hf_kwargs())).eval()
        missing, unexpected = m.load_state_dict(sd, strict=False)
        assert not unexpected and all(k.endswith("position_ids") for k in missing), (missing, unexpected)
        o = m(ids, output_hidden_states=True)
        out[name + "/ids"] = ids.numpy()
        out[name + "/hs_m2"] = o.hidden_states[-2].numpy()
        out[name + "/n_hidden"] = np.array(len(o.hidden_states))
        out[name + "/last"] = o.last_hidden_state.numpy()
        out[name + "/pooled"] = o[0 if proj else 1].numpy()                # text_embeds | pooler_output
    os.makedirs(OUT, exist_ok=True)
    np.savez_compressed(os.path.join(OUT, "clip_text.npz"), **out)
    print("clip_text:", {k: tuple(v.shape) for k, v in out.items()})


if __name__ == "__main__":
    torch.set_grad_enabled(False)
    gen_clip_text()
