#!/usr/bin/env python
"""SDXL prompt encoding on one GPU: ms per ``encode_prompt`` (CLIP-L + OpenCLIP-bigG, negative and positive prompts in one pass,
CUDA graph) at n = 2 sequences per tower (one CFG pair) and n = 16 (eight requests), against the fp32-restatement oracle run in
eager bf16 on the same GPU.  Prints one JSON line.

Timing: CUDA events around each call, warmed, median over --calls calls.  Weights: random at the real widths (timing does not
depend on their values).  Streamed weight bytes are analytic: the bf16 GEMM weights of every layer run (CLIP-L stops after
layer 11 of 12: its last layer only feeds the pooled output SDXL discards) plus bigG's projection; token tables are gathered, not
streamed, and not counted.  Usage: python tools/bench_text_encoders.py [--calls 50]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

from instructany2pix_b200 import ops
from instructany2pix_b200.text_encoder import B200CLIPTextModel, B200CLIPTextModelWithProjection, encode_prompt
from oracle import clip_text as O

HBM_TBPS = 7.7


def random_sd(cfg, proj, dev):
    sd = {}
    for k, shp in O.state_dict_shapes(cfg, proj).items():
        if len(shp) == 1:
            sd[k] = (1.0 if k.endswith("norm1.weight") or k.endswith("norm2.weight") or k.endswith("final_layer_norm.weight") else 0.0) \
                + 0.05 * torch.randn(shp, device=dev)
        else:
            sd[k] = (torch.rand(shp, device=dev) * 2 - 1) * (0.02 if "embedding" in k else shp[1] ** -0.5)
    return sd


def weight_bytes(cfg, layers, proj):
    C, F = cfg.hidden_size, cfg.intermediate_size
    return 2 * (layers * (4 * C * C + 2 * C * F) + (cfg.projection_dim * C if proj else 0))


def time_calls(fn, calls):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(calls):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        ts.append((e0, e1))
    torch.cuda.synchronize()
    ms = sorted(a.elapsed_time(b) for a, b in ts)
    return ms[len(ms) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.set_grad_enabled(False)
    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    towers, sds = [], []
    for cfg, proj, cls in ((O.CLIP_L, False, B200CLIPTextModel), (O.BIGG, True, B200CLIPTextModelWithProjection)):
        sd = random_sd(cfg, proj, dev)
        m = cls(cfg.hf_kwargs(), device=dev)
        m.load_state_dict(sd)
        towers.append(m)
        sds.append(({k: v.to(torch.bfloat16) for k, v in sd.items()}, cfg, proj))
        del sd
    wbytes = weight_bytes(O.CLIP_L, O.CLIP_L.num_hidden_layers - 1, False) + weight_bytes(O.BIGG, O.BIGG.num_hidden_layers, True)
    res = dict(tool="bench_text_encoders", gpu=smi, weight_bytes_per_call=wbytes, calls=args.calls)
    for n in (2, 16):
        B = n // 2
        pos = [O.make_ids(f"bench/p{t}", B, 77, pad).to(dev) for t, pad in enumerate((O.PAD_CLIP_L, O.PAD_BIGG))]
        neg = [O.make_ids(f"bench/n{t}", B, 77, pad).to(dev) for t, pad in enumerate((O.PAD_CLIP_L, O.PAD_BIGG))]
        ms = time_calls(lambda: encode_prompt(towers, pos, neg), args.calls)
        l0 = ops.LAUNCHES
        encode_prompt(towers, pos, neg, use_cuda_graph=False)
        launches = ops.LAUNCHES - l0
        ms_o = time_calls(lambda: O.encode_prompt(sds, pos, neg, dtype=torch.bfloat16), max(args.calls // 5, 5))
        res[f"n{n}"] = dict(ms=round(ms, 4), oracle_eager_bf16_ms=round(ms_o, 4), speedup=round(ms_o / ms, 2),
                            library_launches_per_call=launches, weight_GBps=round(wbytes / ms / 1e6, 1),
                            weight_stream_share_of_7p7TBps=round(wbytes / ms / 1e6 / (HBM_TBPS * 1e3), 3))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
