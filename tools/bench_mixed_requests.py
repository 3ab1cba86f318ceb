#!/usr/bin/env python
"""Mixed requests in one batch on one GPU, at the c3 shapes (SDXL base + IP adapter, 1024^2 = 128x128 latent, batch 4, CFG,
DDIM, CUDA graph).  Three arms, alternated round by round in one process:

  a  scalar settings: guidance 10, the processors' IP scale (today's path)
  b  per-request settings: guidance (5, 7.5, 10, 12) and IP scale (0.3, 0.6, 0.8, 1.0), new values every round
  c  the scalar path's first generate after ``set_scale`` changed the processors' scale (a fresh graph key: warm-up forward,
     capture, then the trajectory) -- what serving mixed IP scales costs without per-row scales

(a) and (b) are ms per CFG step: a whole ``generate`` call (context K/V, time table, N steps) over N, CUDA events, median of the
rounds.  (c) is the whole first call in ms, and its excess over N steps of (a) (the re-capture).  (c) runs on a sampler of its
own so that its graphs do not evict those of (a) and (b).  Weights are random at the real widths (timing does not depend on
their values).  Prints one JSON line.  Usage: python tools/bench_mixed_requests.py [--steps 50] [--rounds 3]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

import bench
from instructany2pix_b200.attention_processor import B200IPAttnProcessor
from instructany2pix_b200.sampler import B200Sampler

G_MIXED = [5.0, 7.5, 10.0, 12.0]
S_MIXED = [0.3, 0.6, 0.8, 1.0]


def set_scale(unet, s):
    """IPAdapter.set_scale (ip_adapter.py:211-214): the scale of every IP processor"""
    for p in unet.attn_processors.values():
        if isinstance(p, B200IPAttnProcessor):
            p.scale = s


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.set_grad_enabled(False)
    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    B, L, N = 4, 128, args.steps
    unet, _ = bench.build_models(dev, False)
    d = {k: v.to(dev) for k, v in bench.host_inputs(B, L, 1000).items()}
    g = torch.Generator(device=dev).manual_seed(7)
    ctx = torch.cat([d["ctx"], torch.randn(2 * B, 4, 2048, generator=g, device=dev).to(d["ctx"].dtype)], 1)
    added = dict(text_embeds=d["pooled"], time_ids=d["tid"])
    s_ab, s_c = B200Sampler(unet), B200Sampler(unet)
    run = lambda s, **kw: s.generate(d["lat"], ctx, added, num_inference_steps=N, **kw)
    set_scale(unet, 1.0)
    run(s_ab, guidance_scale=10.0)                                       # capture (a) and (b) once, outside the timed rounds
    run(s_ab, guidance_scale=G_MIXED, ip_scale=S_MIXED)
    a, b, c = [], [], []
    for r in range(args.rounds):
        a.append(timed(lambda: run(s_ab, guidance_scale=10.0)) / N)
        gs, ss = G_MIXED[r % B:] + G_MIXED[:r % B], S_MIXED[r % B:] + S_MIXED[:r % B]     # new values every round
        b.append(timed(lambda: run(s_ab, guidance_scale=gs, ip_scale=ss)) / N)
        set_scale(unet, 0.5 + 0.01 * r)                                  # a value no graph was captured for
        c.append(timed(lambda: run(s_c, guidance_scale=10.0)))
        set_scale(unet, 1.0)
    ma, mb, mc = statistics.median(a), statistics.median(b), statistics.median(c)
    print(json.dumps(dict(tool="bench_mixed_requests", gpu=smi, workload="c3 shapes: B=4, 128x128 latent, CFG, DDIM, CUDA graph",
                          steps=N, rounds=args.rounds,
                          a_scalar_ms_per_cfg_step=round(ma, 3), b_per_request_ms_per_cfg_step=round(mb, 3),
                          b_over_a=round(mb / ma, 4),
                          c_first_generate_after_set_scale_ms=round(mc, 1), c_recapture_ms=round(mc - N * ma, 1),
                          a_rounds=[round(v, 3) for v in a], b_rounds=[round(v, 3) for v in b], c_rounds=[round(v, 1) for v in c])))


if __name__ == "__main__":
    main()
