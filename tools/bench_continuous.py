#!/usr/bin/env python
"""Continuous batching against static batches on one GPU, at the c3 shapes (SDXL base + IP adapter, 1024^2 = 128x128 latent,
S = 4 slots / batch 4, CFG, DDIM, CUDA graph).  Prints one JSON line with the GPU name and power limit.

  a  overhead: ``B200Sampler.generate`` at batch 4 against ``B200ContinuousSampler`` with all four slots busy (four requests
     submitted together, then drained), ms per CFG step = a whole call (context K/V, time tables, N steps) over N, CUDA events,
     median of the rounds; the two arms alternate round by round.
  b  a fixed trace of 16 requests mixing 25 and 50 steps, arrivals given as step indices (arrival time = index x the measured
     ms per step of (a)'s engine arm).  The engine serves it step by step (a request is submitted at the boundary of its
     arrival index; a boundary with nothing pending costs one idle step of time and no GPU work).  The static arm is what a
     caller does without the engine: FIFO batches of up to 4 requests of one step count, run one after another with
     ``generate`` (one sampler per batch size, all captured before timing, so no re-capture is timed).  Per arm: makespan,
     mean and p95 latency (arrival to result), and slot occupancy (useful row-steps over 4 x steps run).

Weights are random at the real widths (timing does not depend on their values).
Usage: python tools/bench_continuous.py [--steps 50] [--rounds 3]"""
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
from instructany2pix_b200.batcher import B200ContinuousSampler
from instructany2pix_b200.sampler import B200Sampler

TRACE_STEPS = [50, 25, 25, 50, 25, 50, 25, 25, 50, 25, 50, 50, 25, 25, 50, 25]
TRACE_ARRIVAL = [0, 0, 0, 0, 5, 10, 10, 15, 20, 30, 30, 40, 50, 60, 60, 70]


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def p95(v):
    v = sorted(v)
    return v[min(len(v) - 1, int(round(0.95 * (len(v) - 1))))]


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
    pair = lambda i: (d["lat"][i:i + 1], ctx[[i, B + i]], {k: v[[i, B + i]] for k, v in added.items()})

    # ---- (a) overhead with all slots busy
    sampler = B200Sampler(unet)
    cs = B200ContinuousSampler(unet, slots=B, latent_hw=(L, L), max_steps=max(N, max(TRACE_STEPS)))

    def engine_full():
        for i in range(B):
            cs.submit(*pair(i), num_inference_steps=N, guidance_scale=10.0)
        cs.drain()

    run_gen = lambda: sampler.generate(d["lat"], ctx, added, num_inference_steps=N, guidance_scale=10.0)
    run_gen()
    engine_full()                                                   # capture both outside the timed rounds
    a_gen, a_eng = [], []
    for _ in range(args.rounds):
        a_gen.append(timed(run_gen) / N)
        a_eng.append(timed(engine_full) / N)
    t_step = statistics.median(a_eng)

    # ---- (b) the trace, engine
    n_req = len(TRACE_STEPS)
    cs.useful_row_steps = cs.executed_row_steps = 0
    torch.cuda.synchronize()
    t0 = torch.cuda.Event(enable_timing=True)
    t0.record()
    events, idle_before, finish, rid_of = [], [], {}, {}
    idle, i = 0, 0
    while len(finish) < n_req:
        for j in range(n_req):
            if TRACE_ARRIVAL[j] == i:
                r = cs.submit(*pair(j % B), num_inference_steps=TRACE_STEPS[j], guidance_scale=10.0)
                rid_of[r] = j
        if cs.pending():
            done = cs.step()
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            events.append(ev)
            idle_before.append(idle)
            for r, _ in done:
                finish[rid_of[r]] = len(events) - 1
        else:
            idle += 1                                               # nothing pending: one step of time passes, no GPU work
        i += 1
    torch.cuda.synchronize()
    clock = [t0.elapsed_time(ev) + idle_before[k] * t_step for k, ev in enumerate(events)]      # end of step k
    eng_lat = [clock[finish[j]] - TRACE_ARRIVAL[j] * t_step for j in range(n_req)]
    eng = dict(makespan_ms=round(clock[-1], 1), mean_latency_ms=round(statistics.mean(eng_lat), 1),
               p95_latency_ms=round(p95(eng_lat), 1), occupancy=round(cs.useful_row_steps / cs.executed_row_steps, 4),
               replays=len(events), idle_steps=idle)

    # ---- (b) the trace, static FIFO batches per step count
    samplers = {b: B200Sampler(unet) for b in range(1, B + 1)}
    for b, s in samplers.items():                                   # capture every batch size outside the timed run
        s.generate(d["lat"][:b], torch.cat([ctx[:b], ctx[B:B + b]]), {k: torch.cat([v[:b], v[B:B + b]]) for k, v in added.items()},
                   num_inference_steps=25, guidance_scale=10.0)
    waiting, now, st_lat, rows_run = [], 0.0, [0.0] * n_req, 0
    pending = sorted(range(n_req), key=lambda j: TRACE_ARRIVAL[j])
    while pending or waiting:
        waiting += [j for j in pending if TRACE_ARRIVAL[j] * t_step <= now]
        pending = [j for j in pending if TRACE_ARRIVAL[j] * t_step > now]
        if not waiting:
            now = TRACE_ARRIVAL[pending[0]] * t_step
            continue
        n_steps = TRACE_STEPS[waiting[0]]
        batch = [j for j in waiting if TRACE_STEPS[j] == n_steps][:B]
        waiting = [j for j in waiting if j not in batch]
        b = len(batch)
        idx = [j % B for j in batch]
        lat = torch.cat([d["lat"][k:k + 1] for k in idx])
        c = torch.cat([ctx[idx], ctx[[B + k for k in idx]]])
        a = {k: torch.cat([v[idx], v[[B + q for q in idx]]]) for k, v in added.items()}
        now += timed(lambda: samplers[b].generate(lat, c, a, num_inference_steps=n_steps, guidance_scale=10.0))
        rows_run += B * n_steps
        for j in batch:
            st_lat[j] = now - TRACE_ARRIVAL[j] * t_step
    useful = sum(TRACE_STEPS)
    static = dict(makespan_ms=round(now, 1), mean_latency_ms=round(statistics.mean(st_lat), 1), p95_latency_ms=round(p95(st_lat), 1),
                  occupancy=round(useful / rows_run, 4))

    print(json.dumps(dict(tool="bench_continuous", gpu=smi, workload="c3 shapes: S = 4 / batch 4, 128x128 latent, CFG, DDIM, CUDA graph",
                          steps=N, rounds=args.rounds,
                          a_generate_ms_per_cfg_step=round(statistics.median(a_gen), 3),
                          a_engine_ms_per_cfg_step=round(t_step, 3),
                          a_engine_over_generate=round(t_step / statistics.median(a_gen), 4),
                          a_generate_rounds=[round(v, 3) for v in a_gen], a_engine_rounds=[round(v, 3) for v in a_eng],
                          b_trace=dict(steps=TRACE_STEPS, arrival_step=TRACE_ARRIVAL), b_engine=eng, b_static_fifo=static)))


if __name__ == "__main__":
    main()
