#!/usr/bin/env python
"""Benchmark of the B200-native InstructAny2Pix denoising hot path.

    python bench.py --gpus N --steps K --warmup W [--workload c3|c2|c4|b1|c1] [--impl reference] [--dump-outputs DIR]

A "step" is ONE complete 50-step DDIM + CFG sampling trajectory for the per-GPU batch (the unit of BASELINE.json's
metric, images/sec at 1024^2): 50 x (CUDA-graph replay of the SDXL-class UNet at CFG batch 2B + fused CFG/DDIM kernel),
preceded by the per-request hoisted work (cross-attention K/V of all 70 layers, time-embedding table).  Workloads
(BASELINE.json configs): c3 = 1024^2 (128x128 latent) batch 4 [default: the config the metric is quoted on that fits one
GPU], c2 = 512^2 batch 1, c4 = prior + 1024^2 batch 8, b1 = one interactive 1024^2 request, c1 = the embedding prior alone
(25-step CFG sampling of one sample; its own metric, see bench_prior).  Weights are random-init of the named architecture, inputs
synthetic (no network).  Multi-GPU (torchrun, one rank per GPU): every rank samples its own batch -- whole trajectories
shard by prompt/seed, no collective inside the loop -- so scaling is "weak"; time = max over ranks.

JSON keys beyond the base contract: "roofline" (dominant kernel = tcgen05 implicit GEMM, measured with CUDA events around
every launch of one eager UNet forward), "cpu_baseline" (the oracle port of the reference path on the host cores, bounded
sample, warmed once), "gpu_eager_baseline" (the reference-equivalent PyTorch eager bf16 path -- the oracle's restated modules on
the same GPU, cuDNN / cuBLAS / SDPA -- one CFG UNet step, N = 1 only), "e2e" (whole request batches through the public API and
``parallel.run_sharded``: pinned-host inputs -> device, trajectory, VAE decode, ordered gather of every rank's images on rank 0
(NCCL), device -> host; ``first_batch_sha256`` is identical for every GPU count).

--dump-outputs DIR writes what the last timed step returned to its caller (rank 0) as DIR/<name>.npy in float32: "latents" of
the device-resident trajectory and "e2e_images" of the last end-to-end batch (c1: "embedding" and "e2e_embedding").  Weights
and inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

F_UNET = {128: 6.7104e12, 64: 1.5367e12}          # FLOPs / sample-forward with K,V hoisted (BASELINE.md section 2)
WORKLOADS = {
    "c2": dict(L=64, B=1, prior=False, name="SDXL-class UNet 512^2 (64x64 latent) 50-step DDIM CFG, batch 1"),
    "c3": dict(L=128, B=4, prior=False, name="SDXL-class UNet 1024^2 (128x128 latent) 50-step DDIM CFG, decoupled image+text cross-attn, batch 4"),
    "c4": dict(L=128, B=8, prior=True, name="instruction-edit: prior + 1024^2 UNet sampling, batch 8 per GPU"),
    "b1": dict(L=128, B=1, prior=False, name="single interactive request: SDXL-class UNet 1024^2 50-step DDIM CFG, batch 1"),
    "c1": dict(L=None, B=1, prior=True, name="instructany2pix/prior embedding-prior sampling (GPT-2-medium trunk, 25 DDPM steps, CFG), 1 sample"),
    # the refinement pass every request ends with (pipeline.py:128-131, :358-361: piperf(image=..., strength=0.5); SURVEY 8f-3)
    "rf": dict(L=128, B=4, prior=False, refiner=True, name="SDXL-refiner UNet 1024^2 img2img: strength 0.5 of a 50-step Euler schedule (25 CFG steps), batch 4"),
}
PRIOR_STEPS = 25


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(burst=d["bf16_tflops"], sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), hbm=d["hbm_gbs"], src="measured")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, src="fallback")


def ncu_traffic_prior():
    """DRAM bytes (read + write) of ONE prior_trunk_kernel launch from the committed `ncu --set full` capture (not measured live)."""
    p = os.path.join(ROOT, "profiles", "prior_trunk_traffic_r02.json")
    if os.path.exists(p):
        return json.load(open(p))["dram_bytes_per_launch"]
    return None


def ncu_traffic():
    """DRAM bytes (read + write) per tc_gemm_kernel launch, averaged over the 480 launches of one UNet step, from the committed
    ncu capture (profiles/gemm_traffic_r02.json; not measured live -- a run under ncu is never a bench value)."""
    p = os.path.join(ROOT, "profiles", "gemm_traffic_r02.json")
    if os.path.exists(p):
        return json.load(open(p))["dram_bytes_per_launch"]
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True).start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


DUMP_MAX_ELEMS = 1 << 22          # float32 elements per dumped array (16 MB): the two arrays of a run stay well under 64 MB


def dump_outputs(out_dir, arrays):
    """Write each tensor as ``out_dir/<name>.npy`` in float32.  A tensor of more than DUMP_MAX_ELEMS elements is replaced by a
    sample of its flattened elements at fixed (seeded, ascending) indices, the same on every run."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().to("cpu", torch.float32)
        if t.numel() > DUMP_MAX_ELEMS:
            idx = torch.randint(t.numel(), (DUMP_MAX_ELEMS,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx]
        np.save(os.path.join(out_dir, f"{name}.npy"), t.numpy())


# ------------------------------------------------------------------------------------------------ model + inputs
def build_models(dev, want_prior, refiner=False):
    from instructany2pix_b200.attention_processor import B200IPAttnProcessor
    from instructany2pix_b200.unet import REFINER_CONFIG, B200UNet

    g = torch.Generator(device=dev)
    g.manual_seed(0)
    if refiner:
        unet = B200UNet(device=dev, **REFINER_CONFIG)            # SDXL-refiner config: 2 259 526 660 parameters, text-only cross-attention
    else:
        unet = B200UNet(device=dev)                              # SDXL-base config: 2 567 463 684 parameters
        procs = {}
        for name, p in unet.attn_processors.items():
            if name.endswith("attn2.processor"):
                hs = dict(unet.named_modules())[name[: -len(".processor")]].to_q.weight.shape[0]
                procs[name] = B200IPAttnProcessor(hs, unet.config.cross_attention_dim, scale=1.0, num_tokens=4, device=dev)
            else:
                procs[name] = p
        unet.set_attn_processor(procs)                           # +340 787 200 IP-adapter parameters
    for name, p in unet.named_parameters():                      # PyTorch-default-scale random init, on the device
        if p.ndim >= 2:
            fan_in = p[0].numel()
            p.copy_(((torch.rand(p.shape, generator=g, device=dev) * 2 - 1) * fan_in ** -0.5).to(p.dtype))
        elif name.endswith("weight"):
            p.fill_(1.0)
        else:
            p.copy_(0.02 * torch.randn(p.shape, generator=g, device=dev))
    unet.invalidate()
    prior = None
    if want_prior:
        from instructany2pix_b200.prior import B200Prior
        prior = B200Prior(device=dev)
        for name, p in prior.named_parameters():
            if p.ndim >= 2:
                p.copy_(0.02 * torch.randn(p.shape, generator=g, device=dev))
            elif name.endswith("weight"):
                p.fill_(1.0)
            else:
                p.zero_()
        prior.set_clip_hidden(0.5 * torch.randn(1, 2, 1024, generator=g, device=dev))
    return unet, prior


def build_vae(dev, with_encoder=False):
    """SDXL AutoencoderKL decoder (random init of the named architecture) for the end-to-end leg: latents -> images
    (+ the encoder for the refiner workload: image -> latents)."""
    from instructany2pix_b200.vae import B200VAE
    g = torch.Generator(device=dev)
    g.manual_seed(1)
    vae = B200VAE(device=dev, with_encoder=with_encoder)
    for name, p in vae.named_parameters():
        if p.ndim >= 2:
            fan_in = p[0].numel()
            p.copy_(((torch.rand(p.shape, generator=g, device=dev) * 2 - 1) * fan_in ** -0.5).to(p.dtype))
        elif name.endswith("weight"):
            p.fill_(1.0)
        else:
            p.zero_()
    vae.invalidate()
    return vae


REFINER = False          # set by main() for the "rf" workload: text context 1280 wide, five micro-conditioning ids, an input image


def request_inputs(i, L):
    """Synthetic conditioning of ONE request (SURVEY 8d), a function of its GLOBAL index only: [negative ; positive] prompt tokens,
    pooled embeddings, micro-conditioning ids, start noise, LLM image embedding (refiner: the image to refine instead)."""
    g = torch.Generator()
    g.manual_seed(1000 + i)
    ctx = torch.randn(2, 77, 1280 if REFINER else 2048, generator=g)
    pooled = torch.randn(2, 1280, generator=g)
    H = float(L * 8)
    tid = torch.tensor([[H, H, 0.0, 0.0, 6.0]] if REFINER else [[H, H, 0.0, 0.0, H, H]]).repeat(2, 1)   # refiner: (size, crop, aesthetic score)
    tid[0, -1] = 2.5 if REFINER else tid[0, -1]                 # negative_aesthetic_score
    lat = torch.randn(4, L, L, generator=g)
    e = torch.randn(1, 1024, generator=g)
    e = e / e.norm(dim=-1, keepdim=True) * 100.0
    out = dict(ctx=ctx, pooled=pooled, tid=tid, lat=lat, llm=e)
    if REFINER:
        out["image"] = torch.rand(3, 8 * L, 8 * L, generator=g) * 2 - 1
    return out


def host_batch(indices, L):
    """A request batch in PINNED host memory, laid out as the public API takes it: the [negative ; positive] halves stacked over the
    batch (ip_adapter.py:341-342), what a caller holds before the device sees anything."""
    rs = [request_inputs(i, L) for i in indices]
    pin = lambda t: t.contiguous().pin_memory() if torch.cuda.is_available() else t.contiguous()
    half = lambda k, j: torch.stack([r[k][j] for r in rs])
    out = dict(ctx=pin(torch.cat([half("ctx", 0), half("ctx", 1)])), pooled=pin(torch.cat([half("pooled", 0), half("pooled", 1)])),
               tid=pin(torch.cat([half("tid", 0), half("tid", 1)])), lat=pin(torch.stack([r["lat"] for r in rs])),
               llm=pin(torch.stack([r["llm"] for r in rs])))
    if REFINER:
        out["image"] = pin(torch.stack([r["image"] for r in rs]))
    return out


def host_inputs(B, L, seed):
    """the batch of requests [seed, seed + B) (kept for the tools/ scripts)"""
    return host_batch(list(range(seed, seed + B)), L)


def run_trajectory(hot, dev_in, steps):
    """one request batch: (prior ->) LLM embedding -> ImageProj -> 4 IP tokens appended to the text tokens -> CFG sampling;
    refiner: [image -> VAE encode ->] add_noise at strength 0.5 -> the last half of the Euler schedule, text-only CFG"""
    if REFINER:
        init = dev_in["init"] if "init" in dev_in else hot.vae.encode(dev_in["image"], sample=False)
        return hot.sampler.generate(dev_in["lat"], dev_in["ctx"], dict(text_embeds=dev_in["pooled"], time_ids=dev_in["tid"]),
                                    num_inference_steps=steps, guidance_scale=5.0, init_latents=init, strength=0.5)
    y = None
    if hot.prior is not None:
        y = hot.prior.generate_diffusion(3, 0, dev_in["llm"], device=dev_in["llm"].device, dtype=torch.float32,
                                         num_inference_steps=25, guidance_scale=10, score=6.5)[0]
    ctx = hot.ip_context(dev_in["ctx"], dev_in["llm"], prior_embed=y)
    return hot.sampler.generate(dev_in["lat"], ctx, dict(text_embeds=dev_in["pooled"], time_ids=dev_in["tid"]),
                                num_inference_steps=steps, guidance_scale=10.0)


# ------------------------------------------------------------------------------------------------ roofline of the dominant kernel
def profile_dominant_kernel(unet, sampler, dev_in, B, ctx81):
    """CUDA events around every C-ABI launch of ONE eager UNet forward (CFG batch 2B) on the launching stream."""
    from instructany2pix_b200 import ops
    added = dict(text_embeds=dev_in["pooled"], time_ids=dev_in["tid"])
    kv = unet.context_kv(ctx81)
    rb = unet.time_rowbias_table(torch.tensor([981.0]), added, 2 * B)[0].contiguous()
    x = dev_in["lat"].float()
    for _ in range(2):
        unet.forward_core(x, rb, kv, 2 * B)
    torch.cuda.synchronize()
    ops.PROFILE = []
    unet.forward_core(x, rb, kv, 2 * B)
    torch.cuda.synchronize()
    rec, ops.PROFILE = ops.PROFILE, None
    by, shapes = {}, {}
    for name, flops, e0, e1, tag, nbytes in rec:
        ms = e0.elapsed_time(e1)
        d = by.setdefault(name, dict(ms=0.0, flops=0.0, n=0, bytes=0.0))
        d["ms"] += ms
        d["flops"] += flops
        d["bytes"] += nbytes
        d["n"] += 1
        if tag:
            t = shapes.setdefault(tag, dict(ms=0.0, flops=0.0, n=0))
            t["ms"] += ms
            t["flops"] += flops
            t["n"] += 1
    if os.environ.get("IA2P_BENCH_SHAPES"):
        for tag, t in sorted(shapes.items(), key=lambda kv: -kv[1]["ms"]):
            print(f"# {t['ms']:8.3f} ms  n={t['n']:3d}  {t['flops'] / max(t['ms'], 1e-9) / 1e9:7.1f} TFLOP/s  {tag}", file=sys.stderr)
    return by


# ------------------------------------------------------------------------------------------------ CPU baseline (oracle port)
_CPU_UNET = None


def _cpu_unet(threads):
    """the fp32 oracle restatement at SDXL-base width with decoupled cross-attention processors, built once per process"""
    global _CPU_UNET
    torch.set_num_threads(threads)
    if _CPU_UNET is not None:
        return _CPU_UNET
    from oracle.attention import IPAttnProcessor2_0
    from oracle.unet import SDXL_BASE, OracleUNet
    with torch.device("meta"):
        m = OracleUNet(SDXL_BASE)
    m = m.to_empty(device="cpu")
    procs = {}
    for name, p in m.attn_processors.items():
        if name.endswith("attn2.processor"):
            hs = dict(m.named_modules())[name[: -len(".processor")]].to_q.weight.shape[0]
            procs[name] = IPAttnProcessor2_0(hs, 2048)
        else:
            procs[name] = p
    m.set_attn_processor(procs)
    with torch.no_grad():
        for n, p in m.named_parameters():
            if p.ndim >= 2:
                p.uniform_(-0.02, 0.02)
            elif n.endswith("weight"):
                p.fill_(1.0)
            else:
                p.zero_()
    _CPU_UNET = m
    return m


def cpu_unet_step_seconds(L, threads):
    """One CFG UNet step (2 sample-forwards, batch 1) + the CFG/DDIM arithmetic of the fp32 oracle restatement on the host
    cores (model construction excluded)."""
    m = _cpu_unet(threads)
    with torch.no_grad():
        x = torch.randn(2, 4, L, L)
        ctx = torch.randn(2, 81, 2048)
        added = dict(text_embeds=torch.randn(2, 1280), time_ids=torch.tensor([[L * 8.0, L * 8.0, 0, 0, L * 8.0, L * 8.0]] * 2))
        t0 = time.time()
        eps = m(x, torch.tensor(981), ctx, added_cond_kwargs=added)[0]
        eu, ec = eps.chunk(2)
        _ = 1.0 * x[:1] + 0.1 * (eu + 10.0 * (ec - eu))
        return time.time() - t0


def make_config(wl, world, NS, graph=True):
    """the ``config`` object of the JSON line -- shared by the B200 arm and the reference arm (same workload, same keys)"""
    if wl["L"] is None:
        return dict(workload=wl["name"], per_gpu_batch=wl["B"], num_inference_steps=PRIOR_STEPS, guidance_scale=10.0,
                    parallelism=f"replicas x{world} (whole trajectories per GPU, no in-loop collective)",
                    l2_policy="inputs larger than L2: the 604 MB of trunk weights stream from HBM every step; no explicit flush", cuda_graph=graph)
    return dict(workload=wl["name"], per_gpu_batch=wl["B"], latent=wl["L"], num_inference_steps=NS, guidance_scale=10.0,
                parallelism=f"replicas x{world} (whole trajectories per GPU, no in-loop collective)",
                l2_policy="inputs larger than L2 (5.8 GB weights + activations stream every step); no explicit flush",
                cuda_graph=graph, residual_stream="fp32")


def metric_name(wl):
    if wl.get("refiner"):
        return "images/sec 1024^2 refiner img2img (25 of 50 Euler steps, CFG)"
    if wl["L"] is None:
        return "prior samples/sec (25-step DDPM CFG embedding-prior sampling)"
    return "images/sec 1024^2 50-step DDIM CFG" if wl["L"] == 128 else "images/sec 512^2 50-step DDIM CFG"


# ---- the embedding prior on the host cores (oracle port)
_CPU_PRIOR = None


def cpu_prior_seconds(threads, steps=PRIOR_STEPS):
    """One complete 25-step CFG sampling of one sample with the fp32 oracle restatement of the reference prior (prior/model.py:527-658
    + the GPT-2-medium trunk) on the host cores; model construction excluded."""
    global _CPU_PRIOR
    torch.set_num_threads(threads)
    if _CPU_PRIOR is None:
        from oracle.prior import OraclePrior
        _CPU_PRIOR = OraclePrior(n_layer=24).eval()
    g = torch.Generator().manual_seed(3)
    src = torch.randn(1, 1, 1024, generator=g)
    src = src / src.norm() * 100.0
    clip_hidden = 0.5 * torch.randn(1, 2, 1024, generator=g)
    with torch.no_grad():
        t0 = time.time()
        _CPU_PRIOR.generate_diffusion(3, 0, src, clip_hidden, num_inference_steps=steps, guidance_scale=10, score=6.5)
        return time.time() - t0


def reference_arm(args, wl):
    """--impl reference: the reference's own CPU implementation of the path on all host cores -- the oracle port (diffusers /
    transformers are not installable here and /root/reference does not exist on the GPU box, DESIGN.md section 5), same config
    object, metric and unit as the B200 arm.  Each step is a BOUNDED SAMPLE of the workload, and ``ms_per_step`` is its measured
    time: UNet workloads: one CFG UNet step (2 sample-forwards at batch 1) of the 50 a trajectory has -> images/sec = 1 / (50 t);
    c1: one whole 25-step prior sampling."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    L = wl["L"]
    ts = []
    for i in range(max(args.warmup, 1) + args.steps):
        dt = cpu_prior_seconds(cores) if L is None else cpu_unet_step_seconds(L, cores)
        if i >= max(args.warmup, 1):
            ts.append(dt)
    t = sum(ts) / len(ts)
    if L is None:
        v, unit = 1.0 / t, "samples/sec"
        sample = f"{len(ts)} x one complete {PRIOR_STEPS}-step CFG prior sampling of one sample, fp32 oracle port of prior/model.py:527-658"
    else:
        v, unit = 1.0 / (50.0 * t), "images/sec"
        sample = (f"{len(ts)} x one CFG UNet step (2 sample-forwards, batch 1, {L}x{L} latent) of the fp32 oracle port; "
                  "images/sec = 1 / (50 steps x measured step time), VAE decode not included")
    out = dict(metric=metric_name(wl), value=v, unit=unit, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup, ms_per_step=t * 1e3,
               higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic", impl="reference",
               config=make_config(wl, args.gpus, args.num_inference_steps),
               cpu_baseline=dict(value=v, unit=unit, cores=cores, kind="port", sample=sample),
               e2e=dict(value=v, unit=unit, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(out))


# ------------------------------------------------------------------------------------------------ GPU comparator (PyTorch eager)
def eager_gpu_step_ms(dev, B, L, iters=3):
    """SURVEY 8(d)'s GPU comparator: the reference-equivalent PyTorch EAGER bf16 path on the same B200 -- the oracle's restated SDXL
    UNet + decoupled cross-attention processors moved to the device in bf16 (cuDNN convs, cuBLAS linears, SDPA flash attention,
    K/V re-projected every step, ~2 000 launches per forward) -- one CFG UNet step at the workload's shapes incl. the CFG + DDIM
    arithmetic.  A reported baseline like the CPU one: the oracle is only ever the thing compared against."""
    from oracle.attention import IPAttnProcessor2_0
    from oracle.unet import SDXL_BASE, OracleUNet
    dt = torch.bfloat16
    with torch.device("meta"):
        m = OracleUNet(SDXL_BASE)
    m = m.to_empty(device=dev).to(dt)
    procs = {}
    for name, p in m.attn_processors.items():
        if name.endswith("attn2.processor"):
            hs = dict(m.named_modules())[name[: -len(".processor")]].to_q.weight.shape[0]
            procs[name] = IPAttnProcessor2_0(hs, 2048).to(dev, dt)
        else:
            procs[name] = p
    m.set_attn_processor(procs)
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    for n, p in m.named_parameters():
        if p.ndim >= 2:
            p.copy_(((torch.rand(p.shape, generator=g, device=dev) * 2 - 1) * p[0].numel() ** -0.5).to(dt))
        elif n.endswith("weight"):
            p.fill_(1.0)
        else:
            p.zero_()
    x = torch.randn(B, 4, L, L, device=dev, dtype=dt)
    ctx = torch.randn(2 * B, 81, 2048, device=dev, dtype=dt)
    added = dict(text_embeds=torch.randn(2 * B, 1280, device=dev, dtype=dt),
                 time_ids=torch.tensor([[L * 8.0, L * 8.0, 0, 0, L * 8.0, L * 8.0]] * (2 * B), device=dev, dtype=dt))

    def step():
        eps = m(torch.cat([x, x]), torch.tensor(981, device=dev), ctx, added_cond_kwargs=added)[0]
        eu, ec = eps.chunk(2)
        return 1.0 * x + 0.1 * (eu + 10.0 * (ec - eu))

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    del m
    torch.cuda.empty_cache()
    return ms


# ------------------------------------------------------------------------------------------------ c1: the embedding prior alone
def bench_prior(args, wl, dev, rank, world, local):
    """BASELINE.json configs[0]: the embedding-prior denoiser alone -- one sample, 25 DDPM steps with classifier-free guidance
    (``InstructAny2PixPrior.generate_diffusion``, prior/model.py:527-658; the production call uses no_diffusion=True = 1 step of the
    same loop).  Every step streams the GPT-2-medium trunk (24 layers, 302 M parameters = 604 MB of bf16 weights) through the
    small-M GEMM kernel for 2 CFG rows x 14 tokens: HBM-bound, so the roofline is bytes / time against the measured copy bandwidth."""
    import torch.distributed as dist

    from instructany2pix_b200 import ops
    from instructany2pix_b200.prior import B200Prior
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    prior = B200Prior(device=dev)
    for name, p in prior.named_parameters():
        if p.ndim >= 2:
            p.copy_(0.02 * torch.randn(p.shape, generator=g, device=dev))
        elif name.endswith("weight"):
            p.fill_(1.0)
        else:
            p.zero_()
    prior.set_clip_hidden(0.5 * torch.randn(1, 2, 1024, generator=g, device=dev))
    B = wl["B"]
    hg = torch.Generator().manual_seed(1000 + rank)
    src_h = torch.randn(B, 1, 1024, generator=hg)
    src_h = (src_h / src_h.norm(dim=-1, keepdim=True) * 100.0).pin_memory()
    src_d = src_h.to(dev)
    kw = dict(num_inference_steps=PRIOR_STEPS, guidance_scale=10, score=6.5, dtype=torch.float32)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        prior.generate_diffusion(3, 0, src_d, device=dev, **kw)
    sync_all()
    clocks = ClockSampler(local)
    clocks.start()
    l0 = ops.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        emb, _ = prior.generate_diffusion(3, 0, src_d, device=dev, **kw)       # noise drawn on the device, result stays there
    e1.record()
    sync_all()
    clk = clocks.stop()
    ms = e0.elapsed_time(e1)
    launches_eager = ops.LAUNCHES - l0
    # the captured trunk evaluation alone (one CUDA-graph replay = one prior step's device work but the fused CFG / DDPM kernel)
    trunk_us = None
    if prior.use_cuda_graph and prior._graphs:
        gr = next(iter(prior._graphs.values()))[0]
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        g0.record()
        for _ in range(50):
            gr.replay()
        g1.record()
        torch.cuda.synchronize()
        trunk_us = g0.elapsed_time(g1) * 1e3 / 50
    # kernels per trunk evaluation (graph replays re-issue them)
    ops.PROFILE = []
    prior.use_cuda_graph, keep = False, prior.use_cuda_graph
    prior.generate_diffusion(3, 0, src_d, device=dev, **{**kw, "num_inference_steps": 1})
    torch.cuda.synchronize()
    rec, ops.PROFILE = ops.PROFILE, None
    prior.use_cuda_graph = keep
    per_step_kernels = sum(ops._KERNELS_PER_CALL.get(r[0], 1) for r in rec)
    trunk_ms = sum(r[2].elapsed_time(r[3]) for r in rec if r[0] in ("ia2p_gemm_smallm", "ia2p_prior_trunk"))
    fused = any(r[0] == "ia2p_prior_trunk" for r in rec)
    # end to end: pinned host embedding -> device, sampling, result -> host (the reference call passes device='cpu': pipeline.py:313)
    sync_all()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(args.steps):
        y, _ = prior.generate_diffusion(3, 0, src_h.to(dev, non_blocking=True), device="cpu", **kw)
    f1.record()
    sync_all()
    ms_e2e = f0.elapsed_time(f1)
    if world > 1:
        tt = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms, ms_e2e = tt.tolist()
    if rank != 0:
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(embedding=emb, e2e_embedding=y))
    pk = peaks()
    ms_step = ms / args.steps
    step_us = ms_step * 1e3 / PRIOR_STEPS
    wbytes = sum(p.numel() * 2 for n, p in prior.named_parameters() if p.ndim >= 2 and ".h." in n)      # trunk matrices, bf16
    ach = wbytes / (step_us * 1e-6) / 1e9
    out = dict(metric=metric_name(wl), value=world * B * args.steps / (ms / 1e3), unit="samples/sec", n_gpus=world, steps=args.steps,
               warmup=args.warmup, ms_per_step=ms_step, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16 weights, fp32 activations (hi/lo split)",
               data="synthetic", config=make_config(wl, world, PRIOR_STEPS, prior.use_cuda_graph), prior_step_us=step_us, clocks=clk,
               e2e=dict(value=world * B * args.steps / (ms_e2e / 1e3), unit="samples/sec",
                        h2d_bytes_per_step=src_h.numel() * 4 + B * 1024 * 4 * PRIOR_STEPS, d2h_bytes_per_step=B * 1024 * 4,
                        includes="H2D of the LLM embedding, 25 CFG steps with the per-step noise drawn on the host like the reference call "
                                 "(device='cpu', pipeline.py:313) and copied in, D2H of the embedding"),
               gpu_launches=int(launches_eager + (args.steps * PRIOR_STEPS * per_step_kernels if prior.use_cuda_graph else 0)),
               roofline=dict(kernel=("prior_trunk_kernel (the whole GPT-2-medium trunk of a step as one persistent cooperative kernel, 128 CTAs, grid "
                                     "barriers between phases; " if fused else "gemm_smallm_kernel (GPT-2-medium trunk, ") + "M = 2 CFG rows x 14 tokens)", bound="hbm", achieved=ach, peak=pk["hbm"],
                             unit="GB/s", frac=ach / pk["hbm"], traffic=ncu_traffic_prior() if fused else None, peak_source=pk["src"] + " hbm_gbs",
                             algorithmic_bytes_per_step=wbytes, launches_per_step=per_step_kernels, eager_trunk_gemm_ms_per_step=trunk_ms,
                             trunk_graph_replay_us=trunk_us, trunk_graph_gbs=None if not trunk_us else wbytes / (trunk_us * 1e-6) / 1e9,
                             floor_us=wbytes / (pk["hbm"] * 1e9) * 1e6))
    if not args.no_cpu_baseline and world == 1:
        cores = os.cpu_count() or 1
        cpu_prior_seconds(cores)
        t = cpu_prior_seconds(cores)
        out["cpu_baseline"] = dict(value=1.0 / t, unit="samples/sec", cores=cores, kind="port",
                                   sample=f"one complete {PRIOR_STEPS}-step CFG prior sampling of one sample (after one warm-up run) with the fp32 "
                                          f"oracle port of prior/model.py:527-658 = {t:.2f} s; the reference's own prior code runs only in the "
                                          "build container (profiles/prior_reference_cpu_r02.json: same speed as the port)")
    print(json.dumps(out))


# ------------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--num-inference-steps", type=int, default=50)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the b200 implementation")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        return reference_arm(args, wl)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG", "WARN")               # keep NCCL's version banner out of stdout: ONE JSON line
        dist.init_process_group("nccl", device_id=dev)
    torch.set_grad_enabled(False)
    torch.manual_seed(1234)                                       # every rank builds the SAME random-init weights (incl. default-init modules)
    if wl["L"] is None:
        bench_prior(args, wl, dev, rank, world, local)
        if world > 1:
            dist.destroy_process_group()
        return

    import hashlib

    from instructany2pix_b200 import ops, parallel
    global REFINER
    REFINER = bool(wl.get("refiner"))
    L, B, NS = wl["L"], wl["B"], args.num_inference_steps
    unet, prior = build_models(dev, wl["prior"], refiner=REFINER)
    vae = build_vae(dev, with_encoder=REFINER)
    from instructany2pix_b200.hotpath import B200HotPath
    from instructany2pix_b200.image_proj import B200ImageProj
    from instructany2pix_b200.scheduler import B200EulerDiscreteScheduler
    proj = B200ImageProj(device=dev)                             # Linear(1024 -> 4 x 2048) + LayerNorm(2048), PyTorch-default init
    hot = B200HotPath(unet, vae, scheduler=B200EulerDiscreteScheduler() if REFINER else None, prior=prior,
                      use_cuda_graph=not args.no_graph, image_proj=proj)
    sampler = hot.sampler
    n_unet_steps = int(NS * 0.5) if REFINER else NS              # img2img at strength 0.5 runs the last half of the schedule
    host = host_batch(list(range(rank * B, rank * B + B)), L)    # device-resident leg: this rank's first request batch
    dev_in = {k: v.to(dev) for k, v in host.items()}
    if REFINER:                                                  # device-resident leg: the image is already encoded
        dev_in["init"] = vae.encode(dev_in.pop("image"), sample=False)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(max(args.warmup, 1)):
        lat_w = run_trajectory(hot, dev_in, NS)
    vae.decode(lat_w)                                            # warm-up of the decode path (function attributes, allocator)
    # ---- device-resident timing (value)
    sync_all()
    clocks = ClockSampler(local)
    clocks.start()
    l0 = ops.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        lat = run_trajectory(hot, dev_in, NS)
    e1.record()
    sync_all()
    clk = clocks.stop()
    ms = e0.elapsed_time(e1)
    launches_eager = ops.LAUNCHES - l0
    # ---- end to end through the public API: `steps` request batches per GPU, dealt out in whole batches over the ranks
    # (parallel.run_sharded): pinned host inputs -> device, trajectory, VAE decode, ordered gather of all images on rank 0 over
    # NCCL, device -> host.  Request contents and seeds are functions of the GLOBAL request index and batches are the same for every
    # GPU count, so the images (first_batch_sha256: requests 0..B-1) are bit-identical for 1, 2, 4 and 8 GPUs.
    n_items = world * B * args.steps
    mine = parallel.shard_indices(n_items, rank, world, B)
    pinned = {tuple(mine[c:c + B]): host_batch(mine[c:c + B], L) for c in range(0, len(mine), B)}     # what the callers hold
    h2d = sum(v.numel() * v.element_size() for hb in pinned.values() for v in hb.values()) * world / args.steps
    t_dec = []

    def work(idxs):
        cur = {k: v.to(dev, non_blocking=True) for k, v in pinned[tuple(idxs)].items()}
        out = run_trajectory(hot, cur, NS)
        v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        v0.record()
        img = vae.decode(out)                                    # sdxl_pipeline.py:859-871: latents -> (B,3,8L,8L) images
        v1.record()
        t_dec.append((v0, v1))
        return img

    # the caller's result buffer: page-locked, allocated once outside the timed region like the pinned inputs above (a pageable
    # destination made the read-back of the 96 fp32 images of an 8-GPU job 4 % of its end-to-end time)
    res = torch.empty((n_items, 3, 8 * L, 8 * L), dtype=torch.float32, pin_memory=True) if rank == 0 else None
    sync_all()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    gathered = parallel.run_sharded(n_items, B, work)            # rank 0: [n_items, 3, 8L, 8L] on the device, global order
    if rank == 0:
        res.copy_(gathered, non_blocking=True)                   # device -> host read of every image of the job
    f1.record()
    sync_all()
    ms_e2e = f0.elapsed_time(f1)
    ms_decode = t_dec[-1][0].elapsed_time(t_dec[-1][1])          # last batch's decode
    if world > 1:
        tt = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms, ms_e2e = tt.tolist()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    d2h = res.numel() * res.element_size() / args.steps
    sha = hashlib.sha256(res[:B].numpy().tobytes()).hexdigest()[:16]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(latents=lat, e2e_images=res[-B:]))

    pk = peaks()
    ms_step = ms / args.steps
    value = world * B * args.steps / (ms / 1e3)
    e2e_value = n_items / (ms_e2e / 1e3)
    unet_step_ms = ms_step / n_unet_steps
    # launches: graph replays re-issue the captured kernels
    by = profile_dominant_kernel(unet, sampler, dev_in, B, dev_in["ctx"] if REFINER else hot.ip_context(dev_in["ctx"], dev_in["llm"]))
    # FLOPs of one CFG step: the analytic count of the SDXL-base forward (BASELINE.md section 2), else what the ops of one forward count
    step_flops = 2 * B * F_UNET[L] if not REFINER else sum(d["flops"] for d in by.values())
    whole_frac = step_flops / (unet_step_ms * 1e-3) / (pk["sustained"] * 1e12)
    n_forward_kernels = sum(d["n"] * ops._KERNELS_PER_CALL.get(k, 1) for k, d in by.items())
    gpu_launches = launches_eager + (0 if args.no_graph else args.steps * n_unet_steps * n_forward_kernels)
    tc = dict(ms=0.0, flops=0.0, n=0, bytes=0.0)
    for k in ("ia2p_gemm_bf16", "ia2p_gemm_ln_bf16", "ia2p_conv3x3_nhwc_bf16", "ia2p_conv_up2x_nhwc_bf16"):
        if k in by:
            for f in tc:
                tc[f] += by[k][f] * (ops._KERNELS_PER_CALL.get(k, 1) if f == "n" else 1)
    total_ms = sum(d["ms"] for d in by.values())
    ach = tc["flops"] / (tc["ms"] * 1e-3) / 1e12 if tc["ms"] else 0.0
    roof = dict(kernel="tc_gemm_kernel (tcgen05 implicit GEMM: linears + 3x3 convs)", bound="tensor", achieved=ach,
                peak=pk["sustained"], unit="TFLOP/s", frac=ach / pk["sustained"], traffic=ncu_traffic(), peak_source=pk["src"] + " bf16_tflops_sustained",
                frac_of_burst=ach / pk["burst"], frac_of_nominal_2250=ach / 2250.0,
                algorithmic_bytes_per_launch=tc["bytes"] / max(tc["n"], 1), algorithmic_flops_per_launch=tc["flops"] / max(tc["n"], 1),
                launches_per_forward=tc["n"], avg_launch_ms=tc["ms"] / max(tc["n"], 1), share_of_forward=tc["ms"] / total_ms if total_ms else None,
                forward_breakdown_ms={k: round(d["ms"], 3) for k, d in sorted(by.items(), key=lambda kv: -kv[1]["ms"])})
    out = dict(metric=metric_name(wl), value=value, unit="images/sec", n_gpus=world, steps=args.steps, warmup=args.warmup, ms_per_step=ms_step,
               higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16", data="synthetic",
               config=make_config(wl, world, NS, not args.no_graph),
               unet_step_ms=unet_step_ms, unet_tensor_frac=whole_frac, unet_tensor_frac_of_burst=step_flops / (unet_step_ms * 1e-3) / (pk["burst"] * 1e12),
               unet_tensor_frac_of_nominal_2250=step_flops / (unet_step_ms * 1e-3) / 2.25e15, clocks=clk,
               e2e=dict(value=e2e_value, unit="images/sec", h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                        includes="per request batch: H2D of the text conditioning + LLM embedding + noise, (prior,) image projector -> IP tokens, "
                                 "50-step trajectory, VAE decode to fp32 images; then ordered gather of every rank's images on rank 0 (NCCL) and D2H",
                        requests=n_items, first_batch_sha256=sha, vae_decode_ms=ms_decode),
               gpu_launches=int(gpu_launches), roofline=roof)
    if REFINER:
        out["config"].update(num_inference_steps=NS, strength=0.5, unet_steps=n_unet_steps, guidance_scale=5.0, scheduler="EulerDiscrete")
        out["e2e"]["includes"] = ("per request batch: H2D of the image to refine + text conditioning + noise, VAE encode, add_noise, 25 CFG steps of the "
                                  "refiner UNet, VAE decode to fp32 images; then ordered gather on rank 0 and D2H")
    if world == 1 and not args.no_eager_baseline and not REFINER:
        t = eager_gpu_step_ms(dev, B, L)
        out["gpu_eager_baseline"] = dict(unet_step_ms=t, value=B / (NS * t * 1e-3), unit="images/sec", speedup_of_this_build=t / unet_step_ms,
                                         what="PyTorch eager bf16 (the oracle's restated UNet + processors on the same GPU: cuDNN / cuBLAS / SDPA), "
                                              "one CFG UNet step incl. CFG + DDIM arithmetic, x50 for images/sec")
    if not args.no_cpu_baseline and world == 1 and not REFINER:  # contract: rank 0 at N = 1 only
        cores = os.cpu_count() or 1
        cpu_unet_step_seconds(L, cores)                          # warm-up: allocator, thread pool, oneDNN primitives
        t = cpu_unet_step_seconds(L, cores)
        out["cpu_baseline"] = dict(value=1.0 / (50.0 * t), unit="images/sec", cores=cores, kind="port",
                                   sample=f"1 CFG UNet step (2 sample-forwards, batch 1, {L}x{L} latent) of the fp32 oracle port after one "
                                          f"warm-up step = {t:.1f} s; images/sec = 1 / (50 x that)")
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
