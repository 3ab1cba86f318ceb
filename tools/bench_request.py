"""One whole 1024^2 edit request on the B200, stage by stage: VAE encode -> DDIM inversion (25 steps) -> polar start latent ->
CFG generation (25 Euler steps) -> decode to 8-bit images -> refinement pass (strength 0.5 of a 50-step Euler schedule: refiner
encode of the 8-bit images, 25 CFG steps of the SDXL-refiner UNet, decode), at batch 1 and 4.  Full-width SDXL base (with IP
processors), refiner and VAE with random weights (``bench.build_models`` / ``build_vae``).

Prints one JSON line: per-stage milliseconds from CUDA events (the stages ``B200HotPath.edit`` runs, called one by one, plus one
timed ``edit`` call end to end), the two 8-bit image kernels' DRAM rates against the 7.7 TB/s HBM3e figure (L2 overwritten with a
256 MB write before every timed launch), and the device-to-host copy of the request's images as fp32 NCHW against uint8 NHWC
(pinned host buffers).  The card's name, power limit and maximum SM clock are read in the same process.

    python tools/bench_request.py [--batches 1 4] [--reps 2] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12        # HGX B200 data sheet, one GPU


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")] if q.returncode == 0 else (torch.cuda.get_device_name(), None, None)
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def timed(fn, events):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    events.append((e0, e1))
    return out


def request_inputs(B, dev):
    g = torch.Generator().manual_seed(B)
    H = 1024.0
    r = lambda *s: torch.randn(*s, generator=g).to(dev)
    img = (torch.rand(B, 3, 1024, 1024, generator=g) * 2 - 1).to(dev)
    return dict(image=img, ctx_inv=r(B, 77, 2048), added_inv=dict(text_embeds=r(B, 1280), time_ids=torch.tensor([[H, H, 0, 0, H, H]] * B).to(dev)),
                ctx_cfg=r(2 * B, 81, 2048), added_cfg=dict(text_embeds=r(2 * B, 1280), time_ids=torch.tensor([[H, H, 0, 0, H, H]] * 2 * B).to(dev)),
                ctx_rf=r(2 * B, 77, 1280),
                added_rf=dict(text_embeds=r(2 * B, 1280), time_ids=torch.tensor([[H, H, 0, 0, 2.5]] * B + [[H, H, 0, 0, 6.0]] * B).to(dev)))


def run_stages(hot, x, steps, rf_steps, strength):
    """the stages of B200HotPath.edit(..., refinement=strength), each between CUDA events -> {stage: (start, end)}"""
    from instructany2pix_b200.sampler import randn_per_request
    from instructany2pix_b200.scheduler import B200DDIMScheduler
    ev = {}
    t = lambda name, fn: timed(fn, ev.setdefault(name, []))
    z0 = t("encode", lambda: hot.vae.encode(x["image"]))
    inv = B200DDIMScheduler.from_config(hot.sampler.scheduler.config)
    z_inv = t("invert", lambda: hot.sampler.invert(z0, x["ctx_inv"], x["added_inv"], num_inference_steps=steps, scheduler=inv))
    z_t = t("start_latent", lambda: hot.sampler.start_latent(z_inv, alpha=0.7))
    z = t("generate", lambda: hot.sampler.generate(z_t, x["ctx_cfg"], x["added_cfg"], num_inference_steps=steps, guidance_scale=10.0))
    u8 = t("decode_u8", lambda: hot.vae.decode(z, output="u8"))
    z0r = t("refiner_encode_u8", lambda: hot.refiner_vae.encode(u8))
    zr = t("refiner_generate", lambda: hot.refiner.generate(randn_per_request(z0r.shape, z0r.device), x["ctx_rf"], x["added_rf"],
                                                            num_inference_steps=rf_steps, guidance_scale=5.0, init_latents=z0r,
                                                            strength=strength))
    t("refiner_decode_float", lambda: hot.refiner_vae.decode(zr))
    t("refiner_decode_u8", lambda: hot.refiner_vae.decode(zr, output="u8"))
    return ev


def kernel_rates(B, dev, reps=20):
    """ops.image_u8 on the padded conv_out tensor and ops.conv_in_u8 with the SDXL encoder's conv_in, each launch after a 256 MB
    write that evicts L2.  DRAM bytes: image_u8 touches one 32-byte sector per pixel (its 16-byte read) and writes 3 bytes;
    conv_in_u8 reads 3 bytes and writes 128 fp32 channels per pixel."""
    from instructany2pix_b200 import ops
    npix = B * 1024 * 1024
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    y = torch.randn(B, 1024, 1024, 32, device=dev)
    u8 = torch.randint(0, 256, (B, 1024, 1024, 3), dtype=torch.uint8, device=dev)
    w, b = torch.randn(128, 3, 3, 3, device=dev) * 0.2, torch.randn(128, device=dev)
    cases = dict(image_u8=(lambda: ops.image_u8(y), npix * (32 + 3)),
                 conv_in_u8=(lambda: ops.conv_in_u8(u8, w, b, out_dtype=torch.float32), npix * (3 + 128 * 4)))
    out = {}
    for name, (fn, nbytes) in cases.items():
        fn()
        ev = []
        for _ in range(reps):
            flush.fill_(1)
            timed(fn, ev)
        torch.cuda.synchronize()
        ms = statistics.median(a.elapsed_time(e) for a, e in ev)
        out[name] = dict(ms=round(ms, 4), dram_bytes=nbytes, gb_per_s=round(nbytes / ms / 1e6, 1),
                         share_of_7_7_tb_s=round(nbytes / (ms * 1e-3) / HBM_BYTES_PER_S, 3))
    return out


def d2h(B, dev, reps=10):
    """device-to-host copy of the request's images into pinned memory: fp32 (B,3,H,W) against uint8 (B,H,W,3)"""
    out = {}
    for name, t in (("fp32_nchw", torch.randn(B, 3, 1024, 1024, device=dev)),
                    ("u8_nhwc", torch.randint(0, 256, (B, 1024, 1024, 3), dtype=torch.uint8, device=dev))):
        host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        host.copy_(t, non_blocking=True)
        ev = []
        for _ in range(reps):
            timed(lambda: host.copy_(t, non_blocking=True), ev)
        torch.cuda.synchronize()
        ms = statistics.median(a.elapsed_time(e) for a, e in ev)
        nbytes = t.numel() * t.element_size()
        out[name] = dict(bytes=nbytes, ms=round(ms, 4), gb_per_s=round(nbytes / ms / 1e6, 1))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[1, 4])
    ap.add_argument("--steps", type=int, default=25)
    ap.add_argument("--refiner-steps", type=int, default=50)
    ap.add_argument("--refinement", type=float, default=0.5)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_request.py measures on a CUDA device; none found")
    torch.set_grad_enabled(False)
    import bench
    from instructany2pix_b200.hotpath import B200HotPath
    from instructany2pix_b200.sampler import B200Sampler
    from instructany2pix_b200.scheduler import B200EulerDiscreteScheduler
    dev = torch.device("cuda", 0)
    info = gpu_info()
    unet, _ = bench.build_models(dev, False)
    rf_unet, _ = bench.build_models(dev, False, refiner=True)
    vae = bench.build_vae(dev, with_encoder=True)
    hot = B200HotPath(unet, vae, scheduler=B200EulerDiscreteScheduler(),
                      refiner=B200Sampler(rf_unet, scheduler=B200EulerDiscreteScheduler()))
    result = dict(tool="tools/bench_request.py", gpu=info, steps=args.steps, refiner_steps=args.refiner_steps,
                  refinement=args.refinement, batches={})
    for B in args.batches:
        x = request_inputs(B, dev)
        run_stages(hot, x, args.steps, args.refiner_steps, args.refinement)          # warm-up: graph captures, workspaces
        per = []
        for _ in range(args.reps):
            ev = run_stages(hot, x, args.steps, args.refiner_steps, args.refinement)
            torch.cuda.synchronize()
            per.append({k: v[0][0].elapsed_time(v[0][1]) for k, v in ev.items()})
        stages = {k: round(statistics.median(p[k] for p in per), 2) for k in per[0]}
        edit_ev = []
        for _ in range(args.reps):
            timed(lambda: hot.edit(x["image"], x["ctx_inv"], x["added_inv"], x["ctx_cfg"], x["added_cfg"], num_inference_steps=args.steps,
                                   refiner_ctx=x["ctx_rf"], refiner_added=x["added_rf"], refinement=args.refinement,
                                   refiner_steps=args.refiner_steps, output="u8"), edit_ev)
        torch.cuda.synchronize()
        result["batches"][str(B)] = dict(
            stages_ms=stages, stages_sum_ms=round(sum(v for k, v in stages.items() if k != "refiner_decode_float"), 2),
            edit_u8_ms=round(statistics.median(a.elapsed_time(e) for a, e in edit_ev), 2),
            u8_kernels=kernel_rates(B, dev), d2h=d2h(B, dev))
        del x
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
