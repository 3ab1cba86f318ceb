"""Continuous (in-flight) batching of the CFG sampling loop: ``B200ContinuousSampler``.

The UNet batch is a fixed set of S **slots**.  Each slot runs one request at its own position in its own schedule, so requests
with different step counts, img2img strengths, guidance and IP scales share one batch, and a slot whose request finishes is
refilled at the next step boundary instead of waiting for the whole batch.  Per step the device sees ONE CUDA-graph replay:

  * ``ia2p_rowbias_gather``: every slot's time-embedding row and step coefficients (g, c_x, c_e, s_in) from per-slot tables at the
    slot's step counter, which the same call then advances on the device (the host uploads nothing per step);
  * ``B200UNet.forward_core`` at UNet batch 2S (slot s owns rows s and S + s, CFG order [uncond slots ; cond slots]) with per-row
    IP scales;
  * ``ia2p_cfg_step_coef_rows``: the CFG combine + scheduler update with per-row coefficients, and for Euler the slot's next
    scaled UNet input.

An idle slot reads the tables' last (sentinel) row: zero time bias and the identity update g = 0, c_x = 1, c_e = 0, which leaves its
latents unchanged.  Admission (K/V rows, time table, coefficient rows, IP scale, start latent) is enqueued on the stream outside
the graph, through pinned staging buffers; nothing in ``submit`` or ``step`` waits for the device.

Supported: DDIM and Euler (the base loop and the refiner's img2img loop, per-request ``strength``).  Not slotted: LCM (it
re-noises after the update), inpainting, the inversion pass of ``B200HotPath.edit``.  Idle slots still cost compute: the UNet
batch does not shrink.
"""
from __future__ import annotations

import collections
import math

import torch

from . import ops
from .scheduler import B200DDIMScheduler, B200EulerDiscreteScheduler, B200LCMScheduler

_IDENTITY = (0.0, 1.0, 0.0, 1.0)          # (g, c_x, c_e, s_in) of the sentinel row: x unchanged


class B200ContinuousSampler:
    def __init__(self, unet, slots=4, latent_hw=(128, 128), scheduler=None, max_steps=50, n_text=77, n_ip=4,
                 use_cuda_graph=True):
        scheduler = scheduler if scheduler is not None else B200DDIMScheduler()
        if isinstance(scheduler, B200LCMScheduler) or not isinstance(scheduler, (B200DDIMScheduler, B200EulerDiscreteScheduler)):
            raise NotImplementedError(f"{type(scheduler).__name__}: continuous batching runs DDIM and Euler (LCM re-noises after "
                                      "the update)")
        if int(getattr(unet.config, "in_channels", 4)) != 4:
            raise NotImplementedError("continuous batching runs 4-channel UNets (no 9-channel inpainting)")
        if slots < 1 or max_steps < 1 or n_text < 1 or n_ip < 0:
            raise ValueError(f"slots {slots}, max_steps {max_steps}, n_text {n_text}, n_ip {n_ip}")
        self.unet = unet
        self.scheduler = scheduler
        self.S = int(slots)
        self.hw = (int(latent_hw[0]), int(latent_hw[1]))
        self.max_steps = int(max_steps)
        self.n_text, self.n_ip = int(n_text), int(n_ip)
        self.use_cuda_graph = use_cuda_graph
        self.euler = hasattr(scheduler, "input_scale")      # the UNet sees x / sqrt(sigma^2 + 1); DDIM: x itself
        self._queue = collections.deque()
        self._slots = [None] * self.S
        self._next_rid = 0
        self._buf = None
        self._staging = collections.deque()                   # (event, pinned tensors) until the copies have run
        self.captures = 0
        self.executed_row_steps = 0                           # S per replay
        self.useful_row_steps = 0                             # slots that ran a request step

    # ------------------------------------------------------------------ requests
    @torch.no_grad()
    def submit(self, noise, ctx, added_pair, num_inference_steps=50, guidance_scale=10.0, ip_scale=None, init_latents=None,
               strength=1.0, inpaint_mask=None):
        """Queue one request; returns its id at once.  ``noise`` (1, 4, H, W); ``ctx`` (2, n_text + n_ip, D) = [uncond; cond];
        ``added_pair``: text_embeds (2, P), time_ids (2, k).  ``init_latents`` + ``strength`` < 1: img2img, only the last
        int(N * strength) steps run from ``add_noise(init_latents, noise, t_start)``.  ``ip_scale`` None: the processors' scale
        now.  Every argument is checked here, before any device work."""
        if inpaint_mask is not None:
            raise NotImplementedError("inpainting is not slotted: use B200Sampler.generate(inpaint_mask=...)")
        N = int(num_inference_steps)
        if not 1 <= N <= self.max_steps:
            raise ValueError(f"num_inference_steps {num_inference_steps} outside 1..max_steps = {self.max_steps}")
        shape = (1, 4) + self.hw
        if tuple(noise.shape) != shape:
            raise ValueError(f"noise: expected latents of shape {shape}, got {tuple(noise.shape)}")
        if init_latents is None and strength != 1.0:
            raise ValueError(f"strength {strength} needs init_latents")
        if init_latents is not None and tuple(init_latents.shape) != shape:
            raise ValueError(f"init_latents: expected latents of shape {shape}, got {tuple(init_latents.shape)}")
        unet = self.unet
        n_ip_unet, proc_scale = unet._ip_state()
        if n_ip_unet != self.n_ip:
            raise ValueError(f"the UNet's processors take {n_ip_unet} IP tokens, the engine was built for n_ip = {self.n_ip}")
        D = int(unet.config.cross_attention_dim)
        if tuple(ctx.shape) != (2, self.n_text + self.n_ip, D):
            raise ValueError(f"ctx: expected (2, n_text + n_ip = {self.n_text} + {self.n_ip}, {D}), got {tuple(ctx.shape)}")
        te, tid = added_pair["text_embeds"], added_pair["time_ids"]
        if te.ndim != 2 or te.shape[0] != 2 or tid.ndim != 2 or tid.shape[0] != 2:
            raise ValueError(f"added_pair: text_embeds and time_ids need 2 rows, got {tuple(te.shape)} and {tuple(tid.shape)}")
        g = float(guidance_scale)
        if not math.isfinite(g):
            raise ValueError(f"guidance_scale: non-finite value {guidance_scale}")
        if ip_scale is not None:
            if self.n_ip == 0:
                raise ValueError("ip_scale given, but the UNet has no IP-adapter processors")
            ip = float(ip_scale)
            if not math.isfinite(ip):
                raise ValueError(f"ip_scale: non-finite value {ip_scale}")
        else:
            ip = proc_scale
        # the schedule, exactly as B200Sampler.generate walks it (fp64 on the host)
        s = self.scheduler
        s.set_timesteps(N)
        ts = s.timesteps
        if init_latents is not None:
            n_run = min(int(N * strength), N)
            if n_run < 1:
                raise ValueError(f"strength {strength} leaves no denoising step of {N}")
            ts = ts[max(N - n_run, 0):]
        ts_list = ts.tolist()
        coef = []
        for i, t in enumerate(ts_list):
            c_x, c_e = s.coefficients(t)
            s_next = s.input_scale(ts_list[i + 1]) if self.euler and i + 1 < len(ts_list) else 1.0
            coef.append((g, c_x, c_e, s_next))
        start = s.add_noise_coefficients(ts_list[0]) if init_latents is not None else None
        req = dict(rid=self._next_rid, noise=noise, ctx=ctx, added=added_pair, init=init_latents, ts=[float(t) for t in ts_list],
                   coef=coef, ip=ip, start=start, sigma0=s.init_noise_sigma, s_in0=s.input_scale(ts_list[0]) if self.euler else None)
        self._next_rid += 1
        self._queue.append(req)
        return req["rid"]

    def pending(self):
        """requests queued or in a slot"""
        return len(self._queue) + sum(r is not None for r in self._slots)

    @torch.no_grad()
    def step(self):
        """One step boundary: admit queued requests into free slots (FIFO), replay the step once, and return
        [(rid, final latents (1, 4, H, W) fp32 on the device)] of the requests whose last step this was, in admission order."""
        if not self.pending():
            return []
        self._check_unet()
        self._reap_staging()
        for s in range(self.S):
            if self._slots[s] is None and self._queue:
                self._admit(s, self._queue.popleft())
        active = [s for s in range(self.S) if self._slots[s] is not None]
        if not active:
            return []
        self._replay()
        self.executed_row_steps += self.S
        self.useful_row_steps += len(active)
        done = []
        b = self._buf
        for s in active:
            slot = self._slots[s]
            slot["k"] += 1
            if slot["k"] == slot["n"]:
                out = torch.empty((1, 4) + self.hw, device=b["x"].device, dtype=torch.float32)
                out.copy_(b["x"][s:s + 1])
                done.append((slot["rid"], out))
                self._slots[s] = None
        return sorted(done, key=lambda d: d[0])

    @torch.no_grad()
    def drain(self):
        """step until the queue and the slots are empty -> {rid: final latents}"""
        out = {}
        while self.pending():
            out.update(self.step())
        return out

    # ------------------------------------------------------------------ device state
    def _unet_key(self):
        return (self.unet._proc_version, id(self.unet.prepare()))

    def _check_unet(self):
        if self._buf is not None and self._buf["key"] != self._unet_key():
            if any(r is not None for r in self._slots):
                raise RuntimeError("the UNet's attention processors or weights changed while requests are in flight")
            self._buf = None                                   # nothing in flight: rebuild (and re-capture) for the new UNet
        if self._buf is None:
            self._build()

    def _build(self):
        unet = self.unet
        P = unet.prepare()
        dev = unet.device
        S, R = self.S, self.max_steps + 1
        sum_c = P["temb_slices"][-1][1]
        f32 = dict(device=dev, dtype=torch.float32)
        coef_tab = torch.tensor(_IDENTITY, **f32).repeat(S, R, 1)
        wkv = P["wkv_text"].shape[0]
        # zeros everywhere: an idle slot's rows must hold finite data (0 * NaN is not 0)
        b = dict(key=self._unet_key(), blocks=list(P["temb_slices"]),
                 x=torch.zeros((S, 4) + self.hw, **f32),
                 xin=torch.zeros((S, 4) + self.hw, **f32) if self.euler else None,
                 rb=torch.zeros(2 * S * sum_c, **f32),
                 coef=coef_tab[:, 0].t().contiguous(),                                  # [4, S]: g, c_x, c_e, s_in
                 tables=torch.zeros(S, R, 2 * sum_c, **f32),
                 coef_tables=coef_tab,
                 step=torch.full((S,), R - 1, device=dev, dtype=torch.int32),
                 kv_t=torch.zeros(2 * S * self.n_text, wkv, device=dev, dtype=torch.bfloat16),
                 kv_i=torch.zeros(2 * S * self.n_ip, P["wkv_ip"].shape[0], device=dev, dtype=torch.bfloat16) if self.n_ip else None,
                 ips=torch.zeros(2 * S, **f32) if self.n_ip else None,
                 graph=None, eps=None)
        self._buf = b

    def _body(self):
        b, S = self._buf, self.S
        ops.rowbias_gather(b["tables"], b["coef_tables"], b["step"], b["blocks"], b["rb"], b["coef"])
        kv = (b["kv_t"], b["kv_i"], self.n_text, self.n_ip)
        b["eps"] = self.unet.forward_core(b["xin"] if self.euler else b["x"], b["rb"], kv, 2 * S, out_dtype=torch.float32,
                                          ip_scales=b["ips"])
        c = b["coef"]
        ops.cfg_step_coef_rows(b["eps"], b["x"], c[0], c[1], c[2], s_in=c[3] if self.euler else None, x_out=b["x"],
                               x_in_next=b["xin"])

    def _replay(self):
        b = self._buf
        if not self.use_cuda_graph:
            self._body()
            return
        if b["graph"] is None:
            kv = (b["kv_t"], b["kv_i"], self.n_text, self.n_ip)
            st = torch.cuda.Stream()
            st.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(st):      # warm-up outside capture (first-use function attributes, workspaces); no state changes
                self.unet.forward_core(b["xin"] if self.euler else b["x"], b["rb"], kv, 2 * self.S, out_dtype=torch.float32,
                                       ip_scales=b["ips"])
            torch.cuda.current_stream().wait_stream(st)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._body()
            b["graph"] = g
            self.captures += 1
        b["graph"].replay()

    # ------------------------------------------------------------------ admission (enqueued on the stream, no synchronisation)
    def _stage(self, host, dtype):
        """a host tensor on the engine's device: through a pinned buffer kept alive until its copy has run"""
        dev = self._buf["x"].device
        if host.device == dev:
            return host.to(dtype)
        if dev.type != "cuda":
            return host.to(dev, dtype)
        pinned = torch.empty(host.shape, dtype=dtype, pin_memory=True)
        pinned.copy_(host)
        out = torch.empty(host.shape, dtype=dtype, device=dev)
        out.copy_(pinned, non_blocking=True)
        self._keep(pinned)
        return out

    def _keep(self, *tensors):
        ev = torch.cuda.Event()
        ev.record()
        self._staging.append((ev, tensors))

    def _reap_staging(self):
        while self._staging and self._staging[0][0].query():
            self._staging.popleft()

    def _admit(self, s, req):
        unet, b, S = self.unet, self._buf, self.S
        nt, ni = self.n_text, self.n_ip
        n = len(req["ts"])
        start = self.max_steps - n                       # the request's rows end right before the sentinel row
        # host values of the request in one pinned block: timesteps, coefficient rows, IP scale
        vals = torch.tensor(req["ts"] + [v for row in req["coef"] for v in row] + [req["ip"]], dtype=torch.float64)
        host = self._stage(vals, torch.float32)
        ts, coef, ip = host[:n], host[n:5 * n].view(n, 4), host[5 * n:]
        b["step"][s:s + 1].copy_(self._stage(torch.tensor([start], dtype=torch.int32), torch.int32))
        b["coef_tables"][s, start:self.max_steps].copy_(coef)
        if b["ips"] is not None:
            b["ips"][s:s + 1].copy_(ip)
            b["ips"][S + s:S + s + 1].copy_(ip)
        ctx = self._stage(req["ctx"], req["ctx"].dtype)
        added = {k: self._stage(v, v.dtype) for k, v in req["added"].items()}
        kv_t, kv_i, _, _ = unet.context_kv(ctx)
        b["kv_t"][s * nt:(s + 1) * nt].copy_(kv_t[:nt])
        b["kv_t"][(S + s) * nt:(S + s + 1) * nt].copy_(kv_t[nt:])
        if ni:
            b["kv_i"][s * ni:(s + 1) * ni].copy_(kv_i[:ni])
            b["kv_i"][(S + s) * ni:(S + s + 1) * ni].copy_(kv_i[ni:])
        b["tables"][s, start:self.max_steps].copy_(unet.time_rowbias_table(ts, added, 2))
        # start latent, as B200Sampler.generate makes it
        x = b["x"][s:s + 1]
        noise = self._stage(req["noise"], torch.float32)
        if req["init"] is None:
            x.copy_(noise * req["sigma0"])
        else:
            c_x, c_e = req["start"]
            ops.axpby(noise.contiguous(), self._stage(req["init"], torch.float32).contiguous(), c_x, c_e, out=x)
        if self.euler:
            ops.axpby(x, x, req["s_in0"], 0.0, out=b["xin"][s:s + 1])
        self._slots[s] = dict(rid=req["rid"], n=n, k=0)
