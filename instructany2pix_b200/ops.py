"""Torch-tensor front end of the C ABI (``include/ia2p.h``).

Each function validates device/dtype/layout, allocates the output with torch (the library never allocates), passes raw
device pointers + the CURRENT torch stream to ``libia2p_sm100a.so`` and returns the output tensor.  No op here has a
PyTorch/CPU implementation: a missing library or a non-sm_100 device raises ``IA2PError``.
"""
from __future__ import annotations

import os

import torch

from . import _lib
from ._lib import ACT_GELU_NEW, ACT_NONE, ACT_SILU, BF16, F16, F32, IA2PError  # noqa: F401

_DT = {torch.float32: F32, torch.bfloat16: BF16, torch.float16: F16}


def _stream():
    return torch.cuda.current_stream().cuda_stream


# kernel-launch accounting (bench.py's "gpu_launches") and optional per-call CUDA-event profiling (bench.py's roofline):
# PROFILE, when a list, receives (symbol, flops, start_event, end_event) for every C-ABI call made in eager mode.
LAUNCHES = 0
PROFILE = None
TAG_ALWAYS = False          # tools/timeline_step.py: build the shape tags without event profiling
# GroupNorm statistics from the producing GEMM / conv epilogue (False or IA2P_COLSTATS=0: separate statistics pass over x)
USE_COLSTATS = os.environ.get("IA2P_COLSTATS", "1") != "0"
_KERNELS_PER_CALL = {"ia2p_groupnorm_nhwc": 2, "ia2p_conv_up2x_nhwc_bf16": 4, "ia2p_polar_interpolate": 2}
_FLOPS = 0.0
_BYTES = 0.0                # algorithmic bytes of the call (operands read once + results written once), for bench.py's roofline
_TAG = ""


# ---- weight prefetch plan (ia2p_tc_prefetch_hint): a forward pass issues its tensor-core launches in a fixed order, so after one
# recorded pass every launch can tell the library which weight matrix the NEXT launch will stream; that kernel then pulls it into
# L2 early.  ``plan`` is a dict owned by the caller (B200UNet / B200VAE): {"seq": [(ptr, bytes), ...], "ready": bool}.
# Measured on B200 (c3 step, same box): 66.70 ms without, 66.99 ms with the hints -- the first-wave weight misses are not what the
# short GEMMs wait for -- so the plan is OFF unless IA2P_WEIGHT_PREFETCH=1.
USE_WEIGHT_PREFETCH = os.environ.get("IA2P_WEIGHT_PREFETCH", "0") == "1"
_PLAN = None
_PLAN_POS = 0


def plan_begin(plan):
    global _PLAN, _PLAN_POS
    _PLAN, _PLAN_POS = (plan if USE_WEIGHT_PREFETCH else None), 0
    if _PLAN is not None and not _PLAN.get("ready"):
        _PLAN["seq"] = []


def plan_end():
    global _PLAN
    if _PLAN is not None:
        if not _PLAN.get("ready"):
            _PLAN["ready"] = len(_PLAN["seq"]) > 1
        elif _PLAN_POS != len(_PLAN["seq"]):
            _PLAN["ready"] = False                      # the launch sequence changed (different processors / shapes): re-record
    _PLAN = None


def _plan_step(w):
    """called by every tensor-core op with its weight tensor, right before the launch"""
    global _PLAN_POS
    plan = _PLAN
    if plan is None:
        return
    cur = (w.data_ptr(), w.numel() * w.element_size())
    if not plan.get("ready"):
        plan["seq"].append(cur)
        return
    seq = plan["seq"]
    if _PLAN_POS >= len(seq) or seq[_PLAN_POS] != cur:
        plan["ready"] = False                           # not the recorded order: stop hinting, re-record on the next pass
        plan["seq"] = []
        return
    nxt = seq[(_PLAN_POS + 1) % len(seq)]
    _PLAN_POS += 1
    _lib.load().ia2p_tc_prefetch_hint(nxt[0], nxt[1])


def _run(fn, args, what):
    global LAUNCHES, _FLOPS, _TAG, _BYTES
    LAUNCHES += _KERNELS_PER_CALL.get(fn.__name__, 1)
    prof = PROFILE
    if prof is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        status = fn(*args)
        e1.record()
        prof.append((fn.__name__, _FLOPS, e0, e1, _TAG, _BYTES))
    else:
        status = fn(*args)
    _FLOPS = 0.0
    _BYTES = 0.0
    _TAG = ""
    if status != 0:
        _lib.check(status, what)


def _ptr(t):
    return 0 if t is None else t.data_ptr()


class pdl:
    """``with ops.pdl():`` -- the launches inside use programmatic dependent launch (ia2p_set_pdl); restores the previous mode."""

    def __init__(self, on=True):
        self.on, self.prev = on, -1

    def __enter__(self):
        self.prev = _lib.load().ia2p_set_pdl(1 if self.on else 0)
        return self

    def __exit__(self, *a):
        _lib.load().ia2p_set_pdl(self.prev)


def _need(t, dtype, name, ndim=None):
    if not t.is_cuda:
        raise IA2PError(f"{name}: expected a CUDA tensor (instructany2pix_b200 has no CPU path)")
    if t.dtype != dtype:
        raise IA2PError(f"{name}: expected {dtype}, got {t.dtype}")
    if ndim is not None and t.ndim != ndim:
        raise IA2PError(f"{name}: expected {ndim} dims, got {tuple(t.shape)}")
    return t


def _rows(t, name):
    """2-D view with unit inner stride -> (tensor, leading dimension)."""
    if t.ndim != 2 or t.stride(1) != 1:
        raise IA2PError(f"{name}: expected a 2-D tensor with unit inner stride, got shape {tuple(t.shape)} stride {t.stride()}")
    return t.stride(0) if t.shape[0] > 1 else max(t.stride(0), t.shape[1])


def require_cuda(t, what):
    if not t.is_cuda:
        raise IA2PError(f"{what}: expected a CUDA tensor; instructany2pix_b200 has no CPU path")


def _f32(t, name):
    return None if t is None else _need(t, torch.float32, name).contiguous()


def _row_scales(t, batch, name):
    """a per-request scale vector: contiguous fp32 [batch] on the CUDA device (its values are read when the kernel runs)"""
    _need(t, torch.float32, name, 1)
    if t.shape[0] != batch:
        raise ValueError(f"{name}: {t.shape[0]} values for a batch of {batch} rows")
    if not t.is_contiguous():
        raise IA2PError(f"{name}: expected a contiguous tensor")
    return t


# ------------------------------------------------------------------------------------------------ sampler epilogues
def cfg_ddim_step(eps2, x, g, c_x, c_e, x_out=None, x_in_next2=None):
    """x_out = c_x*x + c_e*(eps_u + g*(eps_c - eps_u)); eps2 = [uncond; cond] (custom_pipelines.py:348-357).
    ``g``: a float for the whole batch, or a contiguous fp32 CUDA tensor [batch] with one guidance scale per request."""
    lib = _lib.load()
    eps2, x = eps2.contiguous(), x.contiguous()
    batch = x.shape[0]
    n = x.numel() // batch
    assert eps2.numel() == 2 * x.numel()
    if x_out is None:
        x_out = torch.empty_like(x)
    xin = (_ptr(x_in_next2), _DT[x_in_next2.dtype] if x_in_next2 is not None else F32)
    if isinstance(g, torch.Tensor):
        g = _row_scales(g, batch, "cfg_ddim_step: g")
        _run(lib.ia2p_cfg_ddim_step_rows, (eps2.data_ptr(), _DT[eps2.dtype], x.data_ptr(), x_out.data_ptr(), _DT[x.dtype], *xin,
                                           batch, n, g.data_ptr(), float(c_x), float(c_e), _stream()), "cfg_ddim_step_rows")
        return x_out
    _run(lib.ia2p_cfg_ddim_step, (eps2.data_ptr(), _DT[eps2.dtype], x.data_ptr(), x_out.data_ptr(), _DT[x.dtype], *xin,
                                      batch, n, float(g), float(c_x), float(c_e), _stream()), "cfg_ddim_step")
    return x_out


def cfg_step_coef_rows(eps2, x, g, c_x, c_e, s_in=None, x_out=None, x_in_next=None):
    """``cfg_ddim_step`` with every coefficient per row: x_out[b] = c_x[b]*x[b] + c_e[b]*(eps_u + g[b]*(eps_c - eps_u)).
    ``g``, ``c_x``, ``c_e`` (and ``s_in``): contiguous fp32 CUDA tensors [batch], read when the kernel runs.  ``x_in_next``
    [batch, ...] (with ``s_in``) receives s_in[b] * x_out[b], the row's next UNet input (not duplicated)."""
    lib = _lib.load()
    eps2, x = eps2.contiguous(), x.contiguous()
    batch = x.shape[0]
    n = x.numel() // batch
    assert eps2.numel() == 2 * x.numel()
    if (x_in_next is None) != (s_in is None):
        raise ValueError("cfg_step_coef_rows: x_in_next and s_in go together")
    g, c_x, c_e = (_row_scales(t, batch, f"cfg_step_coef_rows: {k}") for k, t in (("g", g), ("c_x", c_x), ("c_e", c_e)))
    if s_in is not None:
        s_in = _row_scales(s_in, batch, "cfg_step_coef_rows: s_in")
        if x_in_next.shape != x.shape or not x_in_next.is_contiguous():
            raise IA2PError(f"cfg_step_coef_rows: x_in_next must be a contiguous {tuple(x.shape)} tensor")
    if x_out is None:
        x_out = torch.empty_like(x)
    _run(lib.ia2p_cfg_step_coef_rows, (eps2.data_ptr(), _DT[eps2.dtype], x.data_ptr(), x_out.data_ptr(), _DT[x.dtype],
                                       _ptr(x_in_next), _DT[x_in_next.dtype] if x_in_next is not None else F32, batch, n,
                                       g.data_ptr(), c_x.data_ptr(), c_e.data_ptr(), _ptr(s_in), _stream()), "cfg_step_coef_rows")
    return x_out


def rowbias_gather(tables, coef_tables, step, blocks, rowbias, coef):
    """The step's blocked rowbias of an S-slot CFG batch from per-slot tables, then step[s] += 1 up to the last (sentinel) row.
    tables fp32 [S, rows, 2 * sumC] (``time_rowbias_table(ts, pair, 2)`` rows), coef_tables fp32 [S, rows, ncoef], step int32 [S],
    blocks: the ResnetBlocks' (lo, hi) column ranges (``prepare()["temb_slices"]``); rowbias fp32 [2 * S * sumC], coef fp32
    [ncoef, S] are written."""
    import ctypes
    lib = _lib.load()
    S, rows, width = tables.shape
    ncoef = coef_tables.shape[-1]
    lo = [int(a) for a, _ in blocks] + [int(blocks[-1][1])]
    if width != 2 * lo[-1] or lo != sorted(lo) or lo[0] != 0 or any(int(a) != b for (a, _), b in zip(blocks[1:], (h for _, h in blocks))):
        raise IA2PError(f"rowbias_gather: blocks {blocks} do not tile a table row of {width} = 2 * sumC columns")
    for t, name, shape, dt in ((tables, "tables", (S, rows, width), torch.float32), (coef_tables, "coef_tables", (S, rows, ncoef), torch.float32),
                               (step, "step", (S,), torch.int32), (rowbias, "rowbias", (S * width,), torch.float32),
                               (coef, "coef", (ncoef, S), torch.float32)):
        _need(t, dt, f"rowbias_gather: {name}")
        if tuple(t.shape) != shape or not t.is_contiguous():
            raise IA2PError(f"rowbias_gather: {name} must be a contiguous {shape} tensor, got {tuple(t.shape)}")
    offs = (ctypes.c_int64 * len(lo))(*lo)
    _run(lib.ia2p_rowbias_gather, (tables.data_ptr(), coef_tables.data_ptr(), step.data_ptr(), rowbias.data_ptr(), coef.data_ptr(),
                                   S, rows, ctypes.addressof(offs), len(blocks), ncoef, _stream()), "rowbias_gather")
    return rowbias


def axpby(eps, x, c_x, c_e, out=None):
    """out = c_x*x + c_e*eps (inverse DDIM step, pnp_pipeline.py:73-85)."""
    lib = _lib.load()
    eps, x = eps.contiguous(), x.contiguous()
    if out is None:
        out = torch.empty_like(x)
    _run(lib.ia2p_axpby, (eps.data_ptr(), _DT[eps.dtype], x.data_ptr(), out.data_ptr(), _DT[x.dtype], x.numel(),
                              float(c_x), float(c_e), _stream()), "axpby")
    return out


def inpaint_blend(latents, orig, noise, mask, c_x, c_e, out=None):
    """out = (1 - mask) * (c_x * orig + c_e * noise) + mask * latents (inpainting loop tail); mask (B,1,H,W), noise may be None."""
    lib = _lib.load()
    latents, orig, mask = _f32(latents, "latents"), _f32(orig, "orig"), _f32(mask, "mask")
    noise = None if noise is None else _f32(noise, "noise")
    B, C, H, W = latents.shape
    assert orig.shape == latents.shape and mask.shape == (B, 1, H, W)
    if out is None:
        out = torch.empty_like(latents)
    _run(lib.ia2p_inpaint_blend, (latents.data_ptr(), orig.data_ptr(), _ptr(noise), mask.data_ptr(), out.data_ptr(), B, C, H * W,
                                      float(c_x), float(c_e), _stream()), "inpaint_blend")
    return out


def polar_interpolate(x, y, alpha, out=None):
    """``InstructAny2PixPipeline.polar_intrtpolate`` (pipeline.py:295-300): blend two latents and restore the blended norm;
    norms are taken over the whole tensor, fp32."""
    lib = _lib.load()
    x, y = _f32(x, "x").contiguous(), _f32(y, "y").contiguous()
    assert x.shape == y.shape
    if out is None:
        out = torch.empty_like(x)
    ws = torch.empty(int(lib.ia2p_polar_workspace_bytes()), device=x.device, dtype=torch.uint8)
    _run(lib.ia2p_polar_interpolate, (x.data_ptr(), y.data_ptr(), out.data_ptr(), x.numel(), float(alpha), ws.data_ptr(),
                                          _stream()), "polar_interpolate")
    return out


def prior_cfg_ddpm_step(x0_pair, x, noise, sqrt_a, sqrt_1ma, g, c_x0, c_x, sigma, out=None):
    lib = _lib.load()
    x0_pair, x = _f32(x0_pair, "x0_pair"), _f32(x, "x")
    noise = _f32(noise, "noise")
    n = x.numel()
    assert x0_pair.numel() == 2 * n
    if out is None:
        out = torch.empty_like(x)
    _run(lib.ia2p_prior_cfg_ddpm_step, (x0_pair.data_ptr(), x.data_ptr(), _ptr(noise), out.data_ptr(), n, float(sqrt_a),
                                            float(sqrt_1ma), float(g), float(c_x0), float(c_x), float(sigma), _stream()),
               "prior_cfg_ddpm_step")
    return out


def timestep_embedding(t, dim, flip_sin_to_cos=True, shift=0.0, dtype=torch.float32):
    lib = _lib.load()
    t = _f32(t.reshape(-1), "t")
    out = torch.empty(t.numel(), dim, device=t.device, dtype=dtype)
    _run(lib.ia2p_timestep_embedding, (t.data_ptr(), t.numel(), dim, int(flip_sin_to_cos), float(shift), out.data_ptr(),
                                           _DT[dtype], _stream()), "timestep_embedding")
    return out


def to_bf16(x):
    """bf16 copy of a stream tensor (tensor-core operand); identity for bf16 input."""
    if x.dtype == torch.bfloat16:
        return x
    lib = _lib.load()
    require_cuda(x, "to_bf16")
    x = x.contiguous()
    y = torch.empty(x.shape, device=x.device, dtype=torch.bfloat16)
    _run(lib.ia2p_cast_to_bf16, (x.data_ptr(), _DT[x.dtype], y.data_ptr(), x.numel(), _stream()), "cast_to_bf16")
    return y


def upsample2x(x):
    """nearest 2x upsample of an NHWC tensor (fp32|bf16) -> bf16."""
    lib = _lib.load()
    require_cuda(x, "upsample2x")
    assert x.ndim == 4
    x = x.contiguous()
    b, h, w, c = x.shape
    y = torch.empty(b, 2 * h, 2 * w, c, device=x.device, dtype=torch.bfloat16)
    _run(lib.ia2p_upsample2x_nhwc, (x.data_ptr(), _DT[x.dtype], y.data_ptr(), b, h, w, c, _stream()), "upsample2x")
    return y


# ------------------------------------------------------------------------------------------------ norms
_GN_WS = {}


def groupnorm(xa, xb, gamma, beta, groups, eps, silu, want_raw=False):
    """GroupNorm(+SiLU) over the channel concat [xa | xb] of NHWC tensors [B, ..., C] (fp32 or bf16) -> bf16.
    ``want_raw``: also return the un-normalised concat as bf16 (operand of the fused 1x1 shortcut conv)."""
    lib = _lib.load()
    require_cuda(xa, "groupnorm")
    if xa.dtype not in (torch.bfloat16, torch.float32):
        raise IA2PError(f"groupnorm: unsupported dtype {xa.dtype}")
    xa = xa.contiguous()
    b, ca = xa.shape[0], xa.shape[-1]
    hw = xa.numel() // (b * ca)
    cb = 0
    if xb is not None:
        xb = _need(xb, xa.dtype, "xb").contiguous()
        cb = xb.shape[-1]
        assert xb.numel() // (b * cb) == hw
    gamma, beta = _f32(gamma, "gamma"), _f32(beta, "beta")
    out = torch.empty(*xa.shape[:-1], ca + cb, device=xa.device, dtype=torch.bfloat16)
    raw = torch.empty_like(out) if want_raw else None
    key = (xa.device, torch.cuda.current_stream().cuda_stream)
    need = lib.ia2p_groupnorm_workspace_bytes(b, groups)
    ws = _GN_WS.get(key)
    if ws is None or ws.numel() < need:
        ws = torch.empty(max(need, 4096), device=xa.device, dtype=torch.uint8)
        _GN_WS[key] = ws
    # statistics straight from the producers' epilogues when every source carries them (attached by gemm / conv3x3 / conv_up2x)
    csa, csb = getattr(xa, "_ia2p_cs", None), (None if xb is None else getattr(xb, "_ia2p_cs", None))
    use_cs = USE_COLSTATS and csa is not None and (xb is None or csb is not None)
    if use_cs:
        use_cs = hw % (128 * csa[1]) == 0 and (csb is None or hw % (128 * csb[1]) == 0)
    if not use_cs:
        csa = csb = None
    _run(lib.ia2p_groupnorm_nhwc, (xa.data_ptr(), ca, _ptr(xb), cb, _DT[xa.dtype], gamma.data_ptr(), beta.data_ptr(),
                                       out.data_ptr(), _ptr(raw), b, hw, groups, float(eps), int(silu),
                                       0 if csa is None else csa[0].data_ptr(), 1 if csa is None else csa[1],
                                       0 if csb is None else csb[0].data_ptr(), 1 if csb is None else csb[1],
                                       ws.data_ptr(), _stream()), "groupnorm")
    return (out, raw) if want_raw else out


def layernorm(x, gamma, beta, eps, out_dtype=None):
    """LayerNorm over the last dim; (in,out) in {(bf16,bf16), (fp32,bf16), (fp32,fp32)}."""
    lib = _lib.load()
    if x.dtype not in (torch.bfloat16, torch.float32):
        raise IA2PError(f"layernorm: unsupported dtype {x.dtype}")
    require_cuda(x, "layernorm")
    out_dtype = out_dtype or x.dtype
    x = x.contiguous()
    cols = x.shape[-1]
    rows = x.numel() // cols
    gamma, beta = _f32(gamma, "gamma"), _f32(beta, "beta")
    out = torch.empty(x.shape, device=x.device, dtype=out_dtype)
    _run(lib.ia2p_layernorm, (x.data_ptr(), _DT[x.dtype], gamma.data_ptr(), beta.data_ptr(), out.data_ptr(),
                                  _DT[out_dtype], rows, cols, float(eps), _stream()), "layernorm")
    return out


def clip_embed(ids, tok, pos, want_ln=False):
    """CLIP token + position embedding: fp32 [n*T, C] = tok[ids] + pos[:T] (ids int64 [n, T], tok bf16 [V, C], pos fp32 [P, C]).
    ``want_ln``: also the bf16 copy and per-row (sum, sum of squares) [n*T, 1, 2] that ``gemm(ln=...)`` folds LayerNorm with.
    Ids on the host are range-checked here (then copied to the table's device); ids already on the device are not
    (that would need a sync): an id outside [0, V) yields a NaN row."""
    lib = _lib.load()
    _need(tok, torch.bfloat16, "tok", 2)
    assert tok.is_contiguous()
    pos = _need(pos, torch.float32, "pos", 2).contiguous()
    if ids.dtype != torch.int64 or ids.ndim != 2:
        raise IA2PError(f"clip_embed: ids must be int64 [n, T], got {ids.dtype} {tuple(ids.shape)}")
    V, C = tok.shape
    if not ids.is_cuda:
        if ids.numel() and (int(ids.min()) < 0 or int(ids.max()) >= V):
            raise IA2PError(f"clip_embed: token ids outside [0, {V})")
        ids = ids.to(tok.device)
    ids = ids.contiguous()
    n, T = ids.shape
    out = torch.empty(n * T, C, device=tok.device, dtype=torch.float32)
    out2 = torch.empty(n * T, C, device=tok.device, dtype=torch.bfloat16) if want_ln else None
    stats = torch.empty(n * T, 1, 2, device=tok.device, dtype=torch.float32) if want_ln else None
    _run(lib.ia2p_clip_embed, (ids.data_ptr(), n, T, tok.data_ptr(), V, pos.data_ptr(), pos.shape[0], C, out.data_ptr(), _ptr(out2),
                                   _ptr(stats), _stream()), "clip_embed")
    return (out, out2, stats) if want_ln else out


# ------------------------------------------------------------------------------------------------ tensor-core GEMM / conv
# split-K workspace of the tensor-core kernels: one per device (the hot path runs on ONE stream per process), registered with the
# library before every tc launch made through this module (a thread-local pointer on the library side; re-registering is ~ns)
# Measured on B200 (tools/small_m.py, small_m_timeline.py; M 512, N 1280, K 5120): the k-loop shrinks 25 -> 9 us with 4 splits, but
# the hand-over (+6 us), the fix-up reads (+8 us) and the now fully exposed 128 x 256 epilogue (+13 us) make the launch SLOWER
# (37 vs 29 us; c2 step 13.9 vs 13.4 ms) than one narrow tile per CTA.  Opt-in (IA2P_GEMM_SPLITK=1) AND only present in experiment
# builds of the library (ia2p_tc_features() & 1): the shipped kernel has the path compiled out (its branches cost c2 7 %).
USE_SPLITK = os.environ.get("IA2P_GEMM_SPLITK", "0") == "1"
_TC_WS = {}


def _ensure_tc_workspace(device):
    if not USE_SPLITK:
        return
    lib = _lib.load()
    key = torch.device(device).index if torch.device(device).index is not None else torch.cuda.current_device()
    ws = _TC_WS.get(key)
    if ws is None:
        if torch.cuda.is_current_stream_capturing():
            return                                     # never allocate inside a graph capture: this call runs without split-K
        ws = torch.zeros(int(lib.ia2p_tc_workspace_bytes()), device=device, dtype=torch.uint8)
        _TC_WS[key] = ws
    lib.ia2p_set_tc_workspace(ws.data_ptr(), ws.numel())


def _colstats_buffer(tiles, n, device):
    """[row tiles][n][2] fp32 for the per-tile column sums a producer epilogue emits (consumed by groupnorm); None if tiles == 0"""
    return torch.empty(tiles, n, 2, device=device, dtype=torch.float32) if tiles > 0 else None


_ACT_EPI = {None: _lib.EPI_NONE, "gelu": _lib.EPI_GELU, "quick_gelu": _lib.EPI_QUICK_GELU}


def gemm(a, w, bias=None, a2=None, rowbias=None, rows_per_batch=0, residual=None, geglu=False, out=None,
         out_dtype=torch.bfloat16, want_ln=False, ln=None, want_colstats=False, act=None):
    """out = epilogue([a | a2] @ w^T).  a: [M,K1] bf16 (row-strided view allowed), w: [N,K1+K2] bf16 contiguous;
    residual bf16|fp32, out bf16|fp32 (fp32 = residual-stream tensors).
    ``act``: None, ``"gelu"`` (exact erf) or ``"quick_gelu"`` applied after the LN correction and bias (bf16 output only).

    LayerNorm folding: ``want_ln=True`` (producer) returns ``(out, out_bf16, stats)`` -- a bf16 copy of the output rows and
    the per-row partial sums; ``ln=(stats, c1, eps)`` (consumer) finishes LayerNorm in the epilogue:
    ``rstd * (a @ w^T - mean * c1) + bias`` with ``w`` pre-scaled by gamma and ``bias`` already holding ``W @ beta``."""
    lib = _lib.load()
    _need(a, torch.bfloat16, "a", 2)
    _need(w, torch.bfloat16, "w", 2)
    if act not in _ACT_EPI:
        raise IA2PError(f"gemm: unsupported activation {act!r} (None, 'gelu', 'quick_gelu')")
    _ensure_tc_workspace(a.device)
    assert w.is_contiguous()
    M, K1 = a.shape
    N = w.shape[0]
    lda = _rows(a, "a")
    K2, lda2 = 0, 0
    if a2 is not None:
        _need(a2, torch.bfloat16, "a2", 2)
        assert a2.shape[0] == M
        K2, lda2 = a2.shape[1], _rows(a2, "a2")
    assert w.shape[1] == K1 + K2, (w.shape, K1, K2)
    n_out = N // 2 if geglu else N
    if out is None:
        out = torch.empty(M, n_out, device=a.device, dtype=out_dtype)
    else:
        require_cuda(out, "gemm(out)")
        assert out.shape == (M, n_out) and out.dtype in (torch.bfloat16, torch.float32)
    ldo = _rows(out, "out")
    ldr, res_dt = 0, BF16
    if residual is not None:
        require_cuda(residual, "gemm(residual)")
        assert residual.shape == (M, n_out) and residual.dtype in (torch.bfloat16, torch.float32)
        ldr, res_dt = _rows(residual, "residual"), _DT[residual.dtype]
    bias, rowbias = _f32(bias, "bias"), _f32(rowbias, "rowbias")
    out2 = stats = None
    if want_ln:
        assert not geglu
        out2 = torch.empty(M, N, device=a.device, dtype=torch.bfloat16)
        stats = torch.empty(M, int(lib.ia2p_gemm_ln_parts(M, N, K1 + K2)), 2, device=a.device, dtype=torch.float32)
    cs = _colstats_buffer((M + 127) // 128, N, a.device) if (want_colstats and USE_COLSTATS and out.dtype == torch.float32 and not geglu) else None
    ln_stats = ln_c1 = None
    ln_parts, ln_eps = 0, 0.0
    if ln is not None:
        ln_stats, ln_c1, ln_eps = ln
        ln_stats, ln_c1 = _f32(ln_stats, "ln_stats"), _f32(ln_c1, "ln_c1")
        assert ln_stats.shape[0] == M and ln_c1.numel() == N
        ln_parts = ln_stats.shape[1]
    global _FLOPS, _TAG, _BYTES
    _FLOPS = 2.0 * M * N * (K1 + K2)
    _BYTES = (2.0 * M * (K1 + K2) + 2.0 * N * (K1 + K2) + M * n_out * out.element_size()
              + (M * n_out * residual.element_size() if residual is not None else 0) + (M * N * 2 + M * 8 * 4 if want_ln else 0))
    if PROFILE is not None or TAG_ALWAYS:
        _TAG = (f"gemm M{M} N{N} K{K1 + K2}{' geglu' if geglu else ''}{' res' + str(residual.dtype)[6:] if residual is not None else ''}"
                f" out{str(out.dtype)[6:]}{' +ln_stats' if want_ln else ''}{' ln_fold' if ln is not None else ''}{' ' + act if act else ''}")
    _plan_step(w)
    _run(lib.ia2p_gemm_ln_bf16, (a.data_ptr(), lda, K1, _ptr(a2), lda2, K2, w.data_ptr(), out.data_ptr(), ldo, M, N,
                                  _ptr(bias), _ptr(rowbias), int(rows_per_batch), _ptr(residual), ldr, res_dt,
                                  _DT[out.dtype], _lib.EPI_GEGLU if geglu else _ACT_EPI[act],
                                  _ptr(out2), N, _ptr(stats), _ptr(cs), _ptr(ln_stats), ln_parts, _ptr(ln_c1), float(ln_eps),
                                  _stream()), "gemm_bf16")
    if cs is not None:
        out._ia2p_cs = (cs, 1)
    if want_ln:
        return out, out2, stats
    return out


def conv3x3(x, w, cout, stride=1, sc_a=None, sc_b=None, bias=None, rowbias=None, residual=None, out_dtype=torch.bfloat16,
            want_colstats=False):
    """3x3 pad-1 conv on NHWC bf16; w: [cout, 9*Cin + Csc] bf16, K order (ky,kx,cin) then shortcut channels;
    residual bf16|fp32, out bf16|fp32."""
    lib = _lib.load()
    _need(x, torch.bfloat16, "x", 4)
    _need(w, torch.bfloat16, "w", 2)
    _ensure_tc_workspace(x.device)
    x = x.contiguous()
    assert w.is_contiguous()
    B, H, W, Cin = x.shape
    ca = cb = 0
    if sc_a is not None:
        sc_a = _need(sc_a, torch.bfloat16, "sc_a", 4).contiguous()
        ca = sc_a.shape[-1]
    if sc_b is not None:
        sc_b = _need(sc_b, torch.bfloat16, "sc_b", 4).contiguous()
        cb = sc_b.shape[-1]
    assert w.shape == (cout, 9 * Cin + ca + cb), (tuple(w.shape), cout, Cin, ca, cb)
    Ho, Wo = H // stride, W // stride
    out = torch.empty(B, Ho, Wo, cout, device=x.device, dtype=out_dtype)
    res_dt = BF16
    if residual is not None:
        require_cuda(residual, "conv3x3(residual)")
        residual = residual.contiguous()
        assert residual.shape == out.shape and residual.dtype in (torch.bfloat16, torch.float32)
        res_dt = _DT[residual.dtype]
    bias, rowbias = _f32(bias, "bias"), _f32(rowbias, "rowbias")
    global _FLOPS, _TAG, _BYTES
    _FLOPS = 2.0 * B * Ho * Wo * cout * w.shape[1]
    _BYTES = (2.0 * B * H * W * (Cin + ca + cb) + 2.0 * w.numel() + B * Ho * Wo * cout * out.element_size()
              + (residual.numel() * residual.element_size() if residual is not None else 0))
    if PROFILE is not None or TAG_ALWAYS:
        _TAG = f"conv {H}x{W} C{Cin}->{cout} K{w.shape[1]} s{stride}{' res' if residual is not None else ''} out{str(out_dtype)[6:]}"
    cs = None
    if want_colstats and USE_COLSTATS and out_dtype == torch.float32:
        cs = _colstats_buffer(int(lib.ia2p_conv_colstats_tiles(B, Ho, Wo)), cout, x.device)
    _plan_step(w)
    _run(lib.ia2p_conv3x3_nhwc_bf16, (x.data_ptr(), B, H, W, Cin, stride, w.data_ptr(), _ptr(sc_a), ca, _ptr(sc_b), cb,
                                          out.data_ptr(), _DT[out_dtype], cout, _ptr(bias), _ptr(rowbias), _ptr(residual),
                                          res_dt, _ptr(cs), _stream()), "conv3x3")
    if cs is not None:
        out._ia2p_cs = (cs, 1)
    return out


def conv_up2x(x, w4, cout, bias=None, want_colstats=False):
    """nearest-2x upsample + 3x3 conv as four parity 2x2 convs over the low-res map; x NHWC bf16, w4 [4, cout, 4*Cin] bf16
    (packing.pack_conv3x3_up2x) -> [B, 2H, 2W, cout] fp32."""
    lib = _lib.load()
    _need(x, torch.bfloat16, "x", 4)
    _need(w4, torch.bfloat16, "w4", 3)
    _ensure_tc_workspace(x.device)
    x = x.contiguous()
    B, H, W, Cin = x.shape
    assert w4.is_contiguous() and w4.shape == (4, cout, 4 * Cin)
    out = torch.empty(B, 2 * H, 2 * W, cout, device=x.device, dtype=torch.float32)
    bias = _f32(bias, "bias")
    global _FLOPS, _TAG, _BYTES
    _FLOPS = 2.0 * B * 4 * H * W * cout * 9 * Cin                  # ALGORITHMIC flops of the 3x3 conv on the upsampled map
    _BYTES = 2.0 * B * H * W * Cin + 2.0 * w4.numel() + 4.0 * out.numel()
    if PROFILE is not None or TAG_ALWAYS:
        _TAG = f"conv_up2x {H}x{W}->{2 * H}x{2 * W} C{Cin}->{cout} (4 x K{4 * Cin})"
    cs = _colstats_buffer(4 * int(lib.ia2p_conv_colstats_tiles(B, H, W)), cout, x.device) if (want_colstats and USE_COLSTATS) else None
    _plan_step(w4)
    _run(lib.ia2p_conv_up2x_nhwc_bf16, (x.data_ptr(), B, H, W, Cin, w4.data_ptr(), out.data_ptr(), cout, _ptr(bias), _ptr(cs),
                                            _stream()), "conv_up2x")
    if cs is not None:
        out._ia2p_cs = (cs, 4)                 # one segment of row tiles per output parity
    return out


def conv3x3_down_padend(x, w, cout, bias=None, out_dtype=torch.bfloat16):
    """stride-2 3x3 conv padded at the bottom/right only (VAE encoder Downsample2D); x NHWC bf16, w [cout, 9*Cin] bf16."""
    lib = _lib.load()
    _need(x, torch.bfloat16, "x", 4)
    _need(w, torch.bfloat16, "w", 2)
    _ensure_tc_workspace(x.device)
    x = x.contiguous()
    B, H, W, Cin = x.shape
    assert w.is_contiguous() and w.shape == (cout, 9 * Cin) and H % 2 == 0 and W % 2 == 0
    out = torch.empty(B, H // 2, W // 2, cout, device=x.device, dtype=out_dtype)
    bias = _f32(bias, "bias")
    global _FLOPS
    _FLOPS = 2.0 * B * (H // 2) * (W // 2) * cout * w.shape[1]
    _plan_step(w)
    _run(lib.ia2p_conv3x3_s2_padend_nhwc_bf16, (x.data_ptr(), B, H, W, Cin, w.data_ptr(), out.data_ptr(), _DT[out_dtype], cout,
                                                    _ptr(bias), _stream()), "conv3x3_down_padend")
    return out


def gaussian_sample(moments, noise, scale=1.0):
    """scale * (mean + exp(0.5 clamp(logvar)) * noise) from moments (B, 2C, H, W) fp32; noise None -> scale * mean."""
    lib = _lib.load()
    moments = _f32(moments, "moments").contiguous()
    B, C2, H, W = moments.shape
    noise = None if noise is None else _f32(noise, "noise").contiguous()
    out = torch.empty(B, C2 // 2, H, W, device=moments.device, dtype=torch.float32)
    _run(lib.ia2p_gaussian_sample, (moments.data_ptr(), _ptr(noise), out.data_ptr(), B, C2 // 2, H * W, float(scale), _stream()),
         "gaussian_sample")
    return out


def conv_in(x_nchw, w, bias, out_batch=None, out_dtype=torch.bfloat16):
    """conv_in from NCHW latents to NHWC (bf16|fp32); batch read modulo x.shape[0] (CFG duplication)."""
    lib = _lib.load()
    if not x_nchw.is_cuda:
        raise IA2PError("conv_in: expected a CUDA tensor")
    x_nchw = x_nchw.contiguous()
    in_b, cin, H, W = x_nchw.shape
    B = out_batch or in_b
    w, bias = _f32(w, "w"), _f32(bias, "bias")
    cout = w.shape[0]
    out = torch.empty(B, H, W, cout, device=x_nchw.device, dtype=out_dtype)
    _run(lib.ia2p_conv_in_nchw, (x_nchw.data_ptr(), _DT[x_nchw.dtype], in_b, B, H, W, cin, w.data_ptr(), _ptr(bias),
                                     out.data_ptr(), _DT[out_dtype], cout, _stream()), "conv_in")
    return out


def conv_out(x, w, bias, out_dtype=torch.float32):
    """conv_out from NHWC bf16 to NCHW; w: fp32 [cout, 3, 3, Cin]."""
    lib = _lib.load()
    _need(x, torch.bfloat16, "x", 4)
    x = x.contiguous()
    B, H, W, Cin = x.shape
    w, bias = _f32(w, "w"), _f32(bias, "bias")
    cout = w.shape[0]
    out = torch.empty(B, cout, H, W, device=x.device, dtype=out_dtype)
    _run(lib.ia2p_conv_out_nhwc, (x.data_ptr(), B, H, W, Cin, w.data_ptr(), _ptr(bias), out.data_ptr(), _DT[out_dtype],
                                      cout, _stream()), "conv_out")
    return out


def conv_out_tc(x, w32, b32, cout):
    """conv_out on the tensor cores: 3x3 conv with the ``cout`` (<= 8) output channels zero-padded to 32 (``w32`` [32, 9*Cin]
    bf16, ``b32`` [32] fp32; packing.pack_conv_out) followed by the NHWC-prefix -> NCHW copy.  x NHWC bf16 -> [B, cout, H, W] fp32."""
    lib = _lib.load()
    B, H, W, _ = x.shape
    y = conv3x3(x, w32, 32, bias=b32, out_dtype=torch.float32)
    out = torch.empty(B, cout, H, W, device=x.device, dtype=torch.float32)
    _run(lib.ia2p_nhwc_prefix_to_nchw, (y.data_ptr(), 32, out.data_ptr(), B, H * W, cout, _stream()), "nhwc_prefix_to_nchw")
    return out


def conv_in_u8(x, w, bias, out_dtype=torch.bfloat16):
    """conv_in straight from an 8-bit image: x uint8 [B, H, W, Cin] is read as ``2 * (q / 255) - 1`` in fp32 (diffusers'
    ``VaeImageProcessor.preprocess`` of a PIL image) -> NHWC (bf16|fp32); w fp32 [Cout, Cin, 3, 3]."""
    lib = _lib.load()
    _need(x, torch.uint8, "x", 4)
    x = x.contiguous()
    B, H, W, cin = x.shape
    w, bias = _f32(w, "w"), _f32(bias, "bias")
    if w.shape[1] != cin:
        raise IA2PError(f"conv_in_u8: image has {cin} channels, the weights expect {w.shape[1]}")
    cout = w.shape[0]
    out = torch.empty(B, H, W, cout, device=x.device, dtype=out_dtype)
    global _BYTES
    _BYTES = x.numel() + out.numel() * out.element_size() + 4.0 * w.numel()
    _run(lib.ia2p_conv_in_u8_nhwc, (x.data_ptr(), B, H, W, cin, w.data_ptr(), _ptr(bias), out.data_ptr(), _DT[out_dtype], cout,
                                        _stream()), "conv_in_u8")
    return out


def image_u8(y):
    """The first three channels of an NHWC fp32 tensor y [B, H, W, C >= 4] (C % 4 == 0) as an 8-bit image uint8 [B, H, W, 3]:
    ``round_half_even(clamp(v / 2 + 0.5, 0, 1) * 255)``, bit for bit diffusers' ``postprocess(output_type="pil")``; NaN -> 0."""
    lib = _lib.load()
    _need(y, torch.float32, "y", 4)
    y = y.contiguous()
    B, H, W, ld = y.shape
    out = torch.empty(B, H, W, 3, device=y.device, dtype=torch.uint8)
    global _BYTES
    _BYTES = 16.0 * B * H * W + out.numel()
    _run(lib.ia2p_nhwc_prefix_to_u8_image, (y.data_ptr(), ld, out.data_ptr(), B, H * W, _stream()), "image_u8")
    return out


def conv_out_u8(x, w32, b32):
    """``conv_out_tc`` of the VAE decoder with its image written as uint8 [B, H, W, 3] (``image_u8``) instead of fp32 NCHW."""
    return image_u8(conv3x3(x, w32, 32, bias=b32, out_dtype=torch.float32))


def conv1x1_nchw_small(x, w, bias, scale=1.0):
    """1x1 conv over <= 8 channels, NCHW fp32 -> NCHW fp32: scale * (w x) + bias (VAE post_quant_conv / quant_conv)."""
    lib = _lib.load()
    x = _f32(x, "x").contiguous()
    B, cin, H, W = x.shape
    w, bias = _f32(w, "w").reshape(-1, cin).contiguous(), _f32(bias, "bias")
    cout = w.shape[0]
    out = torch.empty(B, cout, H, W, device=x.device, dtype=torch.float32)
    _run(lib.ia2p_conv1x1_nchw_small, (x.data_ptr(), w.data_ptr(), _ptr(bias), out.data_ptr(), B, cin, cout, H * W, float(scale),
                                           _stream()), "conv1x1_nchw_small")
    return out


# ------------------------------------------------------------------------------------------------ attention
def softmax_rows(scores, scale, out=None):
    """softmax(scale * scores) over the last dim of an fp32 matrix -> bf16."""
    lib = _lib.load()
    _need(scores, torch.float32, "scores", 2)
    rows, cols = scores.shape
    assert scores.stride(1) == 1
    if out is None:
        out = torch.empty(rows, cols, device=scores.device, dtype=torch.bfloat16)
    _run(lib.ia2p_softmax_rows_f32_bf16, (scores.data_ptr(), scores.stride(0), out.data_ptr(), out.stride(0), rows, cols,
                                              float(scale), _stream()), "softmax_rows")
    return out


def flash_self_attn(qkv, batch, n_tokens, heads, out=None):
    """qkv: [batch*n_tokens, 3*C] bf16 (q | k | v); returns [batch*n_tokens, C]."""
    lib = _lib.load()
    _need(qkv, torch.bfloat16, "qkv", 2)
    C = heads * 64
    assert qkv.shape == (batch * n_tokens, 3 * C) and qkv.stride(1) == 1
    ld = qkv.stride(0)
    if out is None:
        out = torch.empty(batch * n_tokens, C, device=qkv.device, dtype=torch.bfloat16)
    es = qkv.element_size()
    global _FLOPS
    _FLOPS = 4.0 * batch * heads * n_tokens * n_tokens * 64
    _run(lib.ia2p_flash_self_attn_bf16, (qkv.data_ptr(), qkv.data_ptr() + C * es, qkv.data_ptr() + 2 * C * es, ld,
                                             out.data_ptr(), out.stride(0), batch, n_tokens, heads, 0.125, _stream()),
               "flash_self_attn")
    return out


def causal_self_attn(qkv, n, T, heads, out=None):
    """Causal self-attention of n sequences of T <= 128 tokens (CLIP text towers).  qkv: [n*T, 3*C] bf16 (q | k | v);
    returns [n*T, C] bf16."""
    lib = _lib.load()
    _need(qkv, torch.bfloat16, "qkv", 2)
    C = heads * 64
    assert qkv.shape == (n * T, 3 * C) and qkv.stride(1) == 1
    if out is None:
        out = torch.empty(n * T, C, device=qkv.device, dtype=torch.bfloat16)
    es = qkv.element_size()
    global _FLOPS
    _FLOPS = 2.0 * n * heads * T * (T + 1) * 64               # causal half of QK^T and PV
    _run(lib.ia2p_causal_self_attn_bf16, (qkv.data_ptr(), qkv.data_ptr() + C * es, qkv.data_ptr() + 2 * C * es, qkv.stride(0),
                                              out.data_ptr(), out.stride(0), n, T, heads, 0.125, _stream()), "causal_self_attn")
    return out


def cross_attn(q, kv_text, n_text, kv_ip, n_ip, ip_scale, batch, n_q, heads, out=None):
    """Decoupled cross-attention.  q: [batch*n_q, C]; kv_text: [batch*n_text, 2C] (k | v); kv_ip: [batch*n_ip, 2C] | None.
    ``ip_scale``: a float for the whole batch, or a contiguous fp32 CUDA tensor [batch] with one IP scale per row."""
    lib = _lib.load()
    _need(q, torch.bfloat16, "q", 2)
    _need(kv_text, torch.bfloat16, "kv_text", 2)
    C = heads * 64
    assert q.shape == (batch * n_q, C) and kv_text.shape == (batch * n_text, 2 * C)
    es = 2
    if n_ip > 0:
        _need(kv_ip, torch.bfloat16, "kv_ip", 2)
        assert kv_ip.shape == (batch * n_ip, 2 * C)
        kip, vip, ldip = kv_ip.data_ptr(), kv_ip.data_ptr() + C * es, kv_ip.stride(0)
    else:
        kip, vip, ldip = 0, 0, 0
    if out is None:
        out = torch.empty(batch * n_q, C, device=q.device, dtype=torch.bfloat16)
    global _FLOPS
    _FLOPS = 4.0 * batch * heads * n_q * (n_text + n_ip) * 64
    if isinstance(ip_scale, torch.Tensor):
        fn, scale, what = lib.ia2p_decoupled_cross_attn_rows_bf16, _row_scales(ip_scale, batch, "cross_attn: ip_scale").data_ptr(), \
            "decoupled_cross_attn_rows"
    else:
        fn, scale, what = lib.ia2p_decoupled_cross_attn_bf16, float(ip_scale), "decoupled_cross_attn"
    _run(fn, (q.data_ptr(), q.stride(0), kv_text.data_ptr(), kv_text.data_ptr() + C * es, kv_text.stride(0), n_text, kip, vip, ldip,
              n_ip, scale, out.data_ptr(), out.stride(0), batch, n_q, heads, 0.125, _stream()), what)
    return out


# ------------------------------------------------------------------------------------------------ prior / embeddings
def gemm_smallm(a, w, bias=None, residual=None, act_in=ACT_NONE, act=ACT_NONE, out=None):
    """out[M,N] fp32 = act(act_in(a) @ w^T + bias) + residual; a fp32 [M,K], w bf16 [N,K]."""
    lib = _lib.load()
    _need(a, torch.float32, "a", 2)
    _need(w, torch.bfloat16, "w", 2)
    a = a.contiguous()
    assert w.is_contiguous() and w.shape[1] == a.shape[1]
    M, K = a.shape
    N = w.shape[0]
    bias = _f32(bias, "bias")
    if residual is not None:
        residual = _f32(residual, "residual")
        assert residual.shape == (M, N)
    if out is None:
        out = torch.empty(M, N, device=a.device, dtype=torch.float32)
    _run(lib.ia2p_gemm_smallm, (a.data_ptr(), K, w.data_ptr(), _ptr(bias), _ptr(residual), N, out.data_ptr(), N, M, N, K,
                                    act_in, act, _stream()), "gemm_smallm")
    return out


def causal_attn_small(qkv, batch, T, heads, out=None):
    lib = _lib.load()
    qkv = _f32(qkv, "qkv")
    E = heads * 64
    assert qkv.numel() == batch * T * 3 * E
    if out is None:
        out = torch.empty(batch, T, E, device=qkv.device, dtype=torch.float32)
    _run(lib.ia2p_causal_attn_small_f32, (qkv.data_ptr(), out.data_ptr(), batch, T, heads, _stream()), "causal_attn_small")
    return out


def prior_trunk_workspace(rows, device):
    """Zero-initialised workspace of ia2p_prior_trunk for `rows` = 2 * batch * T sequence rows (holds the grid-barrier state: allocate
    once, reuse for every call)."""
    n = _lib.load().ia2p_prior_trunk_workspace_bytes(rows)
    return torch.zeros((n + 255) // 256 * 256, dtype=torch.uint8, device=device)


def prior_trunk(seq, wpe, layers, lnf_g, lnf_b, heads, workspace, out=None, cache=None):
    """x0 = ln_f(GPT2(inputs_embeds=seq))[:, -1] in ONE persistent kernel.  seq [B2, T, E] fp32; layers: per layer the 12 tensors
    (wqkv, wo, wfc, wpr bf16 [out, in]; bqkv, bo, bfc, bpr, ln1 gamma, ln1 beta, ln2 gamma, ln2 beta fp32), see include/ia2p.h;
    workspace from prior_trunk_workspace; cache: a dict that keeps the ctypes pointer table between calls."""
    import ctypes
    lib = _lib.load()
    seq = _f32(seq, "seq")
    B2, T, E = seq.shape
    tab = None if cache is None else cache.get("table")
    if tab is None:
        flat = [t for L in layers for t in L]
        for i, t in enumerate(flat):
            _need(t, torch.bfloat16 if i % 12 < 4 else torch.float32, f"layers[{i // 12}][{i % 12}]")
            assert t.is_contiguous()
        tab = (ctypes.c_void_p * len(flat))(*[t.data_ptr() for t in flat])
        if cache is not None:
            cache["table"] = tab
    if out is None:
        out = torch.empty(B2, E, device=seq.device, dtype=torch.float32)
    _run(lib.ia2p_prior_trunk, (seq.data_ptr(), wpe.data_ptr(), tab, len(layers), lnf_g.data_ptr(), lnf_b.data_ptr(), B2, T, E, heads,
                                workspace.data_ptr(), workspace.numel(), out.data_ptr(), _stream()), "prior_trunk")
    return out
