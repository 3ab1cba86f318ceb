"""The CTA-pair tensor-core GEMM / implicit-GEMM conv (``tc_gemm_kernel<BN, 2, EPI>``, cta_group::2) against fp64 references.

The big UNet GEMMs and convs run on CTA pairs.  ``use_pair`` in csrc/gemm_tc.cu picks them for problems with at least two row
tiles, BLOCK_N != 64, at least 2 x SMs output tiles and at least 13 k-blocks (K >= 832); the other kernel tests stay below that.
Every case here

* predicts the launch (tile width, pair or not, epilogue variant, grid, tail split) from the device's SM count with the host
  rules of gemm_tc.cu mirrored in ``plan`` below, and asserts the tile width / CTA group / epilogue template arguments and the
  grid of the ``tc_gemm_kernel`` launches torch.profiler (CUPTI) saw;
* runs on poisoned allocations (tests/_poison.py): anything the kernel leaves unwritten stays NaN;
* compares every element with an fp64 evaluation of the same operation on the kernel's own bf16 operands (``check``);
* is bit-identical on a second call.

Per-element bound, bf16 operands and fp32 accumulation (products are exact in fp32, each of the K additions rounds by at most
2^-23 relative):  |out - ref| <= 2^-8 |ref| (bf16 output rounding; not for fp32 outputs) + K 2^-23 (|A| |W|^T) + 1e-6.
A dropped k-block, a misplaced tile or a missing bias / row bias / residual breaks it by far; a NaN breaks it always.
"""
import json
import math
import os
import re

import pytest
import torch
import torch.nn.functional as F

from tests._poison import is_poison, poisoned

DEV = "cuda"
gpu = pytest.mark.gpu

# ------------------------------------------------------------------------------------------------ launch model (gemm_tc.cu host rules)
# Process-wide switches of gemm_tc.cu (read once per process): the model below mirrors their defaults only.
_PROCESS_SWITCHES = ("IA2P_GEMM_CG", "IA2P_GEMM_EPI", "IA2P_GEMM_EPI3", "IA2P_GEMM_TAILSPLIT", "IA2P_GEMM_PAIR_MINKB",
                     "IA2P_GEMM_BN1280", "IA2P_GEMM_SPLITK", "IA2P_GEMM_MC")
MIN_TILES_WIDE = 120          # kMinTilesForWideBlock
PAIR_MIN_KB = 13              # use_pair: pairs from 13 k-blocks (K >= 832) on


def pick_block_n(N, geglu, m_tiles):
    """pick_block_n (shipped build: no split-K)"""
    e = os.environ.get("IA2P_GEMM_BN", "")
    if e.isdigit():
        v = int(e)
        if v in (64, 128, 160, 256) and N % v == 0 and (not geglu or v % 64 == 0):
            return v
    last = 0
    for c in (256, 160, 128, 64):
        if N % c or (geglu and c % 64):
            continue
        last = c
        if m_tiles * (N // c) >= MIN_TILES_WIDE:
            return c
    return last or 128


def plan(m_tiles, N, K, sms, *, geglu=False, out_f32=False, residual=None, extras=False):
    """What ia2p_gemm_ln_bf16 / conv3x3_impl launch: dict(bn, cg, epi, grid, split).  ``residual``: None | "bf16" | "f32";
    ``extras``: a bf16 copy, LN statistics or column statistics are requested."""
    bn = pick_block_n(N, geglu, m_tiles)
    n_tiles = -(-N // bn)
    num_kb = K // 64
    cg = 2 if (m_tiles >= 2 and bn != 64 and m_tiles * n_tiles >= 2 * sms and num_kb >= PAIR_MIN_KB) else 1
    if not out_f32 and residual is None and not extras:
        epi = 3                                           # tma_epilogue_bf16
    elif out_f32 and not geglu and residual == "f32" and num_kb <= 24:
        epi = 2                                           # tma_residual
    elif out_f32 and not geglu:
        epi = 1                                           # tma_epilogue
    else:
        epi = 0
    units = -(-m_tiles // cg) * n_tiles
    max_units = sms // cg
    rem = units % max_units
    can_split = bn % 64 == 0 and (not geglu or bn % 128 == 0) and N % bn == 0
    split = can_split and units > max_units and rem != 0 and 2 * rem <= max_units
    return dict(bn=bn, cg=cg, epi=epi, grid=min(units, max_units) * cg, split=split)


def conv_tile(B, Ho, Wo):
    """conv3x3_impl / conv_up2x tile of 128 output pixels: (TW, TH, TB, m_tiles)"""
    TW = 1
    while TW < 128 and Wo % (TW * 2) == 0:
        TW *= 2
    TH = 1
    while TW * TH < 128 and Ho % (TH * 2) == 0:
        TH *= 2
    TB = 128 // (TW * TH)
    return TW, TH, TB, (Wo // TW) * (Ho // TH) * -(-B // TB)


_KERNEL = re.compile(r"tc_gemm_kernel<(\d+), ?(\d+), ?(\d+)>")


def launched(fn, tmp_path):
    """run fn() under torch.profiler -> (its result, [(bn, cg, epi, grid_x) of every tc_gemm_kernel launch])"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    path = tmp_path / "trace.json"
    prof.export_chrome_trace(str(path))
    with open(path) as f:
        events = json.load(f)["traceEvents"]
    got = []
    for e in events:
        m = _KERNEL.search(e.get("name", "")) if e.get("cat") == "kernel" else None
        if m:
            got.append((*map(int, m.groups()), e["args"]["grid"][0]))
    return out, got


def expect(p, n=1):
    return [(p["bn"], p["cg"], p["epi"], p["grid"])] * n


# ------------------------------------------------------------------------------------------------ per-element comparison
def _where(shape, idx, bn):
    if len(shape) == 1:
        return f"row {idx} (128-row tile {idx // 128})"
    if len(shape) == 2:
        r, c = divmod(idx, shape[1])
        return f"row {r} col {c} (128-row tile {r // 128}, column tile {c // bn} of BLOCK_N {bn})"
    B, H, W, C = shape
    b, rest = divmod(idx, H * W * C)
    y, rest = divmod(rest, W * C)
    x, c = divmod(rest, C)
    TW, TH, TB, _ = conv_tile(B, H, W)
    tile = ((b // TB) * (H // TH) + y // TH) * (W // TW) + x // TW
    return f"pixel (b {b}, y {y}, x {x}) channel {c} (pixel tile {tile}, column tile {c // bn} of BLOCK_N {bn})"


def check(out, ref64, bound, bn=128, what="out"):
    """|out - ref64| <= bound elementwise (NaN fails); on failure name the worst element, its tile and the count out of bound.
    ``out`` is [rows, cols] (128-row tiles) or NHWC (128-pixel tiles of the conv kernels)."""
    assert out.shape == ref64.shape, (tuple(out.shape), tuple(ref64.shape))
    err = (out.double() - ref64).abs()
    bad = ~(err <= bound)
    n_bad = int(bad.sum())
    if n_bad:
        score = torch.where(bad, torch.nan_to_num(err / bound, nan=math.inf), torch.zeros_like(err)).flatten()
        i = int(score.argmax())
        raise AssertionError(
            f"{what}: {n_bad} of {out.numel()} elements out of bound; worst at {_where(tuple(out.shape), i, bn)}: "
            f"out {out.flatten()[i].item():.6g} ref {ref64.flatten()[i].item():.6g} bound {bound.flatten()[i].item():.3g}")


def gemm_bound(ref, mag, K, bf16_out):
    b = K * 2.0 ** -23 * mag + 1e-6
    return b + 2.0 ** -8 * ref.abs() if bf16_out else b


def rel(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / b.norm()).item()


def bits(t):
    return t.contiguous().view({2: torch.int16, 4: torch.int32}[t.element_size()])


def same_bits(a, b):
    return torch.equal(bits(a), bits(b))


def rnd(*shape, scale=1.0, dtype=torch.bfloat16, seed=0):
    g = torch.Generator(device=DEV)
    g.manual_seed(seed * 1000003 + hash(shape) % 1000003)
    return (torch.randn(*shape, generator=g, device=DEV) * scale).to(dtype)


def operands(M, N, K, seed=0):
    return rnd(M, K, seed=seed), rnd(N, K, scale=K ** -0.5, seed=seed + 1)


def ref_gemm(a, w):
    """fp64 a @ w^T and |a| @ |w|^T of the kernel's bf16 operands"""
    a64, w64 = a.double(), w.double()
    return a64 @ w64.t(), a64.abs() @ w64.abs().t()


# fp64 im2col of the implicit-GEMM convs: rows = output pixels (b, y, x), K order = the packed weights' (tap, channel) order.
def im2col(x, taps, pads, Ho, Wo, stride=1):
    """x NHWC; pads = (top, bottom, left, right); taps = [(ky, kx)] offsets into the padded map"""
    xp = F.pad(x.double(), (0, 0, pads[2], pads[3], pads[0], pads[1]))
    cols = [xp[:, ky:ky + stride * (Ho - 1) + 1:stride, kx:kx + stride * (Wo - 1) + 1:stride, :] for ky, kx in taps]
    return torch.cat(cols, -1).reshape(-1, len(taps) * x.shape[-1])


TAPS3 = [(ky, kx) for ky in range(3) for kx in range(3)]
TAPS2 = [(i, j) for i in range(2) for j in range(2)]


def conv3x3_cols(x, stride=1, pad_end=False):
    B, H, W, _ = x.shape
    pads = (0, 1, 0, 1) if pad_end else (1, 1, 1, 1)
    return im2col(x, TAPS3, pads, H // stride, W // stride, stride)


def up2x_cols(x, py, px):
    """rows of output parity (py, px) of the nearest-2x upsample + 3x3 conv: the 2x2 low-res neighbourhood, rows {y-1, y} for
    py = 0 and {y, y+1} for py = 1 (same for columns) -- the tap order of pack_conv3x3_up2x"""
    B, H, W, _ = x.shape
    return im2col(x, TAPS2, (1 - py, py, 1 - px, px), H, W)


def tile_rows(t, TW, TH, TB):
    """NHWC -> [m_tiles, 128, C] in the kernel's tile order (tiles (b, y, x)-major, rows (tb, th, tw) inside)"""
    B, H, W, C = t.shape
    return t.reshape(B // TB, TB, H // TH, TH, W // TW, TW, C).permute(0, 2, 4, 1, 3, 5, 6).reshape(-1, 128, C)


def check_colstats(cs, tiles, what):
    """cs [m_tiles, C, 2] (fp32 per-tile column sums) against fp64 sums of the kernel's own output rows [m_tiles, 128, C]"""
    t = tiles.double()
    s1, s2, mag = t.sum(1), (t * t).sum(1), (t * t).sum(1) + t.abs().sum(1)
    b = 128 * 2.0 ** -23 * mag + 1e-6
    check(cs[..., 0], s1, b, what=what + " column sums (row = 128-row tile)")
    check(cs[..., 1], s2, b, what=what + " column sums of squares (row = 128-row tile)")


@pytest.fixture
def sms():
    for k in _PROCESS_SWITCHES:
        if os.environ.get(k):
            pytest.skip(f"{k} is set: the launch model mirrors the default tile / pair / epilogue rules only")
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture
def poison():
    with poisoned():
        yield


# ------------------------------------------------------------------------------------------------ host-side tests (no GPU)
def test_poisoned_allocations_on_the_host():
    with poisoned():
        f32, bf, h, u8 = (torch.empty(3, 5, dtype=d) for d in (torch.float32, torch.bfloat16, torch.float16, torch.uint8))
        i64 = torch.empty(4, dtype=torch.int64)
        like = torch.empty_like(f32)
    assert all(torch.isnan(t).all() for t in (f32, bf, h, like)) and (u8 == 255).all() and is_poison(f32).all()
    assert i64.dtype == torch.int64                     # integer tensors other than uint8 are not touched
    assert torch.empty is not None and "poison" not in repr(torch.empty)


def test_launch_model_at_148_sms(monkeypatch):
    """the scheduling facts this sweep is built on, at the B200's 148 SMs (74 pairs)"""
    monkeypatch.delenv("IA2P_GEMM_BN", raising=False)
    p = plan(32, 2560, 1280, 148)                       # M 4096: 16 x 10 = 160 pair units, 160 mod 74 = 12 -> tail split
    assert (p["bn"], p["cg"], p["epi"], p["grid"], p["split"]) == (256, 2, 3, 148, True)
    assert not plan(40, 2560, 1280, 148)["split"]         # M 5120: 200 units, remainder 52 is too large to halve
    assert plan(32, 2560, 768, 148)["cg"] == 1            # 12 k-blocks: single-CTA kernel
    assert plan(32, 2560, 1280, 148, out_f32=True, residual="f32")["epi"] == 2
    assert plan(32, 2560, 2048, 148, out_f32=True, residual="f32")["epi"] == 1
    assert plan(32, 2560, 2048, 148, residual="bf16")["epi"] == 0
    assert plan(16, 10240, 1280, 148, geglu=True)["split"]  # SDXL FF GEGLU at M 2048: 320 units, remainder 24
    assert plan(74, 640, 1280, 148)["bn"] == 160 and not plan(74, 640, 1280, 148)["split"]


def test_conv_references_match_conv2d():
    """the im2col references equal fp64 F.conv2d (integer data: exact) for every tap layout the sweep uses"""
    from instructany2pix_b200.packing import pack_conv3x3, pack_conv3x3_up2x
    g = torch.Generator().manual_seed(3)
    x = torch.randint(-3, 4, (2, 8, 12, 5), generator=g).double()
    w = torch.randint(-3, 4, (6, 5, 3, 3), generator=g).double()
    xn = x.permute(0, 3, 1, 2)
    for stride in (1, 2):
        ref = F.conv2d(xn, w, stride=stride, padding=1).permute(0, 2, 3, 1)
        got = conv3x3_cols(x, stride) @ pack_conv3x3(w, dtype=torch.float64).t()
        assert torch.equal(got.reshape(ref.shape), ref)
    ref = F.conv2d(F.pad(xn, (0, 1, 0, 1)), w, stride=2).permute(0, 2, 3, 1)
    got = conv3x3_cols(x, 2, pad_end=True) @ pack_conv3x3(w, dtype=torch.float64).t()
    assert torch.equal(got.reshape(ref.shape), ref)
    up = F.conv2d(F.interpolate(xn, scale_factor=2.0, mode="nearest"), w, padding=1).permute(0, 2, 3, 1)
    w4 = pack_conv3x3_up2x(w, dtype=torch.float64)
    for par in range(4):
        py, px = divmod(par, 2)
        got = (up2x_cols(x, py, px) @ w4[par].t()).reshape(2, 8, 12, 6)
        assert torch.equal(got, up[:, py::2, px::2])
    t = torch.arange(2 * 8 * 16 * 3.0).reshape(2, 8, 16, 3)
    tl = tile_rows(t, 16, 8, 1)
    assert torch.equal(tl[1, 0], t[1, 0, 0]) and torch.equal(tl[0, 17], t[0, 1, 1])


# ------------------------------------------------------------------------------------------------ GPU
@gpu
def test_ops_receive_poisoned_memory(monkeypatch):
    """with the launches skipped, everything ops allocates for a call comes back as the poison: the helper is not a no-op"""
    from instructany2pix_b200 import ops
    monkeypatch.setattr(ops, "USE_COLSTATS", True)
    monkeypatch.setattr(ops, "_run", lambda *a: None)
    a, w = operands(256, 256, 128)
    with poisoned():
        t, tb, st = ops.gemm(a, w, out_dtype=torch.float32, want_ln=True, want_colstats=True)
        y = ops.polar_interpolate(rnd(64, dtype=torch.float32), rnd(64, dtype=torch.float32), 0.5)
    for x in (t, tb, st, t._ia2p_cs[0], y):
        assert is_poison(x).all()


def _run_checked(fn, tmp_path, want, n_launch=1):
    """profile the first call (asserting the predicted launches), then require a bit-identical second call"""
    out, got = launched(fn, tmp_path)
    assert got == expect(want, n_launch), f"launched {got}, expected {expect(want, n_launch)} (plan {want})"
    first = [x.clone() for x in (out if isinstance(out, tuple) else (out,))]
    again = fn()
    for x, y in zip(first, again if isinstance(again, tuple) else (again,)):
        assert same_bits(x, y), "second call differs"
    return out


SCHEDULES = {                                  # (M, N, K): the scheduling edge each one is for
    "even_tail": (4096, 2560, 832),            # 32 row tiles; BN 256: 160 pair units, remainder 12 -> tail split (148 SMs)
    "odd_tail": (4224, 2560, 832),             # 33 row tiles: the last pair's partner tile lies outside A (TMA zero fill)
    "ragged_odd": (4200, 2560, 832),           # 33 row tiles, the live one of the last pair has 104 rows
    "ragged_even": (4040, 2560, 832),          # 32 row tiles, the last (rank 1) has 72 rows
    "big_remainder": (5120, 2560, 832),        # BN 256: 200 units, remainder 52: too large to split
}


@gpu
@pytest.mark.parametrize("bn", [256, 160, 128])
@pytest.mark.parametrize("case", list(SCHEDULES) + ["whole_waves"])
def test_pair_schedule(case, bn, sms, poison, monkeypatch, tmp_path):
    """plain bf16 GEMMs (TMA-store epilogue) over the scheduling edges of the pair kernel at each pairing tile width"""
    from instructany2pix_b200 import ops
    monkeypatch.setenv("IA2P_GEMM_BN", str(bn))
    if case == "whole_waves":
        # N / BN = SMs / 2 pair units per row-tile pair and 2 * ceil(SMs / (SMs / 2)) row tiles: whole waves, >= 2 x SMs tiles
        G = sms // 2
        M, N, K = 128 * 2 * -(-sms // G), bn * G, 832
    else:
        M, N, K = SCHEDULES[case]
    want = plan(-(-M // 128), N, K, sms)
    assert want["bn"] == bn and want["cg"] == 2
    if case == "whole_waves":
        assert -(-M // 256) * (N // bn) % G == 0 and not want["split"]
    a, w = operands(M, N, K, seed=bn)
    out = _run_checked(lambda: ops.gemm(a, w), tmp_path, want)
    ref, mag = ref_gemm(a, w)
    check(out, ref, gemm_bound(ref, mag, K, True), bn)


@gpu
@pytest.mark.parametrize("K", [768, 832, 5120])
def test_pair_k_threshold(K, sms, poison, tmp_path):
    """the pair kernel from 13 k-blocks on (K 768 stays on the single-CTA kernel), and a long main loop"""
    from instructany2pix_b200 import ops
    M, N = (4096, 2560) if K < 5120 else (3840, 2560)
    want = plan(-(-M // 128), N, K, sms)
    a, w = operands(M, N, K, seed=K)
    out = _run_checked(lambda: ops.gemm(a, w), tmp_path, want)
    ref, mag = ref_gemm(a, w)
    check(out, ref, gemm_bound(ref, mag, K, True), want["bn"])


@gpu
def test_pair_bn160_never_splits(sms, poison, tmp_path):
    """N 640 picks BLOCK_N 160 (4 column tiles); with >= SMs / 2 row tiles it pairs, and 160 / 2 is not a whole number of
    64-column slices, so no remainder is ever split"""
    from instructany2pix_b200 import ops
    M, N, K = 128 * (sms // 2 + 2) + 40, 640, 1280
    want = plan(-(-M // 128), N, K, sms)
    assert (want["bn"], want["cg"], want["split"]) == (160, 2, False)
    a, w = operands(M, N, K, seed=7)
    bias = rnd(N, dtype=torch.float32, seed=8)
    out = _run_checked(lambda: ops.gemm(a, w, bias=bias), tmp_path, want)
    ref, mag = ref_gemm(a, w)
    ref = ref + bias.double()
    check(out, ref, gemm_bound(ref, mag, K, True), 160)


@gpu
@pytest.mark.parametrize("rows_per_batch", [77, 200])
def test_pair_bf16_tma_store_bias_rowbias_strided_out(rows_per_batch, sms, poison, tmp_path):
    """EPI 3 on pairs: bias + per-image row bias (images that start inside a tile and do not divide 128) into a row- and
    column-strided view of a larger buffer whose guard bands must keep their poison"""
    from instructany2pix_b200 import ops
    M, N, K = 4224, 2560, 1280
    want = plan(33, N, K, sms)
    a, w = operands(M, N, K, seed=rows_per_batch)
    bias = rnd(N, dtype=torch.float32, seed=1)
    rowbias = rnd(-(-M // rows_per_batch), N, dtype=torch.float32, seed=2)
    buf = torch.empty(M + 6, N + 128, device=DEV, dtype=torch.bfloat16)
    view = lambda: buf[2:2 + M, 64:64 + N]
    out = _run_checked(lambda: ops.gemm(a, w, bias=bias, rowbias=rowbias, rows_per_batch=rows_per_batch, out=view()), tmp_path, want)
    assert out.data_ptr() == view().data_ptr()
    ref, mag = ref_gemm(a, w)
    ref = ref + bias.double() + rowbias.double().repeat_interleave(rows_per_batch, 0)[:M]
    check(out, ref, gemm_bound(ref, mag, K, True), want["bn"])
    for band in (buf[:2], buf[2 + M:], buf[2:2 + M, :64], buf[2:2 + M, 64 + N:]):
        assert is_poison(band).all(), "the epilogue wrote outside the output view"
    assert rel(out, ref) < 4e-3


EPILOGUES = {   # kind: (M, N, K, out dtype, residual dtype | None)
    "ring_residual": (4096, 2560, 1280, torch.float32, torch.float32),       # EPI 2: fp32 residual ring, K <= 1536
    "fp32_residual": (4224, 2560, 2048, torch.float32, torch.float32),       # EPI 1 with residual, K > 1536, odd tail
    "fp32": (4096, 2560, 2048, torch.float32, None),                         # EPI 1
    "bf16_residual": (4096, 2560, 2048, torch.bfloat16, torch.bfloat16),     # EPI 0 (register stores)
    "bf16_out_fp32_residual": (4224, 2560, 1280, torch.bfloat16, torch.float32),   # EPI 0, odd tail
}


@gpu
@pytest.mark.parametrize("kind", list(EPILOGUES))
def test_pair_epilogues(kind, sms, poison, tmp_path):
    """bias + row bias + residual through the fp32 TMA-store (EPI 1), residual-ring (EPI 2) and register-store (EPI 0) epilogues"""
    from instructany2pix_b200 import ops
    M, N, K, odt, rdt = EPILOGUES[kind]
    res_kind = None if rdt is None else ("f32" if rdt == torch.float32 else "bf16")
    want = plan(-(-M // 128), N, K, sms, out_f32=odt == torch.float32, residual=res_kind)
    a, w = operands(M, N, K, seed=len(kind))
    bias = rnd(N, dtype=torch.float32, seed=3)
    rowbias = rnd(-(-M // 1024), N, dtype=torch.float32, seed=4)
    res = None if rdt is None else rnd(M, N, dtype=rdt, seed=5)
    out = _run_checked(lambda: ops.gemm(a, w, bias=bias, rowbias=rowbias, rows_per_batch=1024, residual=res, out_dtype=odt),
                       tmp_path, want)
    ref, mag = ref_gemm(a, w)
    ref = ref + bias.double() + rowbias.double().repeat_interleave(1024, 0)[:M] + (0 if res is None else res.double())
    check(out, ref, gemm_bound(ref, mag, K, odt == torch.bfloat16), want["bn"])
    assert rel(out, ref) < (4e-3 if odt == torch.bfloat16 else 4e-6)


@gpu
@pytest.mark.parametrize("M,K", [(4096, 1280), (4224, 2048)])
def test_pair_ln_producer_and_colstats(M, K, sms, poison, monkeypatch, tmp_path):
    """LN producer on pairs (fp32 stream + bf16 copy + per-row partial sums) with the GroupNorm column statistics: the stats
    against fp64 row sums over all parts, the copy bit-exact, the column sums per 128-row tile against fp64"""
    from instructany2pix_b200 import ops
    monkeypatch.setattr(ops, "USE_COLSTATS", True)
    N = 2560
    m_tiles = -(-M // 128)
    want = plan(m_tiles, N, K, sms, out_f32=True, residual="f32", extras=True)
    a, w = operands(M, N, K, seed=M)
    res = rnd(M, N, dtype=torch.float32, scale=2.0, seed=6) + 0.7
    t, tb, st = _run_checked(lambda: ops.gemm(a, w, residual=res, out_dtype=torch.float32, want_ln=True, want_colstats=True),
                             tmp_path, want)
    ref, mag = ref_gemm(a, w)
    ref = ref + res.double()
    check(t, ref, gemm_bound(ref, mag, K, False), want["bn"])
    assert torch.equal(tb, t.to(torch.bfloat16))
    t64 = t.double()
    sq = t64 * t64
    b_row = N * 2.0 ** -23 * (sq.sum(1) + t64.abs().sum(1)) + 1e-6
    check(st[..., 0].sum(1, dtype=torch.float64), t64.sum(1), b_row, what="LN row sums")
    check(st[..., 1].sum(1, dtype=torch.float64), sq.sum(1), b_row, what="LN row sums of squares")
    cs, segs = t._ia2p_cs
    assert segs == 1 and cs.shape == (m_tiles, N, 2)
    padded = torch.cat([t, t.new_zeros(m_tiles * 128 - M, N)]).reshape(m_tiles, 128, N)
    check_colstats(cs, padded, "gemm")


def _ln_setup(M, C, seed):
    """an LN producer output (fp32 stream t, its bf16 copy, row statistics) and a LayerNorm"""
    from instructany2pix_b200 import ops
    a0, w0 = operands(M, C, 256, seed=seed)
    res = rnd(M, C, dtype=torch.float32, scale=2.0, seed=seed + 2) + 0.7
    t, tb, st = ops.gemm(a0, w0, residual=res, out_dtype=torch.float32, want_ln=True)
    ln = torch.nn.LayerNorm(C, eps=1e-5).to(DEV)
    ln.weight.data = rnd(C, dtype=torch.float32, seed=seed + 3) * 0.3 + 1.0
    ln.bias.data = rnd(C, dtype=torch.float32, seed=seed + 4) * 0.2
    return t, tb, st, ln


def _ln_fold_ref(t, tb, wp, c1, c2, eps):
    """fp64 rstd (tb @ wp^T - mean c1) + c2 with mean / rstd of the fp32 producer output, and the per-element error bound of
    the kernel's accumulator after the fold"""
    C = t.shape[1]
    t64 = t.double()
    mean, mean_abs = t64.mean(1, keepdim=True), t64.abs().mean(1, keepdim=True)
    rstd = (t64.var(1, unbiased=False, keepdim=True) + eps).rsqrt()
    acc, mag = ref_gemm(tb, wp)
    c1, c2 = c1.double(), c2.double()
    h = rstd * (acc - mean * c1) + c2
    # accumulation (K = C additions) plus the fp32 row statistics (C-term sums: relative error below C 2^-23 as well)
    e = C * 2.0 ** -23 * (rstd * (mag + mean_abs * c1.abs()) + c2.abs()) + 1e-6
    return h, e


def _gelu_err(h, e, g):
    """error of the epilogue's g = gelu(h) (or quick-GELU) for an input off by at most e: |gelu'| <= 1.13, and the
    approximation itself (A&S 7.1.26 erf, 1.5e-7 absolute; tests/test_kernels_gpu.py::test_gelu_accuracy)"""
    return 1.13 * e + 2.0 ** -8 * g.abs() + 1e-7 * h.abs() + 1e-6


@gpu
@pytest.mark.parametrize("geglu", [False, True])
def test_pair_ln_consumer(geglu, sms, poison, tmp_path):
    """LN-folded consumer on pairs: plain (N 2560) and GEGLU at the SDXL feed-forward shape (1280 -> 10240 -> 5120), whose 320
    pair units leave a tail to split at 148 SMs"""
    from instructany2pix_b200 import ops
    from instructany2pix_b200.packing import interleave_geglu
    from instructany2pix_b200.unet import _fold_ln
    M, C = (2048, 1280) if geglu else (4096, 1280)
    N = 10240 if geglu else 2560
    t, tb, st, ln = _ln_setup(M, C, seed=20 + geglu)
    w, b = rnd(N, C, scale=C ** -0.5, seed=30), rnd(N, dtype=torch.float32, scale=0.1, seed=31)
    if geglu:
        w, b = interleave_geglu(w, b)
    wp, c1, c2, eps = _fold_ln(w, b, ln)
    want = plan(M // 128, N, C, sms, geglu=geglu)
    out = _run_checked(lambda: ops.gemm(tb, wp, bias=c2, ln=(st, c1, eps), geglu=geglu), tmp_path, want)
    h, e = _ln_fold_ref(t, tb, wp, c1, c2, eps)
    if not geglu:
        check(out, h, 2.0 ** -8 * h.abs() + e, want["bn"])
        ref_exact = F.layer_norm(t.double(), (C,), ln.weight.double(), ln.bias.double(), eps) @ w.double().t() + b.double()
        assert rel(out, ref_exact) < 8e-3
        return
    # accumulator columns in 64-wide groups [32 value | 32 gate] (interleave_geglu)
    hv, hg = h.reshape(M, N // 64, 2, 32).unbind(2)
    ev, eg = e.reshape(M, N // 64, 2, 32).unbind(2)
    gg = F.gelu(hg)
    ref = (hv * gg).reshape(M, N // 2)
    bound = (ev * gg.abs() + hv.abs() * _gelu_err(hg, eg, gg)).reshape(M, N // 2) + 2.0 ** -8 * ref.abs() + 1e-6
    check(out, ref, bound, want["bn"] // 2)
    assert rel(out, ref) < 4e-3


@gpu
@pytest.mark.parametrize("act", ["gelu", "quick_gelu"])
def test_pair_activation(act, sms, poison, tmp_path):
    from instructany2pix_b200 import ops
    M, N, K = 4096, 2560, 1280
    want = plan(32, N, K, sms)
    a, w = operands(M, N, K, seed=40)
    bias = rnd(N, dtype=torch.float32, seed=41)
    out = _run_checked(lambda: ops.gemm(a, w, bias=bias, act=act), tmp_path, want)
    acc, mag = ref_gemm(a, w)
    h = acc + bias.double()
    ref = F.gelu(h) if act == "gelu" else h * torch.sigmoid(1.702 * h)
    check(out, ref, _gelu_err(h, gemm_bound(h, mag, K, False), ref) + 2.0 ** -8 * ref.abs(), want["bn"])


@gpu
def test_pair_k_concat(sms, poison, tmp_path):
    """two A sources (row-strided views) concatenated along K on pairs"""
    from instructany2pix_b200 import ops
    M, K1, K2, N = 4224, 640, 576, 2560
    big = rnd(M, 1536, seed=50)
    a, a2 = big[:, :K1], big[:, 768:768 + K2]
    w = rnd(N, K1 + K2, scale=(K1 + K2) ** -0.5, seed=51)
    want = plan(33, N, K1 + K2, sms)
    out = _run_checked(lambda: ops.gemm(a, w, a2=a2), tmp_path, want)
    ref, mag = ref_gemm(torch.cat([a, a2], 1), w)
    check(out, ref, gemm_bound(ref, mag, K1 + K2, True), want["bn"])


# ------------------------------------------------------------------------------------------------ convs on pairs
@gpu
def test_pair_conv3x3_resnet_conv2(sms, poison, monkeypatch, tmp_path):
    """ResnetBlock conv2 at SDXL level 2 (B 4, 64 x 64, 320 -> 640): 3x3 conv + fused 1x1 shortcut + bias + temb row bias +
    fp32 residual + GroupNorm column statistics, K = 9 * 320 + 320"""
    from instructany2pix_b200 import ops
    from instructany2pix_b200.packing import pack_conv3x3
    monkeypatch.setattr(ops, "USE_COLSTATS", True)
    B, H, W, Cin, Cout, Csc = 4, 64, 64, 320, 640, 320
    x, sc = rnd(B, H, W, Cin, seed=60), rnd(B, H, W, Csc, seed=61)
    wp = pack_conv3x3(rnd(Cout, Cin, 3, 3, scale=(9 * Cin) ** -0.5, seed=62), rnd(Cout, Csc, 1, 1, scale=Csc ** -0.5, seed=63))
    bias, temb = rnd(Cout, dtype=torch.float32, seed=64), rnd(B, Cout, dtype=torch.float32, seed=65)
    res = rnd(B, H, W, Cout, dtype=torch.float32, seed=66)
    TW, TH, TB, m_tiles = conv_tile(B, H, W)
    K = wp.shape[1]
    want = plan(m_tiles, Cout, K, sms, out_f32=True, residual="f32", extras=True)
    out = _run_checked(lambda: ops.conv3x3(x, wp, Cout, sc_a=sc, bias=bias, rowbias=temb, residual=res, out_dtype=torch.float32,
                                           want_colstats=True), tmp_path, want)
    cols = torch.cat([conv3x3_cols(x), sc.double().reshape(-1, Csc)], 1)
    acc, mag = cols @ wp.double().t(), cols.abs() @ wp.double().abs().t()
    ref = (acc.reshape(B, H, W, Cout) + bias.double() + temb.double()[:, None, None] + res.double())
    check(out, ref, gemm_bound(ref, mag.reshape(ref.shape), K, False), want["bn"])
    check_colstats(out._ia2p_cs[0], tile_rows(out, TW, TH, TB), "conv3x3")


@gpu
@pytest.mark.parametrize("kind", ["stride2", "down_padend"])
def test_pair_conv3x3_downsample(kind, sms, poison, tmp_path):
    """stride-2 3x3 convs on pairs: UNet Downsample2D (pad 1) and the SDXL-VAE encoder's (pad at the bottom / right only,
    128 channels at a 512^2 input)"""
    from instructany2pix_b200 import ops
    from instructany2pix_b200.packing import pack_conv3x3
    B, H, W, Cin, Cout = (4, 128, 128, 128, 640) if kind == "stride2" else (1, 512, 512, 128, 128)
    x = rnd(B, H, W, Cin, seed=70)
    wp = pack_conv3x3(rnd(Cout, Cin, 3, 3, scale=(9 * Cin) ** -0.5, seed=71))
    bias = rnd(Cout, dtype=torch.float32, seed=72)
    _, _, _, m_tiles = conv_tile(B, H // 2, W // 2)
    want = plan(m_tiles, Cout, 9 * Cin, sms)
    assert want["cg"] == 2
    if kind == "stride2":
        out = _run_checked(lambda: ops.conv3x3(x, wp, Cout, stride=2, bias=bias), tmp_path, want)
    else:
        out = _run_checked(lambda: ops.conv3x3_down_padend(x, wp, Cout, bias=bias), tmp_path, want)
    cols = conv3x3_cols(x, 2, pad_end=kind == "down_padend")
    shape = (B, H // 2, W // 2, Cout)
    ref = (cols @ wp.double().t()).reshape(shape) + bias.double()
    mag = (cols.abs() @ wp.double().abs().t()).reshape(shape)
    check(out, ref, gemm_bound(ref, mag, 9 * Cin, True), want["bn"])


@gpu
def test_pair_conv_up2x(sms, poison, monkeypatch, tmp_path):
    """nearest-2x upsample + 3x3 conv as four parity launches on pairs (BLOCK_N 128) with its 4-segment column statistics,
    against fp64 2x2 convs of the packed parity weights"""
    from instructany2pix_b200 import ops
    from instructany2pix_b200.packing import pack_conv3x3_up2x
    monkeypatch.setattr(ops, "USE_COLSTATS", True)
    B, H, W, Cin, Cout = 4, 64, 64, 256, 384
    x = rnd(B, H, W, Cin, seed=80)
    w4 = pack_conv3x3_up2x(rnd(Cout, Cin, 3, 3, scale=(9 * Cin) ** -0.5, seed=81))
    bias = rnd(Cout, dtype=torch.float32, seed=82)
    TW, TH, TB, m_tiles = conv_tile(B, H, W)
    want = plan(m_tiles, Cout, 4 * Cin, sms, out_f32=True)
    assert want["bn"] == 128 and want["cg"] == 2
    out = _run_checked(lambda: ops.conv_up2x(x, w4, Cout, bias=bias, want_colstats=True), tmp_path, want, n_launch=4)
    cs, segs = out._ia2p_cs
    assert segs == 4 and cs.shape == (4 * m_tiles, Cout, 2)
    for par in range(4):
        py, px = divmod(par, 2)
        cols = up2x_cols(x, py, px)
        w64 = w4[par].double()
        ref = (cols @ w64.t()).reshape(B, H, W, Cout) + bias.double()
        mag = (cols.abs() @ w64.abs().t()).reshape(B, H, W, Cout)
        o = out[:, py::2, px::2]
        check(o, ref, gemm_bound(ref, mag, 4 * Cin, False), want["bn"], what=f"parity ({py}, {px})")
        check_colstats(cs[par * m_tiles:(par + 1) * m_tiles], tile_rows(o, TW, TH, TB), f"parity ({py}, {px})")


# ------------------------------------------------------------------------------------------------ programmatic dependent launch
@gpu
def test_pair_chain_bitwise_with_and_without_pdl(sms, poison, monkeypatch):
    """LN producer -> LN-folded GEGLU consumer -> feed-forward out-projection with fp32 residual, all on pairs (BLOCK_N 128), run
    once with programmatic dependent launch (each kernel loads its first weight blocks before waiting for its predecessor) and
    once without: bit-identical results"""
    from instructany2pix_b200 import ops
    from instructany2pix_b200.packing import interleave_geglu
    from instructany2pix_b200.unet import _fold_ln
    monkeypatch.setenv("IA2P_GEMM_BN", "128")
    M, C, F4 = 4096, 1280, 5120
    for n, k in ((C, C), (2 * F4, C), (C, F4)):
        assert plan(M // 128, n, k, sms, geglu=n == 2 * F4)["cg"] == 2
    a, w0 = operands(M, C, C, seed=90)
    res = rnd(M, C, dtype=torch.float32, seed=91)
    ln = torch.nn.LayerNorm(C).to(DEV)
    ln.weight.data = rnd(C, dtype=torch.float32, seed=92) * 0.3 + 1.0
    ln.bias.data = rnd(C, dtype=torch.float32, seed=93) * 0.2
    wi, bi = interleave_geglu(rnd(2 * F4, C, scale=C ** -0.5, seed=94), rnd(2 * F4, dtype=torch.float32, scale=0.1, seed=95))
    wp, c1, c2, eps = _fold_ln(wi, bi, ln)
    w2, b2 = rnd(C, F4, scale=F4 ** -0.5, seed=96), rnd(C, dtype=torch.float32, seed=97)

    def chain():
        t, tb, st = ops.gemm(a, w0, residual=res, out_dtype=torch.float32, want_ln=True)
        h = ops.gemm(tb, wp, bias=c2, ln=(st, c1, eps), geglu=True)
        return t, h, ops.gemm(h, w2, bias=b2, residual=t, out_dtype=torch.float32)

    plain = chain()
    with ops.pdl():
        overlapped = chain()
    torch.cuda.synchronize()
    for x, y in zip(plain, overlapped):
        assert not torch.isnan(x).any() and same_bits(x, y)
