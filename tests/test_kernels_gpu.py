"""GPU unit tests of every C-ABI kernel against a plain torch fp32 reference of the same op (tolerances stated inline).
Every test runs on poisoned allocations (tests/_poison.py), so each one also proves that its kernels write their whole output."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from instructany2pix_b200 import ops  # noqa: E402
from tests._poison import poisoned  # noqa: E402


@pytest.fixture(autouse=True)
def _poisoned_allocations():
    with poisoned():
        yield

DEV = "cuda"
# references must be true fp32 (cuDNN/cuBLAS default to TF32 for fp32 inputs)
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False


def rnd(*shape, scale=1.0, dtype=torch.bfloat16, seed=None):
    g = torch.Generator(device="cpu")
    g.manual_seed(hash(shape) % (2 ** 31) if seed is None else seed)
    return (torch.randn(*shape, generator=g) * scale).to(dtype).to(DEV)


def rel(a, b):
    a, b = a.float(), b.float()
    return ((a - b).norm() / b.norm().clamp_min(1e-12)).item()


# bf16 output rounding is 2^-9 relative per element; accumulation is fp32 -> rel-L2 of a correct kernel ~2e-3
TOL = 4e-3


@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (256, 256, 128), (128, 320, 64), (1000, 640, 1280), (154, 2560, 2048),
                                   (4096, 1280, 640), (512, 64, 192), (300, 1920, 640)])
def test_gemm_plain(M, N, K):
    a, w = rnd(M, K), rnd(N, K, scale=K ** -0.5)
    out = ops.gemm(a, w)
    assert rel(out, a.float() @ w.float().t()) < TOL


@pytest.mark.parametrize("mode", ["plain", "res32_ln", "geglu"])
def test_gemm_tail_split(mode):
    """tile counts that leave a small last wave (here 160 and 320 tiles on 148 SMs) run that wave as half-width tiles."""
    from instructany2pix_b200.packing import interleave_geglu
    M, N, K = (2048, 2560, 192) if mode != "geglu" else (2048 * 2, 2560, 128)
    a, w = rnd(M, K), rnd(N, K, scale=K ** -0.5)
    ref = a.float() @ w.float().t()
    if mode == "plain":
        assert rel(ops.gemm(a, w), ref) < TOL
    elif mode == "res32_ln":
        res = rnd(M, N, dtype=torch.float32)
        t, tb, st = ops.gemm(a, w, residual=res, out_dtype=torch.float32, want_ln=True)
        assert rel(t, ref + res) < 2e-6 and torch.equal(tb, t.to(torch.bfloat16))
        assert rel(st.sum(1)[:, 0], t.sum(1)) < 1e-5 and rel(st.sum(1)[:, 1], (t * t).sum(1)) < 1e-5
    else:
        b = rnd(N, dtype=torch.float32, scale=0.1)
        wi, bi = interleave_geglu(w, b)
        h = ref + b
        assert rel(ops.gemm(a, wi, bias=bi, geglu=True), h[:, :N // 2] * F.gelu(h[:, N // 2:])) < TOL


@pytest.mark.parametrize("bn", [64, 128, 160, 256])
@pytest.mark.parametrize("M", [384, 1000])
def test_gemm_every_tile_width(bn, M, monkeypatch):
    """the tile-width heuristic sends small problems to BLOCK_N 64; force each width over all epilogue variants (bf16 store,
    TMA store, TMA residual ring + LN statistics, LN-folded consumer, GEGLU)."""
    from instructany2pix_b200.packing import interleave_geglu
    from instructany2pix_b200.unet import _fold_ln
    monkeypatch.setenv("IA2P_GEMM_BN", str(bn))
    N, K = 1280, 320
    a, w = rnd(M, K), rnd(N, K, scale=K ** -0.5)
    ref = a.float() @ w.float().t()
    assert rel(ops.gemm(a, w), ref) < TOL
    bias, res = rnd(N, dtype=torch.float32), rnd(M, N, dtype=torch.float32)
    assert rel(ops.gemm(a, w, bias=bias, out_dtype=torch.float32), ref + bias) < 2e-6
    t, tb, st = ops.gemm(a, w, bias=bias, residual=res, out_dtype=torch.float32, want_ln=True)
    assert rel(t, ref + bias + res) < 2e-6 and torch.equal(tb, t.to(torch.bfloat16))
    assert rel(st.sum(1)[:, 0], t.sum(1)) < 1e-5 and rel(st.sum(1)[:, 1], (t * t).sum(1)) < 1e-5
    ln = torch.nn.LayerNorm(N, eps=1e-5).to(DEV)
    ln.weight.data = rnd(N, dtype=torch.float32) * 0.3 + 1.0
    ln.bias.data = rnd(N, dtype=torch.float32) * 0.2
    if bn != 160:                                       # GEGLU needs 64-column value|gate groups
        w2, b2 = rnd(2560, N, scale=N ** -0.5), rnd(2560, dtype=torch.float32, scale=0.1)
        wi, bi = interleave_geglu(w2, b2)
        wp, c1, c2, eps = _fold_ln(wi, bi, ln)
        out = ops.gemm(tb, wp, bias=c2, ln=(st, c1, eps), geglu=True)
        h = F.layer_norm(t, (N,), ln.weight, ln.bias, 1e-5) @ w2.float().t() + b2
        assert rel(out, h[:, :1280] * F.gelu(h[:, 1280:])) < 8e-3
    w3 = rnd(640, N, scale=N ** -0.5)
    wp, c1, c2, eps = _fold_ln(w3, None, ln)
    out = ops.gemm(tb, wp, bias=c2, ln=(st, c1, eps))
    assert rel(out, F.layer_norm(t, (N,), ln.weight, ln.bias, 1e-5) @ w3.float().t()) < 8e-3


@pytest.mark.parametrize("path", ["multicast", "splitk"])
@pytest.mark.parametrize("kind", ["plain", "fp32_ln", "res_ring", "geglu", "conv", "conv_res", "conv_s2", "conv_8x8", "up2x", "kcat"])
def test_few_row_problems(kind, path, monkeypatch):
    """Problems that fit in one wave of tiles (batch-1 512^2, single requests), two opt-in paths (both measured, neither faster than
    one narrow tile per CTA: DESIGN.md).  "multicast" (IA2P_GEMM_MC): clusters of 2 / 4
    CTAs share each A block through TMA multicast (plain rows, 16x8 / 8x8x2 / 32x4 pixel boxes, parity-decimated stride-2 maps,
    two K-concatenated sources).  "splitk" (ops.USE_SPLITK): every tile is computed by several CTAs over disjoint
    k-ranges and the partials are summed in a fixed order.  Both: same results as the reference, bit-reproducible run to run."""
    from instructany2pix_b200 import _lib
    from instructany2pix_b200.packing import interleave_geglu, pack_conv3x3, pack_conv3x3_up2x
    if not _lib.load().ia2p_tc_features() & (1 if path == "splitk" else 2):
        if kind not in ("plain", "conv_8x8"):
            pytest.skip("experiment path not compiled into the shipped library (make variant DEFS=-DIA2P_WITH_SPLITK -DIA2P_WITH_MC)")
        # the shipped build: the same shapes still run (and must be right) on the one-tile-per-CTA path
    monkeypatch.setattr(ops, "USE_SPLITK", path == "splitk")
    if path == "multicast":
        monkeypatch.setenv("IA2P_GEMM_MC", "4")
    if kind == "plain":
        a, w = rnd(384, 2560), rnd(1280, 2560, scale=2560 ** -0.5)
        f = lambda: ops.gemm(a, w)
        ref, tol = a.float() @ w.float().t(), TOL
    elif kind == "fp32_ln":
        a, w = rnd(512, 5120), rnd(1280, 5120, scale=5120 ** -0.5)
        bias, res = rnd(1280, dtype=torch.float32), rnd(512, 1280, dtype=torch.float32)
        f = lambda: ops.gemm(a, w, bias=bias, residual=res, out_dtype=torch.float32, want_ln=True, want_colstats=True)[0]
        ref, tol = a.float() @ w.float().t() + bias + res, 3e-6
    elif kind == "res_ring":
        a, w = rnd(256, 1280), rnd(640, 1280, scale=1280 ** -0.5)
        res = rnd(256, 640, dtype=torch.float32)
        f = lambda: ops.gemm(a, w, residual=res, out_dtype=torch.float32)
        ref, tol = a.float() @ w.float().t() + res, 3e-6
    elif kind == "geglu":
        a, w, b = rnd(256, 1024), rnd(2560, 1024, scale=1024 ** -0.5), rnd(2560, dtype=torch.float32, scale=0.1)
        wi, bi = interleave_geglu(w, b)
        f = lambda: ops.gemm(a, wi, bias=bi, geglu=True)
        h = a.float() @ w.float().t() + b
        ref, tol = h[:, :1280] * F.gelu(h[:, 1280:]), TOL
    elif kind == "kcat":
        a, a2, w = rnd(512, 640), rnd(512, 320), rnd(1280, 960, scale=960 ** -0.5)
        f = lambda: ops.gemm(a, w, a2=a2)
        ref, tol = torch.cat([a, a2], 1).float() @ w.float().t(), TOL
    elif kind == "conv_s2":
        x, w = rnd(2, 32, 32, 128), rnd(512, 128, 3, 3, scale=(9 * 128) ** -0.5)
        f = lambda: ops.conv3x3(x, pack_conv3x3(w), 512, stride=2)
        ref, tol = _conv_ref(x, w, 2), TOL
    elif kind == "conv_8x8":
        x, w = rnd(3, 8, 8, 128), rnd(512, 128, 3, 3, scale=(9 * 128) ** -0.5)     # tile = 2 images x 8 x 8, last one half empty
        f = lambda: ops.conv3x3(x, pack_conv3x3(w), 512)
        ref, tol = _conv_ref(x, w), TOL
    elif kind == "up2x":
        x, w, b = rnd(1, 32, 32, 128), rnd(256, 128, 3, 3, scale=(9 * 128) ** -0.5), rnd(256, dtype=torch.float32)
        f = lambda: ops.conv_up2x(x, pack_conv3x3_up2x(w), 256, bias=b)
        up = F.interpolate(x.float().permute(0, 3, 1, 2), scale_factor=2.0, mode="nearest")
        ref, tol = F.conv2d(up, w.float(), b, padding=1).permute(0, 2, 3, 1), 3e-3
    else:
        x, w = rnd(2, 16, 16, 640), rnd(1280, 640, 3, 3, scale=(9 * 640) ** -0.5)
        res = rnd(2, 16, 16, 1280, dtype=torch.float32) if kind == "conv_res" else None
        f = lambda: ops.conv3x3(x, pack_conv3x3(w), 1280, residual=res, out_dtype=torch.float32, want_colstats=True)
        ref, tol = _conv_ref(x, w) + (0 if res is None else res), 3e-6
    out = f()
    assert rel(out, ref) < tol
    assert torch.equal(out, f())
    if kind == "fp32_ln":
        t, tb, st = ops.gemm(a, w, bias=bias, residual=res, out_dtype=torch.float32, want_ln=True)
        assert torch.equal(tb, t.to(torch.bfloat16)) and rel(st.sum(1)[:, 0], t.sum(1)) < 1e-5


@pytest.mark.parametrize("M,N", [(200, 96), (384, 160), (1000, 224), (128, 32)])
def test_gemm_bf16_tma_store_ragged_widths(M, N):
    """bf16 outputs leave through 64-column TMA-store slices (EPI 3): widths with a 32-column remainder slice, rows past M and a
    row-strided destination must neither lose nor spill a column; bias + per-image row bias applied in the same epilogue."""
    K = 128
    a, w = rnd(M, K), rnd(N, K, scale=K ** -0.5)
    bias = rnd(N, dtype=torch.float32)
    rpb = 8
    rowbias = rnd((M + rpb - 1) // rpb, N, dtype=torch.float32)
    buf = torch.full((M + 3, N + 64), 7.0, device=DEV, dtype=torch.bfloat16)
    out = ops.gemm(a, w, bias=bias, rowbias=rowbias, rows_per_batch=rpb, out=buf[:M, 32:32 + N])
    ref = a.float() @ w.float().t() + bias + rowbias.repeat_interleave(rpb, 0)[:M]
    assert rel(out, ref) < TOL
    assert (buf[:M, :32] == 7.0).all() and (buf[:M, 32 + N:] == 7.0).all() and (buf[M:] == 7.0).all()


def test_gemm_epilogues():
    M, N, K = 768, 640, 320
    a, w = rnd(M, K), rnd(N, K, scale=K ** -0.5)
    bias = rnd(N, dtype=torch.float32)
    rowbias = rnd(3, N, dtype=torch.float32)
    res = rnd(M, N)
    ref = a.float() @ w.float().t() + bias + rowbias.repeat_interleave(256, 0) + res.float()
    out = ops.gemm(a, w, bias=bias, rowbias=rowbias, rows_per_batch=256, residual=res)
    assert rel(out, ref) < TOL


def test_gemm_fp32_stream():
    """residual-stream variant: fp32 residual in, fp32 out (only tensor-core operands are bf16)."""
    M, N, K = 512, 1280, 640
    a, w = rnd(M, K), rnd(N, K, scale=K ** -0.5)
    bias, res = rnd(N, dtype=torch.float32), rnd(M, N, dtype=torch.float32)
    out = ops.gemm(a, w, bias=bias, residual=res, out_dtype=torch.float32)
    assert out.dtype == torch.float32
    assert rel(out, a.float() @ w.float().t() + bias + res) < 2e-6
    out2 = ops.gemm(a, w, residual=res)          # fp32 residual, bf16 out
    assert out2.dtype == torch.bfloat16 and rel(out2, a.float() @ w.float().t() + res) < TOL


@pytest.mark.parametrize("M,C,N,geglu", [(512, 1280, 3840, False), (1000, 640, 640, False), (384, 640, 5120, True), (256, 128, 192, False)])
def test_gemm_layernorm_fold(M, C, N, geglu):
    """producer (fp32 stream + bf16 copy + row statistics) -> consumer (LayerNorm finished in the epilogue)."""
    from instructany2pix_b200.packing import interleave_geglu
    from instructany2pix_b200.unet import _fold_ln
    a0, w0 = rnd(M, 256), rnd(C, 256, scale=256 ** -0.5)
    res = rnd(M, C, dtype=torch.float32, scale=2.0) + 0.7          # non-zero row means
    t, tb, st = ops.gemm(a0, w0, residual=res, out_dtype=torch.float32, want_ln=True)
    t_ref = a0.float() @ w0.float().t() + res
    assert rel(t, t_ref) < 2e-6 and torch.equal(tb, t.to(torch.bfloat16))
    assert rel(st.sum(1)[:, 0], t.sum(1)) < 1e-5 and rel(st.sum(1)[:, 1], (t * t).sum(1)) < 1e-5
    ln = torch.nn.LayerNorm(C, eps=1e-5).to(DEV)
    ln.weight.data = rnd(C, dtype=torch.float32) * 0.3 + 1.0
    ln.bias.data = rnd(C, dtype=torch.float32) * 0.2
    w = rnd(N, C, scale=C ** -0.5)
    b = rnd(N, dtype=torch.float32, scale=0.1)
    if geglu:
        w, b = interleave_geglu(w, b)
    wp, c1, c2, eps = _fold_ln(w, b, ln)
    out = ops.gemm(tb, wp, bias=c2, ln=(st, c1, eps), geglu=geglu)
    h = F.layer_norm(t, (C,), ln.weight, ln.bias, 1e-5) @ w.float().t() + b
    if geglu:
        hv = h.reshape(M, N // 64, 2, 32)
        h = (hv[:, :, 0] * F.gelu(hv[:, :, 1])).reshape(M, N // 2)
    # vs exact fp32 LayerNorm + Linear: operand rounding (raw rows and gamma-scaled weights in bf16) ~ 2^-8
    assert rel(out, h) < 8e-3


def test_gemm_k_concat_and_strided_views():
    M, K1, K2, N = 640, 128, 192, 320
    big = rnd(M, 512)
    a, a2 = big[:, :K1], big[:, 256:256 + K2]          # row-strided views
    w = rnd(N, K1 + K2, scale=(K1 + K2) ** -0.5)
    outbuf = torch.zeros(M, 2 * N, device=DEV, dtype=torch.bfloat16)
    out = ops.gemm(a, w, a2=a2, out=outbuf[:, N:])
    ref = torch.cat([a, a2], 1).float() @ w.float().t()
    assert rel(out, ref) < TOL
    assert outbuf[:, :N].abs().max().item() == 0


@pytest.mark.parametrize("M,C", [(512, 128), (1000, 640)])
def test_gemm_geglu(M, C):
    a = rnd(M, C)
    w = rnd(8 * C, C, scale=C ** -0.5)           # diffusers layout: rows [0,4C) value, [4C,8C) gate
    b = rnd(8 * C, dtype=torch.float32, scale=0.1)
    from instructany2pix_b200.packing import interleave_geglu
    wi, bi = interleave_geglu(w, b)
    out = ops.gemm(a, wi, bias=bi, geglu=True)
    h = a.float() @ w.float().t() + b
    ref = h[:, :4 * C] * F.gelu(h[:, 4 * C:])
    assert out.shape == (M, 4 * C)
    assert rel(out, ref) < TOL


@pytest.mark.parametrize("kind", ["gemm", "gemm_res", "conv", "conv_res", "up2x", "down"])
def test_groupnorm_statistics_from_the_producer_epilogue(kind):
    """the fp32-output epilogue emits per-tile column sums; GroupNorm built on them equals GroupNorm with its own pass."""
    from instructany2pix_b200.packing import pack_conv3x3, pack_conv3x3_up2x
    B, H, W, C = 2, 16, 16, 128                     # hw = 256 = two row tiles per image
    if kind.startswith("gemm"):
        a, w = rnd(B * H * W, 192), rnd(C, 192, scale=192 ** -0.5)
        res = rnd(B * H * W, C, dtype=torch.float32) if kind == "gemm_res" else None
        x = ops.gemm(a, w, bias=rnd(C, dtype=torch.float32), residual=res, out_dtype=torch.float32, want_colstats=True)
        cs, segs = x._ia2p_cs
        x4 = x.reshape(B, H, W, C)
        x4._ia2p_cs = (cs, segs)
    elif kind.startswith("conv"):
        xi, w = rnd(B, H, W, 64), rnd(C, 64, 3, 3, scale=(9 * 64) ** -0.5)
        res = rnd(B, H, W, C, dtype=torch.float32) if kind == "conv_res" else None
        x4 = ops.conv3x3(xi, pack_conv3x3(w), C, bias=rnd(C, dtype=torch.float32), residual=res, out_dtype=torch.float32, want_colstats=True)
        cs, segs = x4._ia2p_cs
    elif kind == "up2x":
        xi, w = rnd(B, H, W, 64), rnd(C, 64, 3, 3, scale=(9 * 64) ** -0.5)
        x4 = ops.conv_up2x(xi, pack_conv3x3_up2x(w), C, bias=rnd(C, dtype=torch.float32), want_colstats=True)
        cs, segs = x4._ia2p_cs
        assert segs == 4
    else:
        xi, w = rnd(B, 2 * H, 2 * W, 64), rnd(C, 64, 3, 3, scale=(9 * 64) ** -0.5)
        x4 = ops.conv3x3(xi, pack_conv3x3(w), C, stride=2, out_dtype=torch.float32, want_colstats=True)
        cs, segs = x4._ia2p_cs
    # the column sums themselves: every channel's total over all tiles equals the tensor's
    assert rel(cs[..., 0].sum(0), x4.double().sum((0, 1, 2))) < 1e-5 and rel(cs[..., 1].sum(0), (x4.double() ** 2).sum((0, 1, 2))) < 1e-5
    g, b = rnd(C, dtype=torch.float32) * 0.2 + 1.0, rnd(C, dtype=torch.float32) * 0.1
    y_cs = ops.groupnorm(x4, None, g, b, 32, 1e-5, True)
    plain = x4.clone()                                # a copy carries no statistics -> separate pass
    y_own = ops.groupnorm(plain, None, g, b, 32, 1e-5, True)
    ref = F.silu(F.group_norm(x4.permute(0, 3, 1, 2), 32, g, b, 1e-5)).permute(0, 2, 3, 1)
    assert rel(y_cs, ref) < TOL and rel(y_own, ref) < TOL
    assert (y_cs.float() - y_own.float()).abs().max() <= 2 ** -7 * ref.abs().max()      # same up to one bf16 ulp
    # concat of two sources, both with statistics
    if kind == "conv":
        x5 = ops.conv3x3(rnd(B, H, W, 64, seed=9), pack_conv3x3(rnd(64, 64, 3, 3, scale=0.04, seed=10)), 64, out_dtype=torch.float32, want_colstats=True)
        g2, b2 = rnd(C + 64, dtype=torch.float32) * 0.2 + 1.0, rnd(C + 64, dtype=torch.float32) * 0.1
        y = ops.groupnorm(x4, x5, g2, b2, 32, 1e-5, False)
        ref = F.group_norm(torch.cat([x4, x5], -1).permute(0, 3, 1, 2), 32, g2, b2, 1e-5).permute(0, 2, 3, 1)
        assert rel(y, ref) < TOL


def test_polar_interpolate_matches_reference_golden():
    """pipeline.py:295-300 run by oracle/gen_golden.py on the reference's own function (tests/golden/scalar_fns.npz), plus a
    full-size latent against the same formula in fp64."""
    import os
    import numpy as np
    from oracle.synth import synth_input
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "scalar_fns.npz"))
    x, y = synth_input("bd/x", (1, 4, 8, 8)), synth_input("polar/y", (1, 4, 8, 8))
    out = ops.polar_interpolate(x.to(DEV), y.to(DEV), 0.7)
    np.testing.assert_allclose(out.cpu().numpy(), gold["polar"], rtol=2e-6, atol=2e-6)
    x, y = rnd(1, 4, 128, 128, dtype=torch.float32, seed=5), rnd(1, 4, 128, 128, dtype=torch.float32, seed=6)
    out = ops.polar_interpolate(x, y, 0.3)
    xd, yd = x.double(), y.double()
    ll = xd * 0.3 + yd * 0.7
    ref = ll / ll.norm() * (xd.norm() * 0.3 + yd.norm() * 0.7)
    assert rel(out, ref) < 1e-6
    assert torch.equal(out, ops.polar_interpolate(x, y, 0.3))        # bit-reproducible (no atomics)


def test_gelu_accuracy():
    """the epilogue's exact-GELU evaluation (A&S 7.1.26) against torch's erf GELU in fp64, through a GEGLU GEMM whose value
    half is the constant 1 and whose gate half sweeps [-10, 10]: |error| must stay below bf16 output rounding (2^-9 rel)."""
    from instructany2pix_b200.packing import interleave_geglu
    M, C = 256, 64
    a = torch.zeros(M, C, device=DEV, dtype=torch.bfloat16)
    a[:, 0] = 1.0
    w = torch.zeros(8 * C, C, device=DEV, dtype=torch.bfloat16)            # rows [0,4C) value, [4C,8C) gate
    g = torch.linspace(-10, 10, 4 * C, device=DEV).to(torch.bfloat16)
    w[:4 * C, 0] = 1.0
    w[4 * C:, 0] = g
    b = torch.zeros(8 * C, device=DEV)
    wi, bi = interleave_geglu(w, b)
    out = ops.gemm(a, wi, bias=bi, geglu=True).float()
    ref = F.gelu(g.double()).float().expand(M, -1)
    assert ((out - ref).abs() <= 2 ** -8 * ref.abs() + 1e-6).all()


def _conv_ref(x, w, stride=1):
    return F.conv2d(x.float().permute(0, 3, 1, 2), w.float(), stride=stride, padding=1).permute(0, 2, 3, 1)


@pytest.mark.parametrize("B,H,W,Cin,Cout,stride", [(2, 16, 16, 64, 64, 1), (1, 32, 32, 128, 160, 1), (3, 8, 8, 64, 128, 1),
                                                   (2, 64, 64, 64, 320, 1), (2, 32, 32, 128, 128, 2), (1, 16, 16, 64, 64, 2),
                                                   (2, 128, 128, 64, 64, 1), (5, 4, 4, 64, 32, 1), (1, 24, 48, 64, 64, 1)])
def test_conv3x3(B, H, W, Cin, Cout, stride):
    from instructany2pix_b200.packing import pack_conv3x3
    x = rnd(B, H, W, Cin)
    w = rnd(Cout, Cin, 3, 3, scale=(9 * Cin) ** -0.5)
    out = ops.conv3x3(x, pack_conv3x3(w), Cout, stride=stride)
    assert rel(out, _conv_ref(x, w, stride)) < TOL


@pytest.mark.parametrize("B,H,W,Cin,Cout", [(2, 16, 16, 64, 64), (1, 32, 32, 128, 160), (2, 64, 64, 64, 320), (3, 8, 8, 64, 128), (1, 24, 48, 64, 64)])
def test_conv_up2x(B, H, W, Cin, Cout):
    """nearest-2x upsample + 3x3 conv as four parity 2x2 convs over the low-res map (pre-summed weights) vs the plain formula."""
    from instructany2pix_b200.packing import pack_conv3x3_up2x
    x = rnd(B, H, W, Cin)
    w = rnd(Cout, Cin, 3, 3, scale=(9 * Cin) ** -0.5)
    b = rnd(Cout, dtype=torch.float32)
    out = ops.conv_up2x(x, pack_conv3x3_up2x(w), Cout, bias=b)
    up = F.interpolate(x.float().permute(0, 3, 1, 2), scale_factor=2.0, mode="nearest")
    ref = F.conv2d(up, w.float(), b, padding=1).permute(0, 2, 3, 1)
    assert out.shape == ref.shape == (B, 2 * H, 2 * W, Cout)
    assert rel(out, ref) < 3e-3          # the summed taps are re-rounded to bf16 (2^-9 on those weights)


def test_conv3x3_fused_shortcut_bias_temb_residual():
    from instructany2pix_b200.packing import pack_conv3x3
    B, H, W, Cin, Cout, Ca, Cb = 2, 16, 16, 128, 64, 64, 128
    x = rnd(B, H, W, Cin)
    w = rnd(Cout, Cin, 3, 3, scale=(9 * Cin) ** -0.5)
    sa, sb = rnd(B, H, W, Ca), rnd(B, H, W, Cb)
    wsc = rnd(Cout, Ca + Cb, 1, 1, scale=(Ca + Cb) ** -0.5)
    bias = rnd(Cout, dtype=torch.float32)
    temb = rnd(B, Cout, dtype=torch.float32)
    res = rnd(B, H, W, Cout)
    out = ops.conv3x3(x, pack_conv3x3(w, wsc), Cout, sc_a=sa, sc_b=sb, bias=bias, rowbias=temb, residual=res)
    ref = _conv_ref(x, w) + torch.cat([sa, sb], -1).float() @ wsc.float().reshape(Cout, -1).t() + bias \
        + temb[:, None, None, :] + res.float()
    assert rel(out, ref) < TOL
    out32 = ops.conv3x3(x, pack_conv3x3(w, wsc), Cout, sc_a=sa, sc_b=sb, bias=bias, rowbias=temb, residual=res.float(),
                        out_dtype=torch.float32)
    assert out32.dtype == torch.float32 and rel(out32, ref) < 2e-6


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("B,HW,Ca,Cb,silu", [(2, 256, 64, 0, True), (2, 1024, 320, 0, True), (3, 64, 640, 320, True),
                                             (1, 4096, 1280, 0, False), (2, 100, 1280, 1280, True)])
def test_groupnorm(B, HW, Ca, Cb, silu, dtype):
    xa = (rnd(B, HW, Ca, scale=2.0, dtype=torch.float32) + 0.5).to(dtype)
    xb = rnd(B, HW, Cb, dtype=dtype) if Cb else None
    C = Ca + Cb
    gamma, beta = rnd(C, dtype=torch.float32) + 1.0, rnd(C, dtype=torch.float32)
    out, raw = ops.groupnorm(xa, xb, gamma, beta, 32, 1e-5, silu, want_raw=True)
    x = xa if xb is None else torch.cat([xa, xb], -1)
    ref = F.group_norm(x.float().permute(0, 2, 1), 32, gamma, beta, 1e-5).permute(0, 2, 1)
    if silu:
        ref = F.silu(ref)
    assert out.dtype == torch.bfloat16 and rel(out, ref) < TOL
    assert torch.equal(raw, x.to(torch.bfloat16))
    assert torch.equal(ops.groupnorm(xa, xb, gamma, beta, 32, 1e-5, silu), out)


@pytest.mark.parametrize("rows,cols,dtype,odt", [(1000, 640, torch.bfloat16, torch.bfloat16), (512, 1280, torch.float32, torch.bfloat16),
                                                 (28, 1024, torch.float32, torch.float32), (7, 64, torch.bfloat16, torch.bfloat16),
                                                 (4, 2048, torch.float32, torch.float32), (300, 640, torch.float32, torch.bfloat16)])
def test_layernorm(rows, cols, dtype, odt):
    x = rnd(rows, cols, dtype=dtype, scale=1.5) + 0.3
    gamma, beta = rnd(cols, dtype=torch.float32) + 1.0, rnd(cols, dtype=torch.float32)
    out = ops.layernorm(x, gamma, beta, 1e-5, out_dtype=odt)
    ref = F.layer_norm(x.float(), (cols,), gamma, beta, 1e-5)
    assert out.dtype == odt and rel(out, ref) < (TOL if odt == torch.bfloat16 else 1e-5)


@pytest.mark.parametrize("B,N,heads", [(2, 256, 2), (1, 1024, 10), (2, 200, 1), (1, 64, 4), (1, 4096, 2)])
def test_flash_self_attn(B, N, heads):
    C = heads * 64
    qkv = rnd(B * N, 3 * C)
    out = ops.flash_self_attn(qkv, B, N, heads)
    q, k, v = [t.float().reshape(B, N, heads, 64).transpose(1, 2) for t in qkv.split(C, dim=1)]
    ref = F.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(B * N, C)
    assert rel(out, ref) < 6e-3        # P is rounded to bf16 before P.V (as in flash-attention): ~2^-9 extra


@pytest.mark.parametrize("B,N,heads,gain", [(1, 1024, 2, 8.0), (2, 300, 1, 8.0), (1, 2048, 1, 20.0), (1, 130, 2, 12.0)])
def test_flash_self_attn_peaked_rows(B, N, heads, gain):
    """Peaked softmax rows: the standing reference maximum (first block: taken from its first 32 keys only) is stale by far more than
    2^20 for many rows, so the sum check must send them through the exact-max path, rescale O in TMEM, and later blocks must survive
    logits hundreds of units below the reference (polynomial exponent clamp).  One key late in the sequence towers over everything."""
    C = heads * 64
    qkv = rnd(B * N, 3 * C)
    qkv[:, :C] *= gain                                            # logits ~ N(0, gain^2)
    qkv[N - 7, C:2 * C] = qkv[5, :C] * 3.0 / gain                  # a key aligned with query 5 of batch 0: a huge logit in the last block
    out = ops.flash_self_attn(qkv, B, N, heads)
    assert torch.isfinite(out.float()).all()
    q, k, v = [t.float().reshape(B, N, heads, 64).transpose(1, 2) for t in qkv.split(C, dim=1)]
    ref = F.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(B * N, C)
    assert rel(out, ref) < 8e-3


@pytest.mark.parametrize("n_text,n_ip,scale,B,N,heads", [
    (77, 4, 1.0, 2, 300, 3), (73, 4, 0.6, 2, 300, 3), (81, 0, 1.0, 2, 300, 3), (77, 4, 0.0, 2, 300, 3),
    (120, 16, 0.5, 2, 300, 3),                 # 136 key columns: falls back to the mma.sync kernel
    (100, 4, 0.8, 1, 128, 2), (112, 16, 1.0, 1, 200, 1), (128, 0, 1.0, 2, 130, 2), (96, 0, 1.0, 1, 64, 4), (1, 1, 1.0, 1, 40, 1),
    (77, 4, 1.0, 8, 1024, 20),                 # c3 level-2 shape: 1280 work items on the persistent grid (several per CTA)
    (77, 4, 1.0, 2, 4096, 10),                 # level-1 shape
])
def test_decoupled_cross_attn(n_text, n_ip, scale, B, N, heads):
    C = heads * 64
    q = rnd(B * N, C)
    kvt = rnd(B * n_text, 2 * C)
    kvi = rnd(B * n_ip, 2 * C) if n_ip else None
    out = ops.cross_attn(q, kvt, n_text, kvi, n_ip, scale, B, N, heads)
    hq = q.float().reshape(B, N, heads, 64).transpose(1, 2)
    sp = lambda t, n: t.float().reshape(B, n, heads, 64).transpose(1, 2)
    ref = F.scaled_dot_product_attention(hq, sp(kvt[:, :C], n_text), sp(kvt[:, C:], n_text))
    if n_ip:
        ref = ref + scale * F.scaled_dot_product_attention(hq, sp(kvi[:, :C], n_ip), sp(kvi[:, C:], n_ip))
    assert rel(out, ref.transpose(1, 2).reshape(B * N, C)) < 6e-3


def test_cfg_ddim_and_axpby():
    B, n = 3, 4 * 32 * 32
    for dt in (torch.float32, torch.bfloat16, torch.float16):
        eps2, x = rnd(2 * B, n, dtype=dt), rnd(B, n, dtype=dt)
        nxt = torch.empty(2 * B, n, device=DEV, dtype=dt)
        out = ops.cfg_ddim_step(eps2, x, 7.5, 1.01, -0.05, x_in_next2=nxt)
        eu, ec = eps2.float().chunk(2)
        ref = 1.01 * x.float() + (-0.05) * (eu + 7.5 * (ec - eu))
        tol = 1e-6 if dt == torch.float32 else 5e-3
        assert rel(out, ref) < tol and rel(nxt, torch.cat([ref, ref])) < tol
        assert rel(ops.axpby(eps2[:B], x, 0.9, 0.2), 0.9 * x.float() + 0.2 * eps2[:B].float()) < tol


def test_prior_step_and_timestep_embedding():
    n = 1024
    x0, x, noise = rnd(2, n, dtype=torch.float32), rnd(n, dtype=torch.float32), rnd(n, dtype=torch.float32)
    sa, s1 = 0.8, 0.6
    out = ops.prior_cfg_ddpm_step(x0, x, noise, sa, s1, 10.0, 0.3, 0.7, 0.05)
    ec, eu = (x - sa * x0[0]) / s1, (x - sa * x0[1]) / s1
    e = eu + 10.0 * (ec - eu)
    ref = 0.3 * (x - s1 * e) / sa + 0.7 * x + 0.05 * noise
    assert rel(out, ref) < 1e-5
    t = torch.tensor([981.0, 1.0, 6.5], device=DEV)
    emb = ops.timestep_embedding(t, 320, True, 0.0)
    half = 160
    f = torch.exp(-math.log(10000) * torch.arange(half, device=DEV, dtype=torch.float32) / half)
    a = t[:, None] * f[None]
    assert rel(emb, torch.cat([a.cos(), a.sin()], -1)) < 2e-4     # fast sin/cos at arguments up to ~1e3


def test_upsample_conv_in_out():
    x = rnd(2, 8, 8, 64)
    up = ops.upsample2x(x)
    assert torch.equal(up, x.repeat_interleave(2, 1).repeat_interleave(2, 2))
    x32 = rnd(2, 8, 8, 64, dtype=torch.float32)
    assert torch.equal(ops.upsample2x(x32), x32.to(torch.bfloat16).repeat_interleave(2, 1).repeat_interleave(2, 2))
    assert torch.equal(ops.to_bf16(x32), x32.to(torch.bfloat16))
    lat = rnd(1, 4, 16, 16, dtype=torch.float32)
    w, b = rnd(64, 4, 3, 3, dtype=torch.float32, scale=0.2), rnd(64, dtype=torch.float32)
    y = ops.conv_in(lat, w, b, out_batch=2)
    ref = F.conv2d(lat, w, b, padding=1).permute(0, 2, 3, 1)
    assert rel(y[0], ref[0]) < TOL and torch.equal(y[0], y[1])
    y32 = ops.conv_in(lat, w, b, out_batch=2, out_dtype=torch.float32)
    assert y32.dtype == torch.float32 and rel(y32[1], ref[0]) < 1e-5
    h = rnd(2, 16, 16, 64)
    wo, bo = rnd(4, 64, 3, 3, dtype=torch.float32, scale=0.05), rnd(4, dtype=torch.float32)
    z = ops.conv_out(h, wo.permute(0, 2, 3, 1).contiguous(), bo)
    assert rel(z, F.conv2d(h.float().permute(0, 3, 1, 2), wo, bo, padding=1)) < 1e-4


@pytest.mark.parametrize("noise", [False, True])
@pytest.mark.parametrize("B", [1, 3])
def test_inpaint_blend(B, noise):
    """out = (1 - mask) (c_x orig + c_e noise) + mask latents, one mask per image broadcast over the channels"""
    lat, orig = rnd(B, 4, 40, 24, dtype=torch.float32, seed=1), rnd(B, 4, 40, 24, dtype=torch.float32, seed=2)
    nz = rnd(B, 4, 40, 24, dtype=torch.float32, seed=3) if noise else None
    mask = torch.rand(B, 1, 40, 24, generator=torch.Generator().manual_seed(4)).round().to(DEV)
    mask[:, :, :3] = 0.25                                     # soft-edged rows as well as hard 0 / 1
    out = ops.inpaint_blend(lat, orig, nz, mask, 0.8, 0.6)
    keep = 0.8 * orig.double() + (0.6 * nz.double() if noise else 0)
    ref = (1 - mask.double()) * keep + mask.double() * lat.double()
    assert ((out.double() - ref).abs() <= 1e-6 * (keep.abs() + lat.double().abs()) + 1e-7).all()
    if B > 1:                                                  # each image blends with its own mask
        assert not torch.equal(mask[0], mask[1])


@pytest.mark.parametrize("C", [3, 4, 8])
def test_conv_out_tc(C):
    """conv_out on the tensor cores: 3x3 conv with the C output channels zero-padded to 32, then the NHWC-prefix -> NCHW copy"""
    from instructany2pix_b200.packing import pack_conv_out
    B, H, W, Cin = 2, 24, 40, 128
    x = rnd(B, H, W, Cin)
    w, b = rnd(C, Cin, 3, 3, scale=(9 * Cin) ** -0.5, dtype=torch.float32), rnd(C, dtype=torch.float32)
    w32, b32 = pack_conv_out(w, b)
    out = ops.conv_out_tc(x, w32, b32, C)
    assert out.shape == (B, C, H, W) and out.dtype == torch.float32
    wq = w32[:C].reshape(C, 3, 3, Cin).permute(0, 3, 1, 2).double()          # the bf16 weights the kernel multiplies by
    xn = x.double().permute(0, 3, 1, 2)
    ref = F.conv2d(xn, wq, b.double(), padding=1)
    mag = F.conv2d(xn.abs(), wq.abs(), b.double().abs(), padding=1)
    assert ((out.double() - ref).abs() <= 9 * Cin * 2.0 ** -23 * mag + 1e-6).all()


@pytest.mark.parametrize("M,N,K,act_in,act", [(22, 3072, 1024, 0, 0), (28, 1024, 4096, 0, 1), (2, 1280, 320, 2, 0),
                                              (70, 1024, 512, 0, 2), (16, 8, 32, 0, 0)])
def test_gemm_smallm(M, N, K, act_in, act):
    a = rnd(M, K, dtype=torch.float32)
    w = rnd(N, K, scale=K ** -0.5)
    bias, res = rnd(N, dtype=torch.float32), rnd(M, N, dtype=torch.float32)
    out = ops.gemm_smallm(a, w, bias=bias, residual=res, act_in=act_in, act=act)
    ai = F.silu(a) if act_in == 2 else a
    h = ai @ w.float().t() + bias
    if act == 1:
        h = 0.5 * h * (1 + torch.tanh(math.sqrt(2 / math.pi) * (h + 0.044715 * h ** 3)))
    elif act == 2:
        h = F.silu(h)
    assert rel(out, h + res) < 2e-5      # hi/lo bf16 split of the fp32 activations: ~2^-16 relative


def test_causal_attn_small():
    B, T, heads = 2, 14, 16
    E = heads * 64
    qkv = rnd(B, T, 3 * E, dtype=torch.float32)
    out = ops.causal_attn_small(qkv, B, T, heads)
    q, k, v = [t.reshape(B, T, heads, 64).transpose(1, 2) for t in qkv.split(E, dim=2)]
    ref = F.scaled_dot_product_attention(q, k, v, is_causal=True).transpose(1, 2).reshape(B, T, E)
    assert rel(out, ref) < 1e-5
