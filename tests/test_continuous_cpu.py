"""Continuous batching (``B200ContinuousSampler``): the host logic -- slots, admission, per-slot schedules, completion -- against the
oracle run one request at a time, with the kernel test double extended by the two per-slot ops."""
import pytest
import torch

from instructany2pix_b200.attention_processor import B200IPAttnProcessor
from instructany2pix_b200.batcher import B200ContinuousSampler
from instructany2pix_b200.scheduler import B200DDIMScheduler, B200EulerDiscreteScheduler, B200LCMScheduler
from oracle import sampler as osampler
from oracle.attention import IPAttnProcessor2_0
from oracle.schedulers import DDIMSchedulerOracle, EulerDiscreteSchedulerOracle
from oracle.synth import synth_input
from oracle.unet import TINY
from tests.test_host_unet_emu import build_pair, make_inputs, rel

torch.set_grad_enabled(False)

L = 8


@pytest.fixture
def slotted(emu, monkeypatch):
    """the test double plus the per-slot ops as torch formulas; ``calls`` counts every op the engine reaches"""
    import instructany2pix_b200.ops as real

    def _col(t, x):
        assert t.dtype == torch.float32 and t.shape == (x.shape[0],)
        return t.reshape(-1, *([1] * (x.ndim - 1)))

    def cfg_step_coef_rows(eps2, x, g, c_x, c_e, s_in=None, x_out=None, x_in_next=None):
        eu, ec = eps2.float().chunk(2)
        v = (_col(c_x, x) * x.float() + _col(c_e, x) * (eu + _col(g, x) * (ec - eu))).to(x.dtype)
        if x_in_next is not None:
            x_in_next.copy_(_col(s_in, x) * v.float())
        x_out.copy_(v)
        return x_out

    def rowbias_gather(tables, coef_tables, step, blocks, rowbias, coef):
        S, rows, _ = tables.shape
        k = step.long().clamp(0, rows - 1)
        cur = tables[torch.arange(S), k]                                        # [S, 2 * sumC], per block [uncond; cond]
        rowbias.copy_(torch.cat([cur[:, 2 * lo:2 * hi].reshape(S, 2, hi - lo).transpose(0, 1).reshape(-1) for lo, hi in blocks]))
        coef.copy_(coef_tables[torch.arange(S), k].t())
        step.copy_(torch.where(step < rows - 1, step + 1, step))
        return rowbias

    def cross_attn(q, kv_text, n_text, kv_ip, n_ip, ip_scale, batch, n_q, heads, out=None):
        if isinstance(ip_scale, torch.Tensor):                            # per-row IP scales, as in test_mixed_requests_cpu
            assert ip_scale.dtype == torch.float32 and ip_scale.shape == (batch,)
            ip_scale = ip_scale.reshape(batch, 1, 1, 1)
        return emu.cross_attn(q, kv_text, n_text, kv_ip, n_ip, ip_scale, batch, n_q, heads, out=out)

    monkeypatch.setattr(real, "cross_attn", cross_attn)
    monkeypatch.setattr(real, "cfg_step_coef_rows", cfg_step_coef_rows)
    monkeypatch.setattr(real, "rowbias_gather", rowbias_gather)
    calls = []
    for name in [n for n in dir(emu) if not n.startswith("_") and callable(getattr(emu, n))] + ["cfg_step_coef_rows", "rowbias_gather"]:
        fn = getattr(real, name, None)
        if fn is not None and name not in ("IA2PError", "pdl", "require_cuda"):
            monkeypatch.setattr(real, name, lambda *a, _fn=fn, _n=name, **k: (calls.append(_n), _fn(*a, **k))[1])
    emu.calls = calls
    return emu


def _set_scale(unet, s):
    for p in unet.attn_processors.values():
        if isinstance(p, (B200IPAttnProcessor, IPAttnProcessor2_0)):
            p.scale = s


def _requests(n):
    lat, ctx, added = make_inputs(TINY, B=n, L=L)
    return [(lat[i:i + 1], ctx[[i, n + i]], {k: v[[i, n + i]] for k, v in added.items()}) for i in range(n)]


def _expected_schedule(sch, N, strength, img2img):
    sch.set_timesteps(N)
    ts = sch.timesteps
    if img2img:
        ts = ts[max(N - min(int(N * strength), N), 0):]
    out = []
    for i, t in enumerate(ts.tolist()):
        c_x, c_e = sch.coefficients(t)
        s_in = sch.input_scale(ts.tolist()[i + 1]) if hasattr(sch, "input_scale") and i + 1 < len(ts) else 1.0
        out.append((float(t), (c_x, c_e, s_in)))
    return out


@pytest.mark.parametrize("sched", ["ddim", "euler"])
def test_mixed_steps_match_each_request_alone(slotted, sched, monkeypatch):
    """steps {2, 3, 5}, different g / IP scales, one img2img request at strength 0.5, five requests on two slots, submitted at
    different steps: each request sees exactly its own timesteps and coefficients, and its final latents match the oracle alone"""
    o, b = build_pair(True)
    bs, make_os = (B200DDIMScheduler(), DDIMSchedulerOracle) if sched == "ddim" else (B200EulerDiscreteScheduler(), EulerDiscreteSchedulerOracle)
    reqs = _requests(5)
    init = synth_input("cont/init", (1, 4, L, L), seed=3) * 0.8
    spec = [dict(N=5, g=7.5, ip=0.3), dict(N=2, g=5.0, ip=1.0), dict(N=3, g=10.0, ip=None),
            dict(N=4, g=6.0, ip=0.0, init=init, strength=0.5), dict(N=2, g=9.0, ip=0.7)]
    when = [0, 0, 0, 1, 3]                                      # submitted before step `when`
    cs = B200ContinuousSampler(b, slots=2, latent_hw=(L, L), scheduler=bs, max_steps=5, n_text=77, n_ip=4, use_cuda_graph=False)
    s0 = b._ip_state()[1]

    seen = {}                                                   # rid -> [(rowbias of its two rows, coef column)]
    import instructany2pix_b200.ops as real
    inner = real.rowbias_gather

    def record(tables, coef_tables, step, blocks, rowbias, coef):
        out = inner(tables, coef_tables, step, blocks, rowbias, coef)
        S = tables.shape[0]
        for s, slot in enumerate(cs._slots):
            if slot is not None:
                rb = torch.cat([rowbias[2 * S * lo:2 * S * hi].view(2 * S, hi - lo)[[s, S + s]] for lo, hi in blocks], 1)
                seen.setdefault(slot["rid"], []).append((rb.clone(), coef[:, s].clone()))
        return out

    monkeypatch.setattr(real, "rowbias_gather", record)
    rids, results, step = {}, {}, 0
    while len(results) < len(spec):
        for i, w in enumerate(when):
            if w == step:
                r = spec[i]
                lat, ctx, added = reqs[i]
                rids[cs.submit(lat, ctx, added, num_inference_steps=r["N"], guidance_scale=r["g"], ip_scale=r["ip"],
                               init_latents=r.get("init"), strength=r.get("strength", 1.0))] = i
        results.update(cs.step())
        step += 1
        assert step < 30
    assert cs.useful_row_steps == sum(len(v) for v in seen.values()) and cs.executed_row_steps == 2 * step
    for rid, i in rids.items():
        r = spec[i]
        lat, ctx, added = reqs[i]
        sched_rows = _expected_schedule(type(bs)(), r["N"], r.get("strength", 1.0), "init" in r)
        assert len(seen[rid]) == len(sched_rows), rid
        table = b.time_rowbias_table(torch.tensor([t for t, _ in sched_rows]), added, 2)
        for k, ((rb, coef), (t, (c_x, c_e, s_in))) in enumerate(zip(seen[rid], sched_rows)):
            assert torch.equal(coef, torch.tensor([r["g"], c_x, c_e, s_in], dtype=torch.float32)), (rid, k)
            blocked = torch.cat([table[k][2 * lo:2 * hi].view(2, hi - lo) for lo, hi in b.prepare()["temb_slices"]], 1)
            assert torch.equal(rb, blocked), (rid, k)
        _set_scale(o, s0 if r["ip"] is None else r["ip"])
        ref = osampler.generate(o, lat, ctx, added, num_inference_steps=r["N"], guidance_scale=r["g"], scheduler=make_os(),
                                init_latents=r.get("init"), strength=r.get("strength", 1.0))
        e = rel(results[rid], ref)
        assert results[rid].shape == (1, 4, L, L) and e < 1.5e-2, (rid, e)
    _set_scale(o, s0)


def test_fifo_admission_result_order_and_idle_slots(slotted):
    o, b = build_pair(True)
    reqs = _requests(4)
    cs2 = B200ContinuousSampler(b, slots=2, latent_hw=(L, L), max_steps=4, use_cuda_graph=False)
    sub = lambda i, n: cs2.submit(*reqs[i], num_inference_steps=n)
    r0, r1, r2, r3 = sub(0, 1), sub(1, 3), sub(2, 2), sub(3, 1)        # FIFO: ids in submission order
    out = []
    for _ in range(3):
        out.append([rid for rid, _ in cs2.step()])
        out.append([s and s["rid"] for s in cs2._slots])
    # step 1: r0 (slot 0), r1 (slot 1) admitted, r0 done; step 2: r2 -> slot 0; step 3: r1 (slot 1) and r2 (slot 0) finish,
    # returned in admission order, not slot order
    assert out == [[r0], [None, r1], [], [r2, r1], [r1, r2], [None, None]]
    assert list(cs2._queue) and cs2._queue[0]["rid"] == r3
    done = dict(cs2.step())                                        # r3 -> slot 0 (first free slot)
    assert list(done) == [r3]
    final = done[r3]
    x1 = cs2._buf["x"][1].clone()                                  # slot 1 is idle and holds r1's final latents
    cs2.submit(*reqs[0], num_inference_steps=3)
    for _ in range(3):
        cs2.step()
        assert torch.equal(cs2._buf["x"][1], x1)                   # the idle slot's latents are bit-unchanged
    assert not torch.equal(cs2._buf["x"][0], final[0])
    assert cs2.pending() == 0 and cs2.drain() == {}


def test_argument_errors_before_any_kernel(slotted):
    from tests.test_host_unet_emu import nine_channel_case
    o, b = build_pair(True)
    lat, ctx, added = _requests(1)[0]
    init = torch.zeros(1, 4, L, L)
    with pytest.raises(NotImplementedError, match="LCM"):
        B200ContinuousSampler(b, latent_hw=(L, L), scheduler=B200LCMScheduler(), use_cuda_graph=False)
    with pytest.raises(NotImplementedError, match="9-channel"):
        B200ContinuousSampler(nine_channel_case()[1], latent_hw=(L, L), use_cuda_graph=False)
    cs = B200ContinuousSampler(b, slots=2, latent_hw=(L, L), max_steps=4, use_cuda_graph=False)
    sub = lambda **k: cs.submit(**{**dict(noise=lat, ctx=ctx, added_pair=added, num_inference_steps=2), **k})
    cases = [(NotImplementedError, "inpaint", dict(inpaint_mask=torch.ones(1, 1, L, L))),
             (ValueError, "max_steps", dict(num_inference_steps=5)),
             (ValueError, "max_steps", dict(num_inference_steps=0)),
             (ValueError, "no denoising step", dict(init_latents=init, strength=0.2)),
             (ValueError, "needs init_latents", dict(strength=0.5)),
             (ValueError, "noise", dict(noise=torch.zeros(1, 4, L, L + 1))),
             (ValueError, "noise", dict(noise=torch.zeros(2, 4, L, L))),
             (ValueError, "init_latents", dict(init_latents=torch.zeros(1, 4, 4, 4))),
             (ValueError, "ctx", dict(ctx=ctx[:, :77])),
             (ValueError, "ctx", dict(ctx=ctx[:1])),
             (ValueError, "added_pair", dict(added_pair={k: v[:1] for k, v in added.items()})),
             (ValueError, "guidance_scale", dict(guidance_scale=float("nan"))),
             (ValueError, "ip_scale", dict(ip_scale=float("inf")))]
    for exc, match, kw in cases:
        with pytest.raises(exc, match=match):
            sub(**kw)
    with pytest.raises(ValueError, match="n_ip"):                  # engine built for another number of IP tokens
        B200ContinuousSampler(b, latent_hw=(L, L), n_ip=16, use_cuda_graph=False).submit(lat, ctx, added, num_inference_steps=2)
    o0, b0 = build_pair(False)
    cs0 = B200ContinuousSampler(b0, latent_hw=(L, L), n_ip=0, use_cuda_graph=False)
    with pytest.raises(ValueError, match="IP-adapter"):
        cs0.submit(lat, ctx[:, :77], added, num_inference_steps=2, ip_scale=0.5)
    with pytest.raises(ValueError, match="ctx"):
        cs0.submit(lat, ctx, added, num_inference_steps=2)
    assert slotted.calls == [] and not cs._queue and cs._buf is None and not cs0._queue
    # a text-only UNet runs (n_ip = 0)
    assert list(cs0.drain()) == [] and cs0.submit(lat, ctx[:, :77], added, num_inference_steps=2) == 0
    assert list(cs0.drain()) == [0]


def test_one_state_for_the_engine_lifetime(slotted):
    o, b = build_pair(True)
    reqs = _requests(3)
    cs = B200ContinuousSampler(b, slots=2, latent_hw=(L, L), max_steps=3, use_cuda_graph=False)
    cs.submit(*reqs[0], num_inference_steps=2)
    cs.step()
    buf = cs._buf
    for wave in range(3):                                          # admission waves with new settings
        for i in range(3):
            cs.submit(*reqs[i], num_inference_steps=1 + (i + wave) % 3, guidance_scale=4.0 + wave + i, ip_scale=0.1 * (i + wave))
        assert len(cs.drain()) >= 3
        assert cs._buf is buf
    cs.submit(*reqs[0], num_inference_steps=3)
    cs.step()
    b.set_attn_processor(b.attn_processors)                        # new processors while a request is in flight
    with pytest.raises(RuntimeError, match="in flight"):
        cs.step()
    cs._slots = [None] * cs.S                                      # nothing in flight: the engine rebuilds for the new UNet
    cs.submit(*reqs[1], num_inference_steps=2)
    assert len(cs.drain()) == 1 and cs._buf is not buf
