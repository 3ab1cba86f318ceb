"""Continuous batching on the B200: the per-slot entry points (ia2p_cfg_step_coef_rows, ia2p_rowbias_gather) against fp32 torch and
bit for bit against the scalar kernels, and ``B200ContinuousSampler`` -- neighbour independence, parity with the oracle run one
request at a time, one capture for the engine's lifetime, no host synchronisation in ``step``.  Every allocation ``ops`` and the
engine make with ``torch.empty`` comes back poisoned (NaN), so anything a kernel leaves unwritten fails a comparison."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from instructany2pix_b200 import ops  # noqa: E402
from instructany2pix_b200.attention_processor import B200IPAttnProcessor  # noqa: E402
from instructany2pix_b200.batcher import B200ContinuousSampler  # noqa: E402
from instructany2pix_b200.sampler import B200Sampler  # noqa: E402
from instructany2pix_b200.scheduler import B200DDIMScheduler, B200EulerDiscreteScheduler  # noqa: E402
from oracle import sampler as osampler  # noqa: E402
from oracle.attention import IPAttnProcessor2_0  # noqa: E402
from oracle.schedulers import DDIMSchedulerOracle, EulerDiscreteSchedulerOracle  # noqa: E402
from oracle.synth import synth_input  # noqa: E402
from oracle.unet import TINY  # noqa: E402
from tests._poison import poisoned  # noqa: E402
from tests.test_host_unet_emu import build_pair, make_inputs  # noqa: E402
from tests.test_unet_parity_gpu import sdxl_pair  # noqa: E402,F401  (module fixture: the SDXL-width oracle + B200 pair)

torch.set_grad_enabled(False)
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False
DEV = "cuda"
TOL = 4e-3          # kernel gate: bf16 output rounding over an fp32 reference
FREE = 5e-2         # free-running final latents against the oracle, as test_unet_parity_gpu.py gates them


def _alone(b, sched, r, kw):
    """the same request alone through B200Sampler.generate: the engine gives exactly these latents"""
    kw = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in kw.items()}
    return B200Sampler(b, scheduler=sched).generate(r[0].cuda(), r[1].cuda(), {k: v.cuda() for k, v in r[2].items()}, **kw)


def _check(tag, got, ref, alone):
    e, e_alone, e_gen = rel(got, ref), rel(alone, ref), rel(got, alone)
    print(f"{tag}: final latent rel-L2 vs oracle {e:.2e} (generate alone {e_alone:.2e}; engine vs generate {e_gen:.2e})")
    assert e < FREE and torch.equal(got, alone), (tag, e, e_alone, e_gen)


@pytest.fixture(autouse=True)
def _poisoned():
    with poisoned():
        yield


def rnd(*shape, seed, dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g).to(dtype).to(DEV)


def rel(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-12)).item()


def bits(t):
    return t.contiguous().view({2: torch.int16, 4: torch.int32}[t.element_size()])


def same_bits(a, b):
    return torch.equal(bits(a), bits(b))


def _set_scale(unet, s):
    for p in unet.attn_processors.values():
        if isinstance(p, (B200IPAttnProcessor, IPAttnProcessor2_0)):
            p.scale = s


# ------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("shape,dt", [((4, 4, 16, 16), torch.float32), ((3, 4, 5, 5), torch.float32),
                                      ((4, 4, 128, 128), torch.float32), ((3, 4, 16, 16), torch.bfloat16),
                                      ((2, 4, 5, 5), torch.bfloat16)])
def test_cfg_step_coef_rows(shape, dt):
    """vectorised (n % 8 == 0) and ragged (n = 100) paths, fp32 and bf16 latents; the last row is an idle slot (identity)"""
    B = shape[0]
    eps2, x = rnd(2 * B, *shape[1:], seed=4, dtype=dt), rnd(*shape, seed=5, dtype=dt)
    g = torch.tensor([5.0, 7.5, 12.0, 9.0][:B - 1] + [0.0], device=DEV)
    cx = torch.tensor([0.98, 1.0, 1.07, 0.91][:B - 1] + [1.0], device=DEV)
    ce = torch.tensor([-0.11, -0.62, 0.05, -1.3][:B - 1] + [0.0], device=DEV)
    s_in = torch.tensor([0.07, 0.31, 0.99, 0.5][:B - 1] + [1.0], device=DEV)
    nxt = torch.empty(shape, device=DEV, dtype=torch.float32)
    out = ops.cfg_step_coef_rows(eps2, x, g, cx, ce, s_in=s_in, x_in_next=nxt)
    col = lambda t: t.reshape(B, 1, 1, 1)
    eu, ec = eps2.float().chunk(2)
    ref = col(cx) * x.float() + col(ce) * (eu + col(g) * (ec - eu))
    assert rel(out, ref) < (1e-6 if dt == torch.float32 else TOL)
    for b in range(B):              # row b: the scalar kernel at that row's values; the next input: axpby at that row's scale
        one = ops.cfg_ddim_step(eps2, x, float(g[b]), float(cx[b]), float(ce[b]))
        assert same_bits(out[b], one[b]), b
        assert same_bits(nxt[b], ops.axpby(out.float(), out.float(), float(s_in[b]), 0.0)[b]), b
    assert same_bits(out[B - 1], x[B - 1])                     # identity coefficients: the idle row is bit-unchanged
    alone = ops.cfg_step_coef_rows(eps2, x, g, cx, ce)         # without the next input: same x_out
    assert same_bits(alone, out)


@pytest.mark.parametrize("S", [1, 3, 4])
def test_rowbias_gather(S):
    """bitwise torch indexing of the per-slot tables, sentinel rows included, with the counters advancing across graph replays"""
    blocks = [(0, 32), (32, 96), (96, 104), (104, 424)]
    sum_c, R = blocks[-1][1], 6
    tables = rnd(S, R, 2 * sum_c, seed=11)
    tables[:, R - 1] = 0.0                                      # the sentinel row
    coef_tables = rnd(S, R, 4, seed=12)
    coef_tables[:, R - 1] = torch.tensor([0.0, 1.0, 0.0, 1.0], device=DEV)
    start = [R - 1 - 3 * (s % 2) - s // 2 for s in range(S)]    # slot 0 starts on the sentinel, the others on request rows
    step = torch.tensor(start, device=DEV, dtype=torch.int32)
    rb = torch.empty(2 * S * sum_c, device=DEV)
    coef = torch.empty(4, S, device=DEV)

    def want(k):
        cur = tables[torch.arange(S), k]
        rows = torch.cat([cur[:, 2 * lo:2 * hi].reshape(S, 2, hi - lo).transpose(0, 1).reshape(-1) for lo, hi in blocks])
        return rows, coef_tables[torch.arange(S), k].t()

    k = torch.tensor(start)
    ops.rowbias_gather(tables, coef_tables, step, blocks, rb, coef)          # eager call
    w_rb, w_coef = want(k)
    assert same_bits(rb, w_rb) and same_bits(coef, w_coef)
    k = torch.clamp(k + 1, max=R - 1)
    assert step.cpu().tolist() == k.tolist()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        ops.rowbias_gather(tables, coef_tables, step, blocks, rb, coef)
    assert step.cpu().tolist() == k.tolist()                                 # capture runs nothing
    for _ in range(R + 1):                                                   # past the end: every slot stays on the sentinel
        g.replay()
        w_rb, w_coef = want(k)
        assert same_bits(rb, w_rb) and same_bits(coef, w_coef)
        k = torch.clamp(k + 1, max=R - 1)
        assert step.cpu().tolist() == k.tolist()
    assert (rb == 0).all() and coef.cpu().tolist() == [[0.0] * S, [1.0] * S, [0.0] * S, [1.0] * S]


# ------------------------------------------------------------------------------------------------ engine
def _requests(n, L):
    lat, ctx, added = make_inputs(TINY, B=n, L=L)
    return [(lat[i:i + 1], ctx[[i, n + i]], {k: v[[i, n + i]] for k, v in added.items()}) for i in range(n)]


def _run(cs, plan):
    """plan: [(submit before step, kwargs)] -> {index in plan: final latents}"""
    rid_of, out, step = {}, {}, 0
    while len(out) < len(plan):
        for i, (w, kw) in enumerate(plan):
            if w == step:
                rid_of[cs.submit(**kw)] = i
        out.update({rid_of[r]: x for r, x in cs.step()})
        step += 1
        assert step < 100
    return out


def test_neighbour_independence():
    """64x64 latent: every level's map is whole 128-row tiles per image, so a request's final latents in slot 0 of a 3-slot engine
    are bit-identical whether its neighbours idle, run other requests (other steps, strengths, g, IP scales), or were admitted
    before, together with or after it"""
    o, b = build_pair(True, device=DEV)
    L = 64
    reqs = _requests(4, L)
    init = synth_input("cont/init64", (1, 4, L, L), seed=3) * 0.8
    mk = lambda i, **kw: dict(noise=reqs[i][0], ctx=reqs[i][1], added_pair=reqs[i][2], **kw)
    A = mk(0, num_inference_steps=4, guidance_scale=7.5, ip_scale=0.6)
    n1 = mk(1, num_inference_steps=3, guidance_scale=12.0, ip_scale=1.0)
    n2 = mk(2, num_inference_steps=5, guidance_scale=4.0, ip_scale=0.0, init_latents=init, strength=0.6)
    x1 = mk(3, num_inference_steps=1, guidance_scale=9.0, ip_scale=0.3)
    engine = lambda: B200ContinuousSampler(b, slots=3, latent_hw=(L, L), max_steps=5)
    alone = _run(engine(), [(0, A)])[0]
    cases = {"together": [(0, A), (0, n1), (0, n2)],
             "before": [(0, A), (1, n1), (2, n2)],
             "after": [(0, x1), (0, n1), (0, n2), (1, A)]}              # x1 frees slot 0 while n1 / n2 are mid-trajectory
    for name, plan in cases.items():
        got = _run(engine(), plan)
        ia = [i for i, (_, kw) in enumerate(plan) if kw is A][0]
        assert same_bits(got[ia], alone), name
    assert torch.isfinite(alone).all()


@pytest.mark.parametrize("sched", ["ddim", "euler"])
@pytest.mark.parametrize("L", [32, 64])
def test_mixed_engine_against_oracle(sched, L):
    """TINY, three slots, five requests with steps {2, 3, 4}, img2img strengths, different g / IP scales, staggered arrivals: each
    request's free-running final latents against the fp32 oracle running it alone, and bitwise equal to ``B200Sampler.generate``
    running it alone (DESIGN section 5's 1e-2 is the teacher-forced per-step gate; the free-running latents of these 2-4 step
    trajectories sit at 0.8-1.3e-2 from the oracle on both paths)"""
    o, b = build_pair(True, device=DEV)
    bs, os_ = (B200DDIMScheduler, DDIMSchedulerOracle) if sched == "ddim" else (B200EulerDiscreteScheduler, EulerDiscreteSchedulerOracle)
    reqs = _requests(5, L)
    init = synth_input(f"cont/init{L}", (1, 4, L, L), seed=3) * 0.8
    spec = [dict(num_inference_steps=4, guidance_scale=7.5, ip_scale=0.3),
            dict(num_inference_steps=2, guidance_scale=5.0, ip_scale=1.0),
            dict(num_inference_steps=4, guidance_scale=6.0, ip_scale=0.0, init_latents=init, strength=0.5),
            dict(num_inference_steps=3, guidance_scale=9.0, ip_scale=0.7),
            dict(num_inference_steps=4, guidance_scale=8.0, ip_scale=0.5, init_latents=init, strength=0.75)]
    when = [0, 0, 1, 2, 2]
    plan = [(w, dict(noise=r[0].cuda(), ctx=r[1].cuda(), added_pair={k: v.cuda() for k, v in r[2].items()},
                     **{k: (v.cuda() if torch.is_tensor(v) else v) for k, v in kw.items()})) for w, r, kw in zip(when, reqs, spec)]
    got = _run(B200ContinuousSampler(b, slots=3, latent_hw=(L, L), scheduler=bs(), max_steps=4), plan)
    s0 = o.attn_processors[[k for k in o.attn_processors if "attn2" in k][0]].scale
    for i, (r, kw) in enumerate(zip(reqs, spec)):
        _set_scale(o, kw["ip_scale"])
        ref = osampler.generate(o, r[0], r[1], r[2], num_inference_steps=kw["num_inference_steps"], guidance_scale=kw["guidance_scale"],
                                scheduler=os_(), init_latents=kw.get("init_latents"), strength=kw.get("strength", 1.0))
        _check(f"{sched} {L}x{L} request {i} ({kw['num_inference_steps']} steps, strength {kw.get('strength', 1.0)}, "
               f"g {kw['guidance_scale']}, IP {kw['ip_scale']})", got[i], ref, _alone(b, bs(), r, kw))
    _set_scale(o, s0)


def test_sdxl_width_two_requests_against_oracle(sdxl_pair):
    """the real SDXL-base configuration at a 32x32 latent: requests with 2 and 3 steps and different g / IP scales, admitted one
    step apart into a two-slot engine, against the fp32 oracle running each alone and bitwise against ``generate`` alone"""
    o, b = sdxl_pair
    L = 32
    reqs = []
    for i in range(2):
        ctx = synth_input(f"cont/sdxl/ctx{i}", (2, 81, 2048))
        added = dict(text_embeds=synth_input(f"cont/sdxl/pooled{i}", (2, 1280)),
                     time_ids=torch.tensor([[256.0, 256.0, 0.0, 0.0, 256.0, 256.0]] * 2))
        reqs.append((synth_input(f"cont/sdxl/lat{i}", (1, 4, L, L)), ctx, added))
    spec = [dict(num_inference_steps=2, guidance_scale=5.0, ip_scale=0.3), dict(num_inference_steps=3, guidance_scale=12.0, ip_scale=1.0)]
    plan = [(i, dict(noise=r[0].cuda(), ctx=r[1].cuda(), added_pair={k: v.cuda() for k, v in r[2].items()}, **kw))
            for i, (r, kw) in enumerate(zip(reqs, spec))]
    got = _run(B200ContinuousSampler(b, slots=2, latent_hw=(L, L), max_steps=3, n_text=77, n_ip=4), plan)
    for i, (r, kw) in enumerate(zip(reqs, spec)):
        _set_scale(o, kw["ip_scale"])
        ref = osampler.generate(o, r[0], r[1], r[2], num_inference_steps=kw["num_inference_steps"], guidance_scale=kw["guidance_scale"])
        _check(f"SDXL width, request {i} ({kw['num_inference_steps']} steps, g {kw['guidance_scale']}, IP {kw['ip_scale']})",
               got[i], ref, _alone(b, B200DDIMScheduler(), r, kw))
    _set_scale(o, 1.0)


def test_one_capture_and_no_synchronisation():
    """three admission waves with new settings on one captured graph; once it is captured, no step -- admitting, completing or
    neither -- synchronises with the device (the capturing step is excluded: torch.cuda.graph synchronises on entry)"""
    o, b = build_pair(True, device=DEV)
    L = 32
    reqs = _requests(4, L)
    init = synth_input("cont/init32", (1, 4, L, L), seed=3) * 0.8
    cs = B200ContinuousSampler(b, slots=2, latent_hw=(L, L), scheduler=B200EulerDiscreteScheduler(), max_steps=4)
    cs.submit(*reqs[0], num_inference_steps=2)
    cs.step()                                                   # capture
    graph = cs._buf["graph"]
    results = {}
    torch.cuda.set_sync_debug_mode("error")
    try:
        for wave in range(3):
            for i in range(3):
                r = reqs[(i + wave) % 4]
                kw = dict(init_latents=init, strength=0.5) if i == 1 else {}
                cs.submit(r[0], r[1], r[2], num_inference_steps=2 + (i + wave) % 3, guidance_scale=5.0 + wave + i,
                          ip_scale=0.2 * (i + 1), **kw)
            while cs.pending():
                results.update(cs.step())
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert cs.captures == 1 and cs._buf["graph"] is graph and len(results) == 10
    assert all(torch.isfinite(v).all() for v in results.values())
