"""sample_long (long audio in overlapping windows, sampled as one batch and blended after every step): the fdm_window_blend
and fdm_ddpm_step_keyed kernels against torch restatements, one window against sample / ddim_sample, several windows
against an eager restatement from public pieces, and the invariances the feature must keep (graph = eager, cached graphs,
fan-out, sharding, the high-precision tail, quant / decode)."""
import pytest
import torch

from helpers import N_SAMPLES, build_product

pytestmark = pytest.mark.gpu
STEPS = [999, 998, 1, 0]
WIN = {"vocaset": (90, 30), "mead": (90, 30), "biwi": (75, 25)}  # (window, overlap): stride a multiple of the period


def _samples(P, T):
    r = 2 if P.pair_audio else 1
    return 320 * (T * r - 1) + 400  # exactly T frames


def _setup(preset, dev, precision="fp32", T=None, n_audio=1, k=1, guided=False):
    from oracle.weights import synthetic_audio
    from utiles.classifierfree import ClassifierFreeSampleModel
    fdm, ae, diff = build_product(preset, device=dev)
    fdm.set_precision(precision)
    ae.set_precision(precision)
    P = fdm.preset
    B = n_audio * k
    n = N_SAMPLES if T is None else _samples(P, T)
    audio = torch.stack([synthetic_audio(c, n) for c in range(n_audio)]).to(dev)
    if T is None:
        T = fdm.encode_audio(audio).shape[1] // (2 if P.pair_audio else 1)
    idh = torch.eye(P.n_id)[[b % P.n_id for b in range(B)]].to(dev)
    emo = torch.eye(7)[[(3 + b) % 7 for b in range(B)]].to(dev) if P.emotion else None
    diff.noise_source, diff.seed = "philox", 11
    if guided:
        diff.denoise_fn = ClassifierFreeSampleModel(fdm, level=2.5)
    conds = (emo, idh) if P.emotion else (idh,)
    return fdm, ae, diff, audio, conds, (B, T * P.fq, P.zdim)


def _blend(x, plan, d):
    """torch restatement of fdm_window_blend on (A*n_w*K, ...) fp32 windows (a new tensor)."""
    v = x.clone().view(plan.A, plan.n_w, plan.K, plan.W, d)
    lam = plan.weights().to(x.device)[:, None]
    o = (1 - lam) * v[:, :-1, :, plan.S:] + lam * v[:, 1:, :, :plan.O]
    v[:, :-1, :, plan.S:] = o
    v[:, 1:, :, :plan.O] = o
    return v.view(x.shape)


def _overlaps_equal(raw, plan, d):
    v = raw.view(plan.A, plan.n_w, plan.K, plan.W, d)
    return torch.equal(v[:, :-1, :, plan.S:], v[:, 1:, :, :plan.O])


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("d", [512, 1024])
def test_blend_kernel_matches_torch(cuda_dev, K, d):
    from fdm_b200 import lib
    from fdm_b200.windows import WindowPlan
    plan = WindowPlan(A=2, K=K, T=30, W=12, O=4, r=1)
    assert plan.n_w == 4
    g = torch.Generator().manual_seed(d + K)
    x0 = torch.randn(plan.n_seq, plan.W, d, generator=g).to(cuda_dev)
    xb0 = torch.randn(plan.n_seq, plan.W, d, generator=g).to(cuda_dev, torch.bfloat16)
    x, xb = x0.clone(), xb0.clone()
    lam = plan.weights().to(cuda_dev)
    lib.window_blend(x, lam, plan.A, plan.n_w, plan.K, plan.S, x_bf16=xb)
    want = _blend(x0, plan, d)
    assert torch.equal(x, want), (x - want).abs().max().item()
    touched = torch.zeros(plan.A, plan.n_w, plan.K, plan.W, dtype=torch.bool)
    touched[:, :-1, :, plan.S:] = True
    touched[:, 1:, :, :plan.O] = True
    touched = touched.view(plan.n_seq, plan.W, 1).to(cuda_dev)
    assert torch.equal(x0[~touched.expand_as(x0)], x[~touched.expand_as(x)])  # rows outside overlaps untouched
    assert torch.equal(xb, torch.where(touched, lib.cast(want, torch.empty_like(xb)), xb0))
    assert _overlaps_equal(x, plan, d)
    one = WindowPlan(A=2, K=K, T=12, W=12, O=4, r=1)  # one window: nothing is launched
    n0 = lib.launch_count
    y = x0[:one.n_seq].clone()
    lib.window_blend(y, lam, one.A, one.n_w, one.K, one.S)
    assert lib.launch_count == n0 and torch.equal(y, x0[:one.n_seq])


def test_keyed_step(cuda_dev):
    from fdm_b200 import lib
    G, n_w, W, S, d, clip0, seed, t = 2, 3, 8, 5, 64, 7, 2 ** 41 + 5, 321
    B = G * n_w
    g = torch.Generator().manual_seed(3)
    x0, xu, xt = (torch.randn(B, W * d, generator=g).to(cuda_dev) for _ in range(3))
    c1, c2, sg = (torch.rand(1000, generator=g).to(cuda_dev) for _ in range(3))
    t_dev = torch.tensor([t], dtype=torch.int32, device=cuda_dev)
    kw = dict(x0_uncond=xu, guidance=2.5, t_dev=t_dev, seed=seed, clip_index0=clip0)
    plain = lib.ddpm_step(x0, xt, torch.empty_like(xt), c1, c2, sg, **kw)
    nulls = lib.ddpm_step(x0, xt, torch.empty_like(xt), c1, c2, sg, noise_keys=(None, None), **kw)
    assert torch.equal(plain, nulls)
    # keyed: window w of long sequence g draws at (clip0 + g, element offset w*S*d/4) -> rows [w*S, w*S + W) of the full draw
    clip = torch.tensor([clip0 + b // n_w for b in range(B)], dtype=torch.int64, device=cuda_dev)
    e4 = torch.tensor([(b % n_w) * S * d // 4 for b in range(B)], dtype=torch.int64, device=cuda_dev)
    zero, one = torch.zeros(1000, device=cuda_dev), torch.ones(1000, device=cuda_dev)
    out = lib.ddpm_step(x0, xt, torch.empty_like(xt), zero, zero, one, t_dev=t_dev, seed=seed, noise_keys=(clip, e4))
    full = lib.philox_normal(torch.empty(G, ((n_w - 1) * S + W) * d, device=cuda_dev), seed, clip0, t)
    for b in range(B):
        w = b % n_w
        assert torch.equal(out[b], full[b // n_w, w * S * d:(w * S + W) * d]), b
    with pytest.raises(lib.FdmError, match="both key arrays"):
        lib.ddpm_step(x0, xt, torch.empty_like(xt), c1, c2, sg, t_dev=t_dev, noise_keys=(clip, None))


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("preset", ["vocaset", "mead"])
@pytest.mark.parametrize("guided", [False, True])
def test_one_window_is_sample(cuda_dev, preset, guided):
    """T <= window: the call is sample() / ddim_sample() of the same arguments, bit for bit (bf16 with the tail)."""
    fdm, ae, diff, audio, conds, shape = _setup(preset, cuda_dev, "bf16", n_audio=2, guided=guided)
    assert shape[1] // fdm.preset.fq <= 14 * fdm.preset.period
    assert torch.equal(diff.sample_long(audio, shape, *conds, steps=STEPS), diff.sample(audio, shape, *conds, steps=STEPS))
    assert torch.equal(diff.sample_long(audio, shape, *conds, ddim_steps=4), diff.ddim_sample(audio, shape, *conds, 4))
    x_T = torch.randn(shape, generator=torch.Generator().manual_seed(1)).to(cuda_dev)
    assert torch.equal(diff.sample_long(audio, shape, *conds, step_range=(4, 0), x_T=x_T),
                       diff.sample(audio, shape, *conds, step_range=(4, 0), x_T=x_T))


def _restated(diff, plan, audio, conds, x_T, steps, d):
    """Eager restatement from public pieces: p_sample (FDM.forward + the DDPM update) on the window batch with the
    full-length Philox draw gathered into windows, the blend in torch, then the assembly."""
    from fdm_b200 import lib
    B, L, z = x_T.shape
    fq = L // plan.T
    full = torch.zeros(B, plan.T_pad * fq, z, device=x_T.device)
    full[:, :L] = x_T
    x = plan.gather(full)
    audio_w = plan.window_audio(audio)
    conds_w = tuple(plan.repeat_rows(c) for c in conds)
    raws = []
    for t in steps:
        zf = lib.philox_normal(torch.empty_like(full), diff.seed, diff.clip_index0, t)
        x = diff.p_sample(x, torch.full((1,), t, dtype=torch.long, device=x.device), audio_w, *conds_w, noise=plan.gather(zf))
        x = _blend(x, plan, d)
        raws.append(x)
    return plan.assemble(x), raws


@pytest.mark.parametrize("preset, n_w, guided", [("vocaset", 2, False), ("vocaset", 3, True), ("mead", 3, True),
                                                 ("biwi", 2, True)])
def test_windows_equal_eager_restatement(cuda_dev, preset, n_w, guided):
    from fdm_b200.windows import plan_windows
    W, O = WIN[preset]
    T = W + (n_w - 2) * (W - O) + 7
    fdm, ae, diff, audio, conds, shape = _setup(preset, cuda_dev, "fp32", T=T, n_audio=2, guided=guided)
    P = fdm.preset
    plan = plan_windows(P, shape, audio.shape[0], audio.shape[1], W, O)
    assert plan.n_w == n_w
    diff.clip_index0 = 3
    x_T = torch.randn(shape, generator=torch.Generator().manual_seed(2)).to(cuda_dev)
    got = diff.sample_long(audio, shape, *conds, window=W, overlap=O, steps=STEPS, x_T=x_T)
    want, raws = _restated(diff, plan, audio, conds, x_T, STEPS, P.d)
    assert got.shape == shape
    assert (got - want).abs().max().item() <= 1e-5
    for i in range(1, len(STEPS) + 1):  # the raw window state after every step: overlap rows bit-identical
        raw = diff._sample_windows(plan, audio, conds, None, STEPS[:i], None, x_T)
        assert _overlaps_equal(raw, plan, P.d), i
        assert (raw - raws[i - 1]).abs().max().item() <= 1e-5, i


def test_default_draw_and_ddim(cuda_dev):
    """Without x_T the start is the full-length draw sample() makes (Philox at clip_index0 + sequence); DDIM windows blend
    too (overlaps identical) and a different seed changes the DDPM result."""
    from fdm_b200 import lib
    from fdm_b200.windows import plan_windows
    W, O = WIN["vocaset"]
    fdm, ae, diff, audio, conds, shape = _setup("vocaset", cuda_dev, "fp32", T=2 * W, n_audio=2, guided=True)
    P = fdm.preset
    plan = plan_windows(P, shape, 2, audio.shape[1], W, O)
    full = lib.philox_normal(torch.empty(shape[0], plan.T_pad * P.fq, P.zdim, device=cuda_dev), 11, 0, 1000)
    assert torch.equal(diff.sample_long(audio, shape, *conds, window=W, overlap=O, steps=STEPS),
                       diff.sample_long(audio, shape, *conds, window=W, overlap=O, steps=STEPS, x_T=full[:, :shape[1]]))
    raw = diff._sample_windows(plan, audio, conds, 5, None, None, None)
    assert _overlaps_equal(raw, plan, P.d)
    assert torch.equal(plan.assemble(raw), diff.sample_long(audio, shape, *conds, window=W, overlap=O, ddim_steps=5))


def test_graph_equals_eager_and_reuses_graphs(cuda_dev):
    W, O = WIN["vocaset"]
    fdm, ae, diff, audio, conds, shape = _setup("vocaset", cuda_dev, "bf16", T=2 * W, n_audio=2, guided=True)
    kw = dict(window=W, overlap=O)
    for call in (lambda a: diff.sample_long(a, shape, *conds, steps=STEPS, **kw),
                 lambda a: diff.sample_long(a, shape, *conds, ddim_steps=4, **kw)):
        got = call(audio)
        diff.use_cuda_graph = False
        eager = call(audio)
        diff.use_cuda_graph = True
        assert torch.equal(got, eager)
    ddpm = lambda a: diff.sample_long(a, shape, *conds, steps=STEPS, **kw)  # noqa: E731
    first = ddpm(audio)
    graphs = set(fdm.engine().graph_cache)
    n = len(graphs)
    assert torch.equal(ddpm(audio), first)
    assert set(fdm.engine().graph_cache) == graphs
    assert torch.equal(ddpm(audio.clone()), first)  # a new audio tensor of the same shape: same graphs
    assert len(fdm.engine().graph_cache) == n and set(fdm.engine().graph_cache) == graphs


def test_bf16_tail_steps_blend(cuda_dev):
    """bf16 with hi_tail_steps = 1 (the last step runs eagerly on the high-precision engine): overlaps identical at the end."""
    from fdm_b200.windows import plan_windows
    W, O = WIN["mead"]
    fdm, ae, diff, audio, conds, shape = _setup("mead", cuda_dev, "bf16", T=2 * W + 11, n_audio=2, guided=True)
    assert fdm.hi_tail_steps == 1
    plan = plan_windows(fdm.preset, shape, 2, audio.shape[1], W, O)
    for ddim in (None, 4):
        raw = diff._sample_windows(plan, audio, conds, ddim, None if ddim else STEPS, None, None)
        assert _overlaps_equal(raw, plan, fdm.preset.d), ddim


def test_fanout_and_sharding(cuda_dev):
    W, O = WIN["vocaset"]
    K = 2
    fdm, ae, diff, audio, conds, shape = _setup("vocaset", cuda_dev, "bf16", T=2 * W + 5, n_audio=2, k=K, guided=True)
    kw = dict(window=W, overlap=O, steps=STEPS)
    full = diff.sample_long(audio, shape, *conds, **kw)
    assert torch.equal(full, diff.sample_long(audio.repeat_interleave(K, 0), shape, *conds, **kw))
    parts = []
    for a0 in (0, 1):  # fanout_shard_range over 2 ranks: one clip, its K sequences, clip_index0 = a0 * K
        s0 = a0 * K
        diff.clip_index0 = s0
        parts.append(diff.sample_long(audio[a0:a0 + 1], (K,) + shape[1:], *(c[s0:s0 + K] for c in conds), **kw))
    diff.clip_index0 = 0
    assert torch.equal(torch.cat(parts), full)


def test_long_latent_through_quant_and_decode(cuda_dev):
    W, O = WIN["vocaset"]
    S = W - O
    T = W + S + S // 2  # 2.5 windows
    fdm, ae, diff, audio, conds, shape = _setup("vocaset", cuda_dev, "bf16", T=T, n_audio=1, guided=True)
    lat = diff.sample_long(audio, shape, *conds, window=W, overlap=O, steps=STEPS)
    assert lat.shape == shape and lat.dtype == torch.float32 and torch.isfinite(lat).all()
    zq, _, (_, _, idx) = ae.quant(lat)
    v = ae.decode(zq)
    assert v.shape == (1, T, ae.args.in_dim) and torch.isfinite(v).all()
