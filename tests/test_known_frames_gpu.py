"""Known frames (latent inpainting and continuation) in p_sample_loop / ddim_sample: the fdm_known_frames kernel against a
torch restatement, the sampling calls against eager restatements of the replacement rule, and the invariances the
feature must keep (no known frames = today's result, graph = eager, fan-out, sharding, continuation)."""
import pytest
import torch

from helpers import N_SAMPLES, build_product

pytestmark = pytest.mark.gpu
PRESETS = ["vocaset", "mead", "biwi"]
STEPS = [999, 998, 1, 0]


def _setup(preset, dev, precision="fp32", n_audio=2, k=1, guided=False):
    from oracle.weights import synthetic_audio
    from utiles.classifierfree import ClassifierFreeSampleModel
    fdm, ae, diff = build_product(preset, device=dev)
    fdm.set_precision(precision)
    ae.set_precision(precision)
    P = fdm.preset
    B = n_audio * k
    audio = torch.stack([synthetic_audio(c, N_SAMPLES) for c in range(n_audio)]).to(dev)
    idh = torch.eye(P.n_id)[[b % P.n_id for b in range(B)]].to(dev)
    emo = torch.eye(7)[[(3 + b) % 7 for b in range(B)]].to(dev) if P.emotion else None
    T = fdm.encode_audio(audio).shape[1] // (2 if P.pair_audio else 1)
    diff.noise_source, diff.seed = "philox", 11
    if guided:
        diff.denoise_fn = ClassifierFreeSampleModel(fdm, level=2.5)
    conds = (emo, idh) if P.emotion else (idh,)
    return fdm, ae, diff, audio, conds, (B, T * P.fq, P.zdim)


def _known(shape, fq, dev, seed=5, frac=0.5):
    g = torch.Generator().manual_seed(seed)
    B, L, z = shape
    known = torch.randn(shape, generator=g).to(dev)
    mask = (torch.rand(B, L // fq, generator=g) < frac).to(dev)
    mask[0, 0] = True
    return known, mask


def _rows(mask, fq, z):
    """(B, T) frame mask -> (B, fq*T, z) element mask."""
    return mask.repeat_interleave(fq, 1)[:, :, None].expand(-1, -1, z)


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mask_kind", ["random", "none", "all"])
@pytest.mark.parametrize("d", [64, 1024])
def test_kernel_matches_torch(cuda_dev, mask_kind, d):
    from fdm_b200 import lib
    B, T, clip0, seed, t = 3, 7, 4, 2 ** 40 + 3, 321
    g = torch.Generator().manual_seed(d)
    x0 = torch.randn(B, T * d, generator=g).to(cuda_dev)
    known = torch.randn(B, T * d, generator=g).to(cuda_dev)
    noise = torch.randn(B, T * d, generator=g).to(cuda_dev)
    m = {"random": torch.rand(B, T, generator=g) < 0.4, "none": torch.zeros(B, T, dtype=torch.bool),
         "all": torch.ones(B, T, dtype=torch.bool)}[mask_kind].to(cuda_dev)
    mel = m.repeat_interleave(d, 1)
    mask = m.to(torch.uint8).reshape(-1).contiguous()
    ka = torch.rand(4, generator=g).to(cuda_dev)
    kb = torch.tensor([0.3, 0.7, 0.0, 0.9]).to(cuda_dev)
    index = torch.tensor([2], dtype=torch.int32, device=cuda_dev)
    seed_dev = torch.tensor([seed], dtype=torch.int64, device=cuda_dev)
    t_dev = torch.tensor([t], dtype=torch.int32, device=cuda_dev)
    z_philox = lib.philox_normal(torch.empty_like(x0), seed, clip0, t)
    for mode, offset, z in (("buffer", 1, noise), ("alias", 1, x0), ("philox", 1, z_philox), ("kb0", 0, None)):
        i = 2 + offset
        x = x0.clone()
        xb0 = torch.randn(B, T * d, generator=g).to(cuda_dev, torch.bfloat16)
        xb = xb0.clone()
        lib.known_frames(x, known, mask, ka, kb, index, offset=offset, noise={"buffer": noise, "alias": x}.get(mode),
                         x_bf16=xb, seed_dev=seed_dev, t_dev=t_dev, clip_index0=clip0)
        new = ka[i] * known if z is None else ka[i] * known + kb[i] * z
        want = torch.where(mel, new, x0)
        assert torch.equal(x, want), (mode, (x - want).abs().max().item())
        cast = lib.cast(x, torch.empty_like(xb))
        assert torch.equal(xb, torch.where(mel, cast, xb0)), mode
    with pytest.raises(lib.FdmError, match="aligned"):
        raw = torch.empty(B * T * d + 1, device=cuda_dev)
        lib.known_frames(raw[1:].view(B, -1), known, mask, ka, kb, index, noise=noise)
    with pytest.raises(lib.FdmError, match="multiple of 4"):
        lib.known_frames(x0[:, :T * 6].contiguous(), known[:, :T * 6].contiguous(), mask, ka, kb, index,
                         noise=noise[:, :T * 6].contiguous())
    with pytest.raises(lib.FdmError, match="seed_dev"):
        lib.known_frames(x0, known, mask, ka, kb, index)


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("preset", PRESETS)
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_empty_mask_is_the_plain_call(cuda_dev, preset, precision):
    from utiles.classifierfree import ClassifierFreeSampleModel
    fdm, ae, diff, audio, conds, shape = _setup(preset, cuda_dev, precision)
    known = torch.randn(shape, device=cuda_dev)
    none = torch.zeros(shape[0], shape[1] // fdm.preset.fq, dtype=torch.bool, device=cuda_dev)
    for guided in (False, True):
        diff.denoise_fn = ClassifierFreeSampleModel(fdm, level=2.5) if guided else fdm
        want = diff.p_sample_loop(shape, audio, *conds, steps=STEPS)
        got = diff.p_sample_loop(shape, audio, *conds, steps=STEPS, known=known, known_mask=none)
        assert torch.equal(got, want), ("ddpm", guided)
        want = diff.ddim_sample(audio, shape, *conds, 4)
        got = diff.ddim_sample(audio, shape, *conds, 4, known=known, known_mask=none)
        assert torch.equal(got, want), ("ddim", guided)


@pytest.mark.parametrize("preset", PRESETS)
def test_known_rows_after_the_last_step(cuda_dev, preset):
    """bf16 (graph-replayed steps plus the high-precision tail), guidance; DDPM ending at noise level 0 and at 500 (the
    VOCASET / BIWI default range), DDIM, and the broadcast forms (1-row known, (T,) mask)."""
    fdm, ae, diff, audio, conds, shape = _setup(preset, cuda_dev, "bf16", guided=True)
    fq, z = fdm.preset.fq, fdm.preset.zdim
    known, mask = _known(shape, fq, cuda_dev)
    mel = _rows(mask, fq, z)
    for out in (diff.p_sample_loop(shape, audio, *conds, step_range=(4, 0), known=known, known_mask=mask),
                diff.p_sample_loop(shape, audio, *conds, step_range=(503, 500), known=known, known_mask=mask),
                diff.ddim_sample(audio, shape, *conds, 5, known=known, known_mask=mask)):
        assert torch.equal(out[mel], known[mel])
        assert not torch.equal(out[~mel], known[~mel])
    m1 = _rows(mask[:1].expand_as(mask), fq, z)
    k1 = known[:1].expand(shape)
    for out in (diff.sample(audio, shape, *conds, steps=STEPS, known=known[:1], known_mask=mask[0]),
                diff.ddim_sample(audio, shape, *conds, 3, known=known[:1], known_mask=mask[0])):
        assert torch.equal(out[m1], k1[m1])


def _ddpm_restated(diff, shape, audio, conds, x_T, steps, noise, known, mel):
    """Eager torch loop of public p_sample calls with the replacement rule between them."""
    sa, sb = diff.sqrt_alphas_cumprod, diff.sqrt_one_minus_alphas_cumprod
    x = torch.where(mel, sa[steps[0]] * known + sb[steps[0]] * x_T, x_T)
    for i, t in enumerate(steps):
        z = noise(t).to(x.device) if t > 0 else None
        x = diff.p_sample(x, torch.full((1,), t, dtype=torch.long, device=x.device), audio, *conds, noise=z)
        if i + 1 < len(steps):
            x = torch.where(mel, sa[t - 1] * known + sb[t - 1] * z, x)
        else:
            x = torch.where(mel, known, x)
    return x


@pytest.mark.parametrize("preset", PRESETS)
@pytest.mark.parametrize("guided", [False, True])
def test_ddpm_equals_eager_restatement(cuda_dev, preset, guided):
    """fp32, injected host noise: the graph-replayed loop equals p_sample calls with the rule applied between them."""
    fdm, ae, diff, audio, conds, shape = _setup(preset, cuda_dev, guided=guided)
    fq, z = fdm.preset.fq, fdm.preset.zdim
    known, mask = _known(shape, fq, cuda_dev)
    mel = _rows(mask, fq, z)
    g = torch.Generator().manual_seed(9)
    x_T = torch.randn(shape, generator=g).to(cuda_dev)
    table = {t: torch.randn(shape, generator=g) for t in STEPS}
    diff.noise_source = lambda t: table[t]
    got = diff.p_sample_loop(shape, audio, *conds, x_T=x_T, steps=STEPS, known=known, known_mask=mask)
    want = _ddpm_restated(diff, shape, audio, conds, x_T, STEPS, lambda t: table[t], known, mel)
    assert torch.equal(got, want), (got - want).abs().max().item()


@pytest.mark.parametrize("preset", PRESETS)
def test_ddim_equals_restatement(cuda_dev, preset):
    """fp32, no guidance: x0_hat from `tap`, the DDIM update in torch, Philox at (seed, clip_index0 + b, t_cur)."""
    from fdm_b200 import lib
    fdm, ae, diff, audio, conds, shape = _setup(preset, cuda_dev)
    fq, z = fdm.preset.fq, fdm.preset.zdim
    known, mask = _known(shape, fq, cuda_dev)
    mel = _rows(mask, fq, z)
    diff.seed, diff.clip_index0 = 1234, 6
    x_T = torch.randn(shape, generator=torch.Generator().manual_seed(2)).to(cuda_dev)
    taps = []
    got = diff.ddim_sample(audio, shape, *conds, 4, x_T=x_T, known=known, known_mask=mask,
                           tap=lambda t, x0: taps.append((t, x0)))
    ac, sa, sb = diff.alphas_cumprod, diff.sqrt_alphas_cumprod, diff.sqrt_one_minus_alphas_cumprod
    import numpy as np
    times = list(reversed(np.linspace(-1, 1000 - 1, 4 + 1).astype(np.int32).tolist()))
    pairs = [(i, j) for i, j in zip(times[:-1], times[1:]) if j >= 0]
    assert [t for t, _ in taps] == [t for t, _ in pairs]
    t0 = taps[0][0]
    x = torch.where(mel, sa[t0] * known + sb[t0] * x_T, x_T)
    for i, ((t, x0), (_, t_next)) in enumerate(zip(taps, pairs)):
        x0 = x0[0].view(shape)
        an = ac[t_next].cpu()
        s_an, c = torch.sqrt(an).to(cuda_dev), torch.sqrt(1 - an - 0.0).to(cuda_dev)
        eps = (diff.sqrt_recip_alphas_cumprod[t] * x - x0) / diff.sqrt_recipm1_alphas_cumprod[t]
        x = x0 * s_an + c * eps
        if i + 1 < len(taps):
            zz = lib.philox_normal(torch.empty(shape, device=cuda_dev), 1234, 6, t)
            x = torch.where(mel, s_an * known + c * zz, x)
        else:
            x = torch.where(mel, known, x)
    assert torch.equal(got, x), (got - x).abs().max().item()


def test_graph_equals_eager_and_reuses_graphs(cuda_dev):
    from fdm_b200 import lib
    fdm, ae, diff, audio, conds, shape = _setup("vocaset", cuda_dev, "bf16", guided=True)
    known, mask = _known(shape, fdm.preset.fq, cuda_dev)
    # (call, steps it runs: a 4-step ddim_sample skips the reference's final (t, -1) pair)
    for call, n_steps in ((lambda **kw: diff.p_sample_loop(shape, audio, *conds, steps=STEPS, **kw), len(STEPS)),
                          (lambda **kw: diff.ddim_sample(audio, shape, *conds, 4, **kw), 3)):
        got = call(known=known, known_mask=mask)
        graphs = set(fdm.engine().graph_cache)
        diff.use_cuda_graph = False
        n0 = lib.launch_count
        eager = call(known=known, known_mask=mask)
        n1 = lib.launch_count
        call()
        n2 = lib.launch_count
        diff.use_cuda_graph = True
        assert torch.equal(got, eager)
        assert (n1 - n0) - (n2 - n1) == n_steps + 1  # one launch per step plus the start state
        known2, mask2 = _known(shape, fdm.preset.fq, cuda_dev, seed=8)
        again = call(known=known2, known_mask=mask2)
        if n_steps == len(STEPS):  # (ddim_sample's per-call coefficient tables are part of its graph key with or without known frames)
            assert set(fdm.engine().graph_cache) == graphs
        diff.use_cuda_graph = False
        assert torch.equal(again, call(known=known2, known_mask=mask2))
        diff.use_cuda_graph = True


def test_fanout_with_known_frames(cuda_dev):
    fdm, ae, diff, audio, conds, shape = _setup("mead", cuda_dev, "bf16", k=3, guided=True)
    known, mask = _known(shape, fdm.preset.fq, cuda_dev)
    rep = audio.repeat_interleave(3, 0)
    assert torch.equal(diff.p_sample_loop(shape, audio, *conds, steps=STEPS, known=known, known_mask=mask),
                       diff.p_sample_loop(shape, rep, *conds, steps=STEPS, known=known, known_mask=mask))
    assert torch.equal(diff.ddim_sample(audio, shape, *conds, 4, known=known, known_mask=mask),
                       diff.ddim_sample(rep, shape, *conds, 4, known=known, known_mask=mask))


@pytest.mark.parametrize("preset", ["vocaset", "biwi"])
def test_shard_equals_rows_of_the_full_call(cuda_dev, preset):
    fdm, ae, diff, audio, conds, shape = _setup(preset, cuda_dev, "bf16", n_audio=4, guided=True)
    known, mask = _known(shape, fdm.preset.fq, cuda_dev)
    full = (diff.p_sample_loop(shape, audio, *conds, steps=STEPS, known=known, known_mask=mask),
            diff.ddim_sample(audio, shape, *conds, 4, known=known, known_mask=mask))
    s0, ns = 1, 2
    diff.clip_index0 = s0
    part = tuple(c[s0:s0 + ns] for c in conds)
    sh = (ns,) + shape[1:]
    kw = dict(known=known[s0:s0 + ns], known_mask=mask[s0:s0 + ns])
    assert torch.equal(diff.p_sample_loop(sh, audio[s0:s0 + ns], *part, steps=STEPS, **kw), full[0][s0:s0 + ns])
    assert torch.equal(diff.ddim_sample(audio[s0:s0 + ns], sh, *part, 4, **kw), full[1][s0:s0 + ns])


def test_continuation_through_quant_and_decode(cuda_dev):
    """Window 2's first O frames are known from window 1's last O frames; its audio starts O frames before window 1 ends
    (VOCASET: one latent frame per 320 audio samples)."""
    from oracle.weights import synthetic_audio
    fdm, ae, diff, _, conds, _ = _setup("vocaset", cuda_dev, "bf16", n_audio=1, guided=True)
    P = fdm.preset
    O = 8
    long = synthetic_audio(0, 2 * N_SAMPLES).to(cuda_dev)
    a1 = long[None, :N_SAMPLES].contiguous()
    T = fdm.encode_audio(a1).shape[1]
    a2 = long[None, (T - O) * 320:(T - O) * 320 + N_SAMPLES].contiguous()
    shape = (1, T * P.fq, P.zdim)
    lat1 = diff.p_sample_loop(shape, a1, *conds, steps=STEPS)
    known = torch.zeros(shape, device=cuda_dev)
    known[:, :O * P.fq] = lat1[:, -O * P.fq:]
    mask = torch.arange(T, device=cuda_dev) < O
    lat2 = diff.p_sample_loop(shape, a2, *conds, steps=STEPS, known=known, known_mask=mask)
    assert torch.equal(lat2[:, :O * P.fq], lat1[:, -O * P.fq:])
    zq1, _, (_, _, i1) = ae.quant(lat1)
    zq2, _, (_, _, i2) = ae.quant(lat2)
    assert torch.equal(i2[:O * P.fq], i1[-O * P.fq:])
    v1, v2 = ae.decode(zq1), ae.decode(zq2)
    assert v1.shape == v2.shape == (1, T, ae.args.in_dim) and torch.isfinite(v2).all()
