"""Fan-out sampling: A audio clips x K conditions in one call (sequence a*K + k on clip a). Every result must equal the
same call on audio.repeat_interleave(K, 0) bit for bit, while the audio encoder, audio_extract and the cross-attention
caches run on the A distinct clips only."""
import pytest
import torch

from helpers import N_SAMPLES, build_product

pytestmark = pytest.mark.gpu
PRESETS = ["vocaset", "mead", "biwi"]
A, K = 2, 3
STEPS = [999, 998, 1, 0]


def _setup(preset, dev, precision, n_audio=A, k=K):
    from oracle.weights import synthetic_audio
    fdm, ae, diff = build_product(preset, device=dev)
    fdm.set_precision(precision)
    ae.set_precision(precision)
    P = fdm.preset
    B = n_audio * k
    audio = torch.stack([synthetic_audio(c, N_SAMPLES) for c in range(n_audio)]).to(dev)
    idh = torch.eye(P.n_id)[[b % P.n_id for b in range(B)]].to(dev)  # sequence a*K + k: identity k
    emo = torch.eye(7)[[(3 + b) % 7 for b in range(B)]].to(dev) if P.emotion else None
    T = fdm.encode_audio(audio).shape[1] // (2 if P.pair_audio else 1)
    diff.noise_source, diff.seed = "philox", 11
    return fdm, ae, diff, audio, idh, emo, (B, T * P.fq, P.zdim)


def _conds(fdm, idh, emo):
    return (emo, idh) if fdm.preset.emotion else (idh,)


@pytest.mark.parametrize("preset", PRESETS)
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_fanout_equals_repeated_batch(cuda_dev, preset, precision):
    """p_sample_loop (Philox noise) and ddim_sample, with and without guidance; bf16 includes the high-precision tail
    step. The fan-out call replays the step graphs the repeated batch captured: same buffers, same shapes."""
    from utiles.classifierfree import ClassifierFreeSampleModel
    fdm, ae, diff, audio, idh, emo, shape = _setup(preset, cuda_dev, precision)
    conds = _conds(fdm, idh, emo)
    rep = audio.repeat_interleave(K, 0)
    for guided in (False, True):
        diff.denoise_fn = ClassifierFreeSampleModel(fdm, level=2.5) if guided else fdm
        want = diff.p_sample_loop(shape, rep, *conds, steps=STEPS)
        graphs = set(fdm.engine().graph_cache)
        got = diff.p_sample_loop(shape, audio, *conds, steps=STEPS)
        assert torch.equal(got, want), (guided, (got - want).abs().max().item())
        assert set(fdm.engine().graph_cache) == graphs
        want = diff.ddim_sample(rep, shape, *conds, 4)
        got = diff.ddim_sample(audio, shape, *conds, 4)
        assert torch.equal(got, want), (guided, (got - want).abs().max().item())


def test_audio_work_runs_per_clip(cuda_dev, monkeypatch):
    """The audio encoder sees A clip rows, audio_extract and the cross-attention GEMMs A*T rows (step and tail engine)."""
    from fdm_b200 import lib
    fdm, ae, diff, audio, idh, emo, shape = _setup("vocaset", cuda_dev, "bf16")
    T = shape[1] // fdm.preset.fq
    fdm.audio_encoder.precision = fdm._audio_mode()
    enc = fdm.audio_encoder._engine()
    enc_rows = []
    encode = enc.encode

    def counting_encode(a, *args, **kw):
        enc_rows.append(a.shape[0])
        return encode(a, *args, **kw)
    monkeypatch.setattr(enc, "encode", counting_encode)
    names = {}
    for eng in (fdm.engine(), fdm.tail_engine()):
        eng.pack()
        names[id(eng.w["ae0_w"])] = names[id(eng.w["ae2_w"])] = "audio_extract"
        for l in range(fdm.preset.layers):
            names[id(eng.w[l]["cv_w"])] = names[id(eng.w[l]["co_w"])] = "cross"
    gemm_rows = {"audio_extract": [], "cross": []}
    gemm = lib.gemm

    def counting_gemm(a, w, out, *args, **kw):
        if id(w) in names:
            gemm_rows[names[id(w)]].append(kw.get("M") or a.shape[0])
        return gemm(a, w, out, *args, **kw)
    monkeypatch.setattr(lib, "gemm", counting_gemm)
    for audio_in, rows in ((audio.clone(), A), (audio.repeat_interleave(K, 0), A * K)):
        enc_rows.clear()
        for v in gemm_rows.values():
            v.clear()
        diff.p_sample_loop(shape, audio_in, idh, steps=[999, 0])
        assert enc_rows == [rows]
        assert gemm_rows["audio_extract"] == [rows * T] * 4  # two GEMMs, step and tail engine
        assert gemm_rows["cross"] == [rows * T] * (4 * fdm.preset.layers)


def test_mead_one_clip_seven_emotions_through_vq(cuda_dev):
    """One clip x the 7 emotion one-hots through ddim_sample, quant (per-sequence emotion codebook slice) and decode."""
    fdm, ae, diff, audio, _, _, shape = _setup("mead", cuda_dev, "bf16", n_audio=1, k=7)
    emo = torch.eye(7, device=cuda_dev)
    idh = torch.eye(fdm.preset.n_id, device=cuda_dev)[:1]  # one row: broadcast to the 7 sequences
    want = diff.ddim_sample(audio.repeat_interleave(7, 0), shape, emo, idh, 4)
    lat = diff.ddim_sample(audio, shape, emo, idh, 4)
    assert torch.equal(lat, want)
    zq, _, (_, _, idx) = ae.quant(lat, emo)
    zq_r, _, (_, _, idx_r) = ae.quant(want, emo)
    assert torch.equal(idx, idx_r) and torch.equal(zq, zq_r)
    assert torch.equal(ae.decode(zq), ae.decode(zq_r))
    L = shape[1]
    for k in range(7):  # each sequence is quantised in its own emotion's slice
        _, _, (_, _, i1) = ae.quant(lat[k:k + 1], emo[k:k + 1])
        assert torch.equal(i1, idx[k * L:(k + 1) * L])


@pytest.mark.parametrize("preset", PRESETS)
def test_forward_and_p_sample_fanout(cuda_dev, preset):
    fdm, ae, diff, audio, idh, emo, shape = _setup(preset, cuda_dev, "fp32")
    conds = _conds(fdm, idh, emo)
    rep = audio.repeat_interleave(K, 0)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(shape, generator=g).to(cuda_dev)
    noise = torch.randn(shape, generator=g).to(cuda_dev)
    t = torch.full((1,), 700, dtype=torch.long, device=cuda_dev)
    assert torch.equal(fdm(audio, t, x, *conds), fdm(rep, t, x, *conds))
    assert torch.equal(diff.p_sample(x, t, audio, *conds, noise=noise), diff.p_sample(x, t, rep, *conds, noise=noise))
    taps = {}
    for name, a in (("fan", audio), ("rep", rep)):
        diff.p_sample_loop(shape, a, *conds, steps=[999, 500], tap=lambda t, x0: taps.setdefault(name, []).append((t, x0)))
    assert len(taps["fan"]) == 2
    for (t1, x1), (t2, x2) in zip(taps["fan"], taps["rep"]):
        assert t1 == t2 and torch.equal(x1, x2)


def test_fanout_errors_and_cache_key(cuda_dev):
    fdm, ae, diff, audio, idh, emo, shape = _setup("vocaset", cuda_dev, "bf16")
    bad = (A * K - 1,) + shape[1:]
    t = torch.full((1,), 5, dtype=torch.long, device=cuda_dev)
    with pytest.raises(ValueError, match=f"{A * K - 1} sequences .* {A} audio clips"):
        diff.p_sample_loop(bad, audio, idh[:1], steps=[1, 0])
    with pytest.raises(ValueError, match="audio clips"):
        diff.ddim_sample(audio, bad, idh[:1], 2)
    with pytest.raises(ValueError, match="audio clips"):
        fdm(audio, t, torch.zeros(bad, device=cuda_dev), idh[:1])
    with pytest.raises(ValueError, match="rows"):  # a condition of A rows is neither B rows nor 1
        diff.p_sample_loop(shape, audio, idh[:A], steps=[1, 0])
    # K = 3, then K = 2 on the same audio and condition tensors: only K tells the two calls apart
    id1 = idh[:1]
    want = {k: diff.p_sample_loop((A * k,) + shape[1:], audio.repeat_interleave(k, 0), id1, steps=STEPS) for k in (3, 2)}
    for k in (3, 2, 3):
        got = diff.p_sample_loop((A * k,) + shape[1:], audio, id1, steps=STEPS)
        assert torch.equal(got, want[k]), k
    # precomputed (A, N, C) features for an (A, L) audio tensor
    audio2 = audio.clone()
    fdm.set_audio_features(audio2, fdm.encode_audio(audio).clone())
    assert torch.equal(diff.p_sample_loop((A * 2,) + shape[1:], audio2, id1, steps=STEPS), want[2])
    with pytest.raises(ValueError, match="features"):
        fdm.set_audio_features(audio2, fdm.encode_audio(audio).repeat_interleave(2, 0))
