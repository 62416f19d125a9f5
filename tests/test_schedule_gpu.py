"""Condition schedules on the GPU: fdm_vq_quantize_runs / fdm_vq_stats_runs against the per-clip entry points run by run (both
paths, D = 64 / 128), constant schedules against the per-sequence calls bit for bit, prefix invariance of a switch (self-
attention is causal, everything else per frame), per-frame encode against a torch restatement, refusals that keep the
prepared state, graph reuse, and MEAD sample_long -> per-frame quant -> decode end to end."""
import pytest
import torch
import torch.nn.functional as F

from helpers import N_SAMPLES, build_product

pytestmark = pytest.mark.gpu
STEPS = [999, 998, 1, 0]


# ---- VQ kernels -------------------------------------------------------------------------------------------------------
def _schedules(B, T, fq):
    """name -> (B, T) int64 slice index per frame."""
    g = torch.Generator().manual_seed(3)
    every = torch.randint(0, 7, (B, T), generator=g)
    rows = {}
    rows["every_frame"] = every
    rows["one_per_clip"] = torch.randint(0, 7, (B, 1), generator=g).expand(B, T).clone()
    for n in (127, 128, 129):  # a run ending at n rows (fq = 1 only reaches every row count)
        s = torch.full((B, T), 2)
        s[:, n // fq:] = 5
        s[1:, : n // fq // 2] = 6
        rows[f"end_{n}"] = s
    return rows


def _per_run_reference(z, cb, runs, algo):
    from fdm_b200 import lib
    clip_run, run_l0, run_off = (t.tolist() for t in runs)
    B, L, D = z.shape
    idx = torch.empty(B * L, dtype=torch.int64, device=z.device)
    bdl = torch.empty(B, D, L, device=z.device)
    rows = torch.empty(B, L, D, device=z.device)
    for b in range(B):
        for r in range(clip_run[b], clip_run[b + 1]):
            l0 = run_l0[r]
            l1 = run_l0[r + 1] if r + 1 < clip_run[b + 1] else L
            i, zq, zr = lib.vq_quantize(z[b:b + 1, l0:l1].contiguous(), cb, 256,
                                        code_offset=torch.tensor([run_off[r]], device=z.device), want_bdl=True,
                                        want_rows=True, algo=algo)
            idx[b * L + l0:b * L + l1] = i[:, 0]
            bdl[b, :, l0:l1] = zq[0]
            rows[b, l0:l1] = zr[0]
    return idx, bdl, rows


@pytest.mark.parametrize("D", [64, 128])
@pytest.mark.parametrize("algo", ["tensor", "ffma"])
@pytest.mark.parametrize("fq", [1, 8])
def test_vq_runs_equal_the_per_clip_entry_point_run_by_run(cuda_dev, D, algo, fq):
    from fdm_b200 import lib
    from fdm_b200.vqvae import slice_runs
    a = lib.VQ_TENSOR if algo == "tensor" else lib.VQ_FFMA
    g = torch.Generator(device=cuda_dev).manual_seed(D + fq)
    B, T = 3, 300 // fq
    L = T * fq
    cb = torch.randn(7 * 256, D, device=cuda_dev, generator=g) * 0.3
    cb[256:512] = cb[:256]  # duplicated codes across slices 0 and 1
    cb[256 * 4 + 17] = cb[256 * 4 + 3]  # and inside one slice (ties: lowest index)
    z = torch.randn(B, L, D, device=cuda_dev, generator=g) * 0.3
    z[0, 5] = cb[256 * 4 + 3]  # an exact tie
    for name, s in _schedules(B, T, fq).items():
        if fq == 8 and name.startswith("end_") and name != "end_128":
            continue  # (fq = 8 runs are multiples of 8 rows: only 128 is reachable)
        runs = slice_runs(s * 256, fq)
        rc = torch.zeros(1, dtype=torch.int64, device=cuda_dev)
        idx, bdl, rows = lib.vq_quantize_runs(z, cb, 256, runs, want_bdl=True, want_rows=True, algo=a, recheck_rows=rc)
        ri, rb, rr = _per_run_reference(z, cb, runs, a)
        assert torch.equal(idx[:, 0], ri), name
        assert torch.equal(bdl, rb), name
        assert torch.equal(rows, rr), name
        # indices only / z_q only: the same values
        i2, _, _ = lib.vq_quantize_runs(z, cb, 256, runs, want_bdl=False, want_rows=False, algo=a)
        assert torch.equal(i2, idx), name
        sq, hist = lib.vq_stats_runs(z, cb, idx.view(-1), 256, runs)
        off_rows = s.repeat_interleave(fq, dim=1).to(cuda_dev) * 256
        e = cb[off_rows.view(-1) + idx.view(-1)]
        assert torch.equal(hist, torch.bincount(idx.view(-1), minlength=256)), name
        want_sq = ((e.double() - z.view(-1, D).double()) ** 2).sum()
        assert abs(sq.item() - want_sq.item()) <= 1e-5 * want_sq.item(), name
        if name == "one_per_clip":  # one run per clip: the per-clip entry points, bit for bit
            off = (s[:, 0] * 256).to(cuda_dev)
            pi, pb, pr = lib.vq_quantize(z, cb, 256, code_offset=off, want_bdl=True, want_rows=True, algo=a)
            assert torch.equal(pi, idx) and torch.equal(pb, bdl) and torch.equal(pr, rows)
            psq, phist = lib.vq_stats(z, cb, idx.view(-1), 256, code_offset=off)
            assert torch.equal(psq, sq) and torch.equal(phist, hist)


def test_vq_runs_refuse_a_small_workspace(cuda_dev):
    import ctypes as C
    from fdm_b200 import lib
    from fdm_b200.vqvae import slice_runs
    z = torch.zeros(2, 64, 64, device=cuda_dev)
    cb = torch.zeros(512, 64, device=cuda_dev)
    rs, keep = lib._vq_runs(slice_runs(torch.zeros(2, 8, dtype=torch.int64), 8), 2, 64, cuda_dev)
    ws = torch.empty(4, dtype=torch.int32, device=cuda_dev)
    rc = lib.load().fdm_vq_quantize_runs(z.data_ptr(), cb.data_ptr(), C.byref(rs), 2, 64, 64, 256, None, None, None, 0, None,
                                         ws.data_ptr(), 16, torch.cuda.current_stream().cuda_stream)
    assert rc != 0 and b"workspace" in lib.load().fdm_last_error()


# ---- sampling -----------------------------------------------------------------------------------------------------------
def _setup(preset, dev, precision, n_audio=2, k=1, guided=False, n_samples=N_SAMPLES):
    from oracle.weights import synthetic_audio
    from utiles.classifierfree import ClassifierFreeSampleModel
    fdm, ae, diff = build_product(preset, device=dev)
    fdm.set_precision(precision)
    ae.set_precision(precision)
    P = fdm.preset
    B = n_audio * k
    audio = torch.stack([synthetic_audio(c, n_samples) for c in range(n_audio)]).to(dev)
    T = fdm.encode_audio(audio).shape[1] // (2 if P.pair_audio else 1)
    idh = torch.eye(P.n_id)[[b % P.n_id for b in range(B)]].to(dev)
    emo = torch.eye(7)[[(3 + b) % 7 for b in range(B)]].to(dev) if P.emotion else None
    diff.noise_source, diff.seed = "philox", 11
    if guided:
        diff.denoise_fn = ClassifierFreeSampleModel(fdm, level=2.5)
    return fdm, ae, diff, audio, idh, emo, (B, T * P.fq, P.zdim)


def _conds(P, idh, emo):
    return (emo, idh) if P.emotion else (idh,)


def _frames(c, T):
    return None if c is None else c[:, None].expand(-1, T, -1).contiguous()


@pytest.mark.parametrize("preset", ["vocaset", "mead"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_constant_schedule_equals_per_sequence_call(cuda_dev, preset, precision):
    """sample / ddim_sample / p_sample / FDM.forward with guidance and fan-out (2 clips x 2 sequences)."""
    fdm, ae, diff, audio, idh, emo, shape = _setup(preset, cuda_dev, precision, k=2, guided=True)
    P = fdm.preset
    T = shape[1] // P.fq
    seq, frm = _conds(P, idh, emo), _conds(P, _frames(idh, T), _frames(emo, T))
    a = diff.sample(audio, shape, *seq, steps=STEPS)
    b = diff.sample(audio, shape, *frm, steps=STEPS)
    assert torch.equal(a, b)
    # the identity per frame only, the emotion per sequence (and the other way round)
    if P.emotion:
        assert torch.equal(a, diff.sample(audio, shape, seq[0], frm[1], steps=STEPS))
        assert torch.equal(a, diff.sample(audio, shape, frm[0], seq[1], steps=STEPS))
    # one row for all sequences
    one = _conds(P, idh[:1], None if emo is None else emo[:1])
    one_f = _conds(P, _frames(idh[:1], T), _frames(None if emo is None else emo[:1], T))
    assert torch.equal(diff.sample(audio, shape, *one, steps=STEPS), diff.sample(audio, shape, *one_f, steps=STEPS))
    x_T = torch.randn(shape, device=cuda_dev)
    assert torch.equal(diff.ddim_sample(audio, shape, *seq, 5, x_T=x_T), diff.ddim_sample(audio, shape, *frm, 5, x_T=x_T))
    noise = torch.randn(shape, device=cuda_dev)
    t = torch.full((shape[0],), 500, device=cuda_dev, dtype=torch.long)
    assert torch.equal(diff.p_sample(x_T, t, audio, *seq, noise=noise), diff.p_sample(x_T, t, audio, *frm, noise=noise))
    f_frm = (_frames(emo, T), _frames(idh, T)) if P.emotion else (_frames(idh, T),)
    f_seq = (emo, idh) if P.emotion else (idh,)
    assert torch.equal(fdm(audio, t[:1], x_T, *f_seq), fdm(audio, t[:1], x_T, *f_frm))


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_constant_schedule_equals_per_sequence_sample_long(cuda_dev, precision):
    T = 200  # 3 windows of 90 frames with 30 shared
    fdm, ae, diff, audio, idh, emo, _ = _setup("mead", cuda_dev, precision, k=2, guided=True,
                                               n_samples=320 * (2 * T - 1) + 400)
    shape = (4, T * 8, 64)
    seq = (emo, idh)
    frm = (_frames(emo, T), _frames(idh, T))
    a = diff.sample_long(audio, shape, *seq, window=90, overlap=30, steps=STEPS)
    assert torch.equal(a, diff.sample_long(audio, shape, *frm, window=90, overlap=30, steps=STEPS))
    a = diff.sample_long(audio, shape, *seq, window=90, overlap=30, ddim_steps=4)
    assert torch.equal(a, diff.sample_long(audio, shape, *frm, window=90, overlap=30, ddim_steps=4))


def _switched(emo, T, j, to):
    s = _frames(emo, T).clone()
    s[:, j:] = torch.eye(7, device=emo.device)[to]
    return s


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_switch_leaves_earlier_frames_unchanged(cuda_dev, precision):
    fdm, ae, diff, audio, idh, emo, shape = _setup("mead", cuda_dev, precision, guided=True)
    T = shape[1] // 8
    j = T // 2
    a = diff.sample(audio, shape, _frames(emo, T), idh, steps=STEPS)
    b = diff.sample(audio, shape, _switched(emo, T, j, 0), idh, steps=STEPS)
    assert torch.equal(a[:, :8 * j], b[:, :8 * j])
    assert not torch.equal(a[:, 8 * j:8 * j + 8], b[:, 8 * j:8 * j + 8])


@pytest.mark.parametrize("j", [70, 100])  # window 1 covers [60, 150): 70 lies in the overlap with window 0, 100 does not
def test_switch_in_the_second_window_of_sample_long(cuda_dev, j):
    T = 200
    fdm, ae, diff, audio, idh, emo, _ = _setup("mead", cuda_dev, "bf16", guided=True, n_samples=320 * (2 * T - 1) + 400)
    shape = (2, T * 8, 64)
    a = diff.sample_long(audio, shape, _frames(emo, T), idh, window=90, overlap=30, steps=STEPS)
    b = diff.sample_long(audio, shape, _switched(emo, T, j, 0), idh, window=90, overlap=30, steps=STEPS)
    assert torch.equal(a[:, :8 * j], b[:, :8 * j])
    assert not torch.equal(a[:, 8 * j:8 * j + 8], b[:, 8 * j:8 * j + 8])


def test_refused_schedule_keeps_the_prepared_state_and_graphs_are_reused(cuda_dev):
    fdm, ae, diff, audio, idh, emo, shape = _setup("mead", cuda_dev, "bf16", guided=True)
    T = shape[1] // 8
    s1 = _switched(emo, T, 5, 1)
    a = diff.sample(audio, shape, s1, idh, steps=STEPS)
    eng = fdm.engine()
    state = [t.clone() for t in eng.addend] + [eng.addend_delta.clone()]
    key = fdm.__dict__["_prep_key"]
    n_graphs = len(eng.graph_cache)
    for bad in (torch.zeros(2, T - 1, 7, device=cuda_dev), torch.zeros(3, T, 7, device=cuda_dev),
                torch.zeros(2, T, 6, device=cuda_dev)):
        with pytest.raises(ValueError):
            diff.sample(audio, shape, bad, idh, steps=STEPS)
        assert fdm.__dict__["_prep_key"] is key
        assert all(torch.equal(x, y) for x, y in zip(state, list(eng.addend) + [eng.addend_delta]))
    # a new schedule of the same shape: the captured graphs are replayed, none are added
    s2 = _switched(emo, T, 9, 4)
    b = diff.sample(audio, shape, s2, idh, steps=STEPS)
    assert len(eng.graph_cache) == n_graphs and not torch.equal(a, b)
    diff.use_cuda_graph = False
    assert torch.equal(b, diff.sample(audio, shape, s2, idh, steps=STEPS))  # graph replay = eager


# ---- EVQ-VAE ------------------------------------------------------------------------------------------------------------
def _encode_frames(sd, verts, emo_frames, n_layers=6, heads=8):
    """oracle/reference_ops.vq_encode (MEAD) with the emotion_mapping output of frame f added to frame f."""
    from oracle import reference_ops as R
    p = "encoder."
    x = F.leaky_relu(F.linear(verts, sd[p + "vertice_mapping.0.weight"], sd[p + "vertice_mapping.0.bias"]), 0.2)
    x = x + F.leaky_relu(F.linear(emo_frames, sd[p + "emotion_mapping.0.weight"], sd[p + "emotion_mapping.0.bias"]), 0.2)
    h = x.t()[None]
    h = F.conv1d(F.pad(h, (2, 2), mode="replicate"), sd[p + "squasher.0.0.weight"], sd[p + "squasher.0.0.bias"])
    x = F.instance_norm(F.leaky_relu(h, 0.2), eps=1e-5)[0].t()
    x = F.linear(x, sd[p + "encoder_linear_embedding.net.weight"], sd[p + "encoder_linear_embedding.net.bias"])
    d = x.shape[-1]
    x = x + R.sin_pe(1, d)[0]
    dh, T = d // heads, x.shape[0]
    for l in range(n_layers):
        a = p + f"encoder_transformer.net.{2 * l}.fn."
        y = F.layer_norm(x, (d,), sd[a + "norm.weight"], sd[a + "norm.bias"], 1e-5)
        qkv = F.linear(y, sd[a + "fn.to_qkv.weight"]).view(T, 3, heads, dh).permute(1, 2, 0, 3)
        o = (torch.softmax((qkv[0] @ qkv[1].transpose(-1, -2)) * (d ** -0.5), -1) @ qkv[2]).permute(1, 0, 2).reshape(T, d)
        x = x + F.linear(o, sd[a + "fn.to_out.weight"], sd[a + "fn.to_out.bias"])
        m = p + f"encoder_transformer.net.{2 * l + 1}.fn."
        y = F.layer_norm(x, (d,), sd[m + "norm.weight"], sd[m + "norm.bias"], 1e-5)
        x = x + F.linear(R._gelu_tanh(F.linear(y, sd[m + "fn.l1.weight"], sd[m + "fn.l1.bias"])), sd[m + "fn.l2.weight"],
                         sd[m + "fn.l2.bias"])
    x = F.linear(x, sd[p + "encoder_linear_embedding_post.net.weight"], sd[p + "encoder_linear_embedding_post.net.bias"])
    return x.reshape(T * 8, 64)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_per_frame_encode_and_quant(cuda_dev, precision):
    from helpers import build_vqvae, encoder_case
    ae = build_vqvae("mead", device=cuda_dev)
    ae.set_precision(precision)
    sd, x, emo, _ = encoder_case("mead", ae)
    emo = emo.reshape(7)
    sd = {k: v.double() if v.is_floating_point() else v for k, v in sd.items()}
    T = x.shape[0]
    sched = emo[None].expand(T, -1).clone()
    sched[T // 3:] = torch.eye(7)[1]
    sched[2 * T // 3:] = 0.6 * torch.eye(7)[1] + 0.4 * torch.eye(7)[5]  # soft rows: still argmax 1
    h = ae.encode(x[None].to(cuda_dev), sched[None].to(cuda_dev))
    want = _encode_frames(sd, x.double(), sched.double()).float()
    if precision == "fp32":
        err = (h[0].cpu() - want).abs().max().item() / max(1.0, want.abs().max().item())
        assert err < 1e-4, err
    else:
        rel = ((h[0].cpu() - want).norm() / want.norm()).item()
        assert rel < 2e-2, rel
    # a constant schedule is the per-clip call, bit for bit (encode and quant)
    const = emo[None, None].expand(1, T, -1).to(cuda_dev)
    hc = ae.encode(x[None].to(cuda_dev), const)
    assert torch.equal(hc, ae.encode(x[None].to(cuda_dev), emo.to(cuda_dev)))
    zq_a, loss_a, (_, _, ia) = ae.quant(hc, emo.to(cuda_dev))
    zq_b, loss_b, (_, _, ib) = ae.quant(hc, const)
    assert torch.equal(ia, ib) and torch.equal(zq_a, zq_b) and torch.equal(loss_a, loss_b)


def test_mead_long_schedule_end_to_end(cuda_dev):
    """sample_long with an emotion switch and a soft cross-fade -> per-frame quant -> decode."""
    T = 200
    fdm, ae, diff, audio, idh, emo, _ = _setup("mead", cuda_dev, "bf16", guided=True, n_samples=320 * (2 * T - 1) + 400)
    eye = torch.eye(7, device=cuda_dev)
    sched = eye[2].expand(2, T, 7).clone()
    sched[:, 80:] = eye[6]
    lam = torch.linspace(0, 1, 40, device=cuda_dev)[:, None]
    sched[1, 120:160] = (1 - lam) * eye[6] + lam * eye[0]  # a cross-fade on the second sequence
    sched[1, 160:] = eye[0]
    lat = diff.sample_long(audio, (2, T * 8, 64), sched, idh, window=90, overlap=30, steps=STEPS)
    zq, loss, (_, _, idx) = ae.quant(lat, sched)
    verts = ae.decode(zq)
    assert verts.shape == (2, T, 5023 * 3) and torch.isfinite(verts).all() and torch.isfinite(loss).all()
    slice_of = torch.argmax(sched, -1).repeat_interleave(8, dim=1)  # (2, 8T)
    cb = ae.quantize.embedding.weight.float()
    want = cb[(slice_of * 256).view(-1) + idx[:, 0]].view(2, T * 8, 64)
    assert torch.equal(zq.transpose(1, 2), want)  # every frame's code comes from its own emotion's slice
