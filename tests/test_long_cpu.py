"""CPU: the window plan of sample_long (windows, audio slices, sequence order, noise keys, assembly), its argument checks
(they run before anything touches a device), and the ctypes mirrors of fdm_noise_keys / fdm_window_args."""
import os
import re
import subprocess
import tempfile

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HDR = os.path.join(ROOT, "include", "fdm_b200.h")


def _preset(name):
    from fdm_b200.presets import PRESETS
    return PRESETS[name]


@pytest.mark.parametrize("T, n_w", [(1, 1), (100, 1), (419, 1), (420, 1), (421, 2), (780, 2), (781, 3), (3000, 9)])
def test_windows_below_at_and_above_the_window(T, n_w):
    from fdm_b200.windows import default_window, plan_windows
    P = _preset("vocaset")
    assert default_window(P) == (420, 60) and default_window(_preset("biwi")) == (350, 50)
    plan = plan_windows(P, (2, T * P.fq, P.zdim), 1, 16000 * 70)
    assert (plan.W, plan.O, plan.S, plan.K, plan.A) == (420, 60, 360, 2, 1)
    assert plan.n_w == n_w
    assert plan.starts() == [360 * w for w in range(n_w)]
    assert plan.T_pad == 360 * (n_w - 1) + 420 >= T
    if n_w > 1:  # the last window starts early enough that its overlap with the one before is real frames
        assert plan.starts()[-1] + plan.O < T


@pytest.mark.parametrize("preset", ["vocaset", "mead", "biwi"])
def test_audio_slices_yield_exactly_the_window(preset):
    from fdm_b200.presets import conv_out_len
    from fdm_b200.windows import plan_windows
    P = _preset(preset)
    r = 2 if P.pair_audio else 1
    T = 1000
    L = 320 * (T * r - 1) + 400 + 1234
    plan = plan_windows(P, (2, T * P.fq, P.zdim), 2, L)
    assert plan.r == r
    for w in range(plan.n_w):
        lo, hi = plan.audio_bounds(w)
        assert lo == w * plan.S * r * 320 and conv_out_len(hi - lo) == plan.W * r
    audio = torch.randn(2, L)
    win = plan.window_audio(audio)
    assert win.shape == (2 * plan.n_w, plan.audio_len)
    for a in range(2):
        for w in range(plan.n_w):
            lo, hi = plan.audio_bounds(w)
            want = torch.zeros(plan.audio_len)
            part = audio[a, lo:hi]
            want[:part.numel()] = part
            assert torch.equal(win[a * plan.n_w + w], want), (a, w)
    assert hi > L  # the last window runs past the audio: zero-padded


def _plan(A=2, K=3, T=50, W=20, O=6):
    from fdm_b200.windows import WindowPlan
    return WindowPlan(A=A, K=K, T=T, W=W, O=O, r=1)


def test_sequence_order_and_gather_with_fanout():
    plan = _plan()
    A, K, fq, z = plan.A, plan.K, 2, 4
    assert (plan.S, plan.n_w, plan.T_pad) == (14, 4, 62)
    # value = 1000 * long sequence + absolute frame, in every element of the frame
    g = torch.arange(A * K)[:, None] * 1000 + torch.arange(plan.T_pad)[None]
    full = g[:, :, None, None].expand(A * K, plan.T_pad, fq, z).reshape(A * K, plan.T_pad * fq, z).float()
    win = plan.gather(full)
    assert win.shape == (A * plan.n_w * K, plan.W * fq, z)
    for a in range(A):
        for w in range(plan.n_w):
            for k in range(K):
                s = plan.seq(a, w, k)
                assert s == (a * plan.n_w + w) * K + k
                rows = win[s].view(plan.W, fq * z)
                want = (a * K + k) * 1000 + w * plan.S + torch.arange(plan.W)
                assert torch.equal(rows, want[:, None].float().expand(-1, fq * z)), (a, w, k)
    ids = torch.eye(8)[: A * K]
    rep = plan.repeat_rows(ids)
    for a in range(A):
        for w in range(plan.n_w):
            for k in range(K):
                assert torch.equal(rep[plan.seq(a, w, k)], ids[a * K + k])
    assert plan.repeat_rows(ids[:1]) is not None and plan.repeat_rows(ids[:1]).shape == (1, 8)
    assert plan.repeat_rows(None) is None


def test_noise_keys_and_weights():
    plan = _plan()
    d = 64
    clip, e4 = plan.noise_keys(5, d)
    assert clip.dtype == e4.dtype == torch.int64 and clip.shape == e4.shape == (plan.n_seq,)
    for a in range(plan.A):
        for w in range(plan.n_w):
            for k in range(plan.K):
                s = plan.seq(a, w, k)
                assert clip[s] == 5 + a * plan.K + k
                assert e4[s] == w * plan.S * d // 4
    lam = plan.weights()
    assert lam.dtype == torch.float32 and lam.shape == (plan.O,)
    assert torch.equal(lam, torch.tensor([(j + 1) / (plan.O + 1) for j in range(plan.O)], dtype=torch.float32))


def test_assembly_indices():
    plan = _plan()
    w, row = plan.assembly_index()
    assert w.shape == row.shape == (plan.T,)
    for f in range(plan.T):
        want_w = min(f // plan.S, plan.n_w - 1)
        assert (w[f], row[f]) == (want_w, f - want_w * plan.S)
        assert 0 <= row[f] < (plan.S if w[f] < plan.n_w - 1 else plan.W)
    # windows gathered from a full-length latent assemble back to its first T frames
    full = torch.randn(plan.A * plan.K, plan.T_pad * 2, 3)
    assert torch.equal(plan.assemble(plan.gather(full)), full[:, :plan.T * 2])
    # rows [S, W) of a window that is not the last are not read
    win = plan.gather(full)
    v = win.view(plan.A, plan.n_w, plan.K, plan.W, -1)
    v[:, :-1, :, plan.S:] = float("nan")
    assert torch.equal(plan.assemble(win), full[:, :plan.T * 2])


@pytest.fixture(scope="module")
def meta_vocaset():
    import warnings
    warnings.simplefilter("ignore")
    os.environ["FDM_B200_RANDOM_AUDIO_ENCODER"] = "1"
    with torch.device("meta"):
        from models.fdm_vocaset import FDM
        from video_diffusion_pytorch.diffusion_BIWI_encoder_decoder import GaussianDiffusion
        return GaussianDiffusion(FDM(feature_dim=1024), timesteps=1000, loss_type="l2")


T_CALL = 500
L_CALL = 320 * (T_CALL - 1) + 400  # exactly T_CALL VOCASET frames


@pytest.mark.parametrize("case, match", [
    ("overlap_zero", r"overlap 0 must lie in \[1, window // 2 = 210\]"),
    ("overlap_half", r"overlap 211 must lie in \[1, window // 2 = 210\]"),
    ("stride_phase", r"multiple of the period 30"),
    ("window_long", r"window 630 is longer than the 600 frames"),
    ("window_type", r"window must be an int"),
    ("audio_short", rf"latent has {T_CALL} frames but the audio only yields {T_CALL - 1}"),
    ("audio_dim", r"audio must be a floating-point \(A, L\) tensor"),
    ("audio_dtype", r"audio must be a floating-point"),
    ("zdim", r"is not \(B, 16\*T, 64\)"),
    ("fq", r"is not \(B, 16\*T, 64\)"),
    ("fanout", r"3 sequences do not split evenly over 2 audio clips"),
    ("cond_rows", r"the call has 4 sequences \(give 4 rows or 1\)"),
    ("cond_count", r"expected 1 condition"),
    ("ddim_and_steps", r"not both"),
    ("ddim_steps", r"ddim_steps must be an int >= 2"),
    ("steps_empty", r"steps is empty"),
    ("x_T_shape", r"x_T must be a floating-point tensor of the call's shape"),
])
def test_sample_long_arguments_are_checked(meta_vocaset, case, match):
    """VOCASET: fq = 16, zdim = 64, period 30; a call of 2 clips x 2 sequences x 500 frames."""
    diff = meta_vocaset
    shape = (4, T_CALL * 16, 64)
    audio, idh = torch.zeros(2, L_CALL), torch.eye(8)[:4]
    args, kw = [audio, shape, idh], {}
    if case == "overlap_zero":
        kw = dict(overlap=0)
    elif case == "overlap_half":
        kw = dict(overlap=211)
    elif case == "stride_phase":
        kw = dict(window=400, overlap=50)
    elif case == "window_long":
        kw = dict(window=630, overlap=30)
    elif case == "window_type":
        kw = dict(window=420.0)
    elif case == "audio_short":
        args[0] = audio[:, :-1]
    elif case == "audio_dim":
        args[0] = audio[None]
    elif case == "audio_dtype":
        args[0] = audio.to(torch.int16)
    elif case == "zdim":
        args[1] = (4, T_CALL * 16, 32)
    elif case == "fq":
        args[1] = (4, T_CALL * 16 + 8, 64)
    elif case == "fanout":
        args[1], args[2] = (3,) + shape[1:], idh[:3]
    elif case == "cond_rows":
        args[2] = idh[:2]
    elif case == "cond_count":
        args.append(idh)
    elif case == "ddim_and_steps":
        kw = dict(ddim_steps=10, steps=[1, 0])
    elif case == "ddim_steps":
        kw = dict(ddim_steps=1)
    elif case == "steps_empty":
        kw = dict(steps=[])
    elif case == "x_T_shape":
        kw = dict(x_T=torch.zeros(4, T_CALL * 16 - 16, 64))
    with pytest.raises(ValueError, match=match):
        diff.sample_long(*args, **kw)


def test_sample_long_takes_no_known_frames_or_tap(meta_vocaset):
    audio, idh = torch.zeros(1, L_CALL), torch.eye(8)[:1]
    for kw in (dict(known=torch.zeros(1, T_CALL * 16, 64), known_mask=torch.zeros(T_CALL, dtype=torch.bool)),
               dict(tap=lambda t, x: None)):
        with pytest.raises(TypeError):
            meta_vocaset.sample_long(audio, (1, T_CALL * 16, 64), idh, **kw)


@pytest.mark.parametrize("cname, pyname", [("fdm_noise_keys", "NoiseKeys"), ("fdm_window_args", "WindowArgs")])
def test_window_structs_mirror_the_header(cname, pyname):
    import ctypes as C
    from fdm_b200 import lib
    cls = getattr(lib, pyname)
    hdr = re.sub(r"/\*.*?\*/", "", open(HDR).read(), flags=re.S)
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (cname, cname), hdr, flags=re.S).group(1)
    width = {"int64_t": 8, "uint64_t": 8, "int32_t": 4, "float": 4}
    fields = []
    for decl in filter(None, (x.strip() for x in body.split(";"))):
        m = re.match(r"(const\s+)?(\w+)\s*(\*?)\s*(.*)", decl)
        for nm in m.group(4).split(","):
            nm = nm.strip()
            fields.append((nm.lstrip("* "), 8 if (m.group(3) or nm.startswith("*")) else width[m.group(2)]))
    assert [(n, C.sizeof(t)) for n, t in cls._fields_] == fields
    with tempfile.TemporaryDirectory() as td:
        src, exe = os.path.join(td, "s.c"), os.path.join(td, "s")
        with open(src, "w") as f:
            f.write('#include <stdio.h>\n#include "%s"\nint main(void){printf("%%zu\\n", sizeof(%s));return 0;}\n' % (HDR, cname))
        subprocess.check_call(["gcc", "-o", exe, src])
        assert int(subprocess.check_output([exe])) == C.sizeof(cls)


def test_new_entry_points_are_bound():
    from fdm_b200 import lib
    handle = lib.load()
    assert handle.fdm_ddpm_step_keyed is not None and handle.fdm_window_blend is not None
    assert handle.fdm_abi_version() == 4
