"""CPU: condition schedules (per-frame identity / emotion rows). The argument checks of the per-frame form (they run before
anything touches a device), the window gather of per-frame conditions, the run table of per-frame codebook slices with a
restatement of the tiles fdm_vq_quantize_runs cuts from it, and the ctypes mirror of fdm_vq_runs."""
import os
import re
import subprocess
import tempfile

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HDR = os.path.join(ROOT, "include", "fdm_b200.h")


# ---- argument checks --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape, match", [
    ((3, 10, 8), r"3 rows; the call has 4 sequences"),
    ((4, 9, 8), r"9 frames; the call has 10"),
    ((1, 11, 8), r"11 frames; the call has 10"),
    ((4, 10, 7), r"rows of 7 entries; it needs 8"),
])
def test_frame_condition_refusals(shape, match):
    from fdm_b200.vqvae import check_frame_cond
    with pytest.raises(ValueError, match=match):
        check_frame_cond(torch.zeros(shape), 4, 10, 8)
    check_frame_cond(torch.zeros(4, 10, 8), 4, 10, 8)
    check_frame_cond(torch.zeros(1, 10, 8), 4, 10, 8)


T_CALL = 500
L_CALL = 320 * (T_CALL - 1) + 400  # exactly T_CALL VOCASET frames


@pytest.mark.parametrize("cond, match", [
    ((4, T_CALL - 1, 8), rf"{T_CALL - 1} frames; the call has {T_CALL}"),
    ((2, T_CALL, 8), r"2 rows; the call has 4 sequences"),
    ((4, T_CALL, 7), r"rows of 7 entries; it needs 8"),
])
def test_sample_long_refuses_bad_schedules(cond, match):
    """sample_long's argument check takes a schedule over the full length T, before any window is planned on a device."""
    from types import SimpleNamespace
    from fdm_b200.modules import GaussianDiffusionBase
    from fdm_b200.presets import PRESETS
    diff = SimpleNamespace(n_cond=1)
    args = (PRESETS["vocaset"], torch.zeros(2, L_CALL), (4, T_CALL * 16, 64))
    with pytest.raises(ValueError, match=match):
        GaussianDiffusionBase._check_long(diff, *args, (torch.zeros(cond),), None, None, None, None, None, None)
    plan = GaussianDiffusionBase._check_long(diff, *args, (torch.zeros(1, T_CALL, 8),), None, None, None, None, None, None)
    assert plan.n_w == 2


def test_mead_quant_and_encode_refuse_bad_schedules():
    from models.utils.config import vq_vae_args
    from models.vq_vae_emotion import VQAutoEncoder
    with torch.device("meta"):
        ae = VQAutoEncoder(vq_vae_args())
    lat = torch.zeros(2, 8 * 12, 64)
    for bad, match in (((2, 11, 7), r"11 frames; the call has 12"), ((3, 12, 7), r"3 rows"), ((2, 12, 6), r"6 entries")):
        with pytest.raises(ValueError, match=match):
            ae.quant(lat, torch.zeros(bad))
        with pytest.raises(ValueError, match=match):
            ae.encode(torch.zeros(2, 12, 5023 * 3), torch.zeros(bad))


# ---- window gather ----------------------------------------------------------------------------------------------------
def _plan(A=2, K=3, T=50, W=20, O=6):
    from fdm_b200.windows import WindowPlan
    return WindowPlan(A=A, K=K, T=T, W=W, O=O, r=1)


def test_window_gather_of_per_frame_conditions():
    plan = _plan()
    A, K, n = plan.A, plan.K, 5
    assert plan.T_pad > plan.T  # the last window has padding frames
    # value = 1000 * long sequence + absolute frame
    cond = (torch.arange(A * K)[:, None, None] * 1000 + torch.arange(plan.T)[None, :, None]).expand(A * K, plan.T, n).float()
    win = plan.window_rows(cond)
    assert win.shape == (plan.n_seq, plan.W, n)
    for a in range(A):
        for w in range(plan.n_w):
            for k in range(K):
                frames = (w * plan.S + torch.arange(plan.W)).clamp(max=plan.T - 1)  # padding frames take row T - 1
                want = ((a * K + k) * 1000 + frames)[:, None].float().expand(-1, n)
                assert torch.equal(win[plan.seq(a, w, k)], want), (a, w, k)
    one = plan.window_rows(cond[:1])  # one row for every sequence
    assert one.shape == (plan.n_seq, plan.W, n)
    assert torch.equal(one[plan.seq(1, 2, 1)], win[plan.seq(0, 2, 0)])


def test_constant_schedule_gathers_like_repeat_rows():
    plan = _plan()
    ids = torch.eye(8)[: plan.A * plan.K]
    win = plan.window_rows(ids[:, None].expand(-1, plan.T, -1))
    rep = plan.window_rows(ids)
    assert torch.equal(rep, plan.repeat_rows(ids))
    assert torch.equal(win, rep[:, None].expand(-1, plan.W, -1))


def test_two_d_condition_with_as_many_rows_as_frames_stays_per_sequence():
    plan = _plan(A=1, K=4, T=4, W=20, O=6)  # T == B
    ids = torch.eye(8)[:4]
    assert torch.equal(plan.window_rows(ids), plan.repeat_rows(ids))
    assert plan.window_rows(ids).shape == (plan.n_seq, 8)


# ---- run table and tiles ----------------------------------------------------------------------------------------------
def tiles_of(runs, L, tile):
    """Restatement of the tile table fdm_vq_quantize_runs builds: (clip, l0, nrows, offset) per tile, in run order."""
    clip_run, run_l0, run_off = (t.tolist() for t in runs)
    out = []
    for b in range(len(clip_run) - 1):
        for r in range(clip_run[b], clip_run[b + 1]):
            end = run_l0[r + 1] if r + 1 < clip_run[b + 1] else L
            for l in range(run_l0[r], end, tile):
                out.append((b, l, min(tile, end - l), run_off[r]))
    return out


def _rows_of(runs, B, L):
    """Per-row offset of a run table (what the kernels must see)."""
    clip_run, run_l0, run_off = (t.tolist() for t in runs)
    rows = torch.empty(B, L, dtype=torch.int64)
    for b in range(B):
        for r in range(clip_run[b], clip_run[b + 1]):
            end = run_l0[r + 1] if r + 1 < clip_run[b + 1] else L
            rows[b, run_l0[r]:end] = run_off[r]
    return rows


def test_runs_split_at_clip_boundaries_and_frame_changes():
    from fdm_b200.vqvae import slice_runs
    off = torch.tensor([[0, 0, 256, 256, 256, 0], [0, 0, 0, 0, 0, 0], [512, 0, 512, 0, 512, 0]])
    clip_run, run_l0, run_off = slice_runs(off, fq=8)
    assert clip_run.tolist() == [0, 3, 4, 10]
    assert run_l0.tolist() == [0, 16, 40, 0, 0, 8, 16, 24, 32, 40]
    assert run_off.tolist() == [0, 256, 0, 0, 512, 0, 512, 0, 512, 0]
    # the second clip starts a run although its offset equals the previous clip's last one
    assert torch.equal(_rows_of((clip_run, run_l0, run_off), 3, 48), off.repeat_interleave(8, dim=1))


def test_one_frame_runs():
    from fdm_b200.vqvae import slice_runs
    off = (torch.arange(37) % 7 * 256)[None].repeat(2, 1)
    runs = slice_runs(off, fq=8)
    assert runs[0].tolist() == [0, 37, 74] and runs[1].tolist() == list(range(0, 37 * 8, 8)) * 2
    tl = tiles_of(runs, 37 * 8, 128)
    assert len(tl) == 74 and all(t[2] == 8 for t in tl)


@pytest.mark.parametrize("tile", [64, 128])
@pytest.mark.parametrize("run_rows", [127, 128, 129])
def test_runs_ending_at_tile_sizes(tile, run_rows):
    """A run of 127 / 128 / 129 rows (fq = 1) followed by another: no tile crosses the boundary, a run's last tile is partial."""
    from fdm_b200.vqvae import slice_runs
    L = 300
    off = torch.zeros(2, L, dtype=torch.int64)
    off[:, run_rows:] = 256
    runs = slice_runs(off, fq=1)
    assert runs[1].tolist() == [0, run_rows] * 2
    tl = tiles_of(runs, L, tile)
    assert all(t[1] // run_rows == (t[1] + t[2] - 1) // run_rows or t[1] >= run_rows for t in tl)
    first = [t for t in tl if t[0] == 0 and t[1] < run_rows]
    assert sum(t[2] for t in first) == run_rows and first[-1][2] == run_rows - tile * (len(first) - 1)
    assert sum(t[2] for t in tl) == 2 * L
    assert len(tl) <= 2 * L // 64 + 4  # fdm_vq_runs_workspace_bytes: ceil(rows / 64) + n_runs tiles at most
    cover = torch.full((2, L), -1, dtype=torch.int64)
    for b, l0, n, o in tl:
        assert (cover[b, l0:l0 + n] == -1).all()
        cover[b, l0:l0 + n] = o
    assert torch.equal(cover, off)


def test_constant_schedule_is_one_run_per_clip():
    from fdm_b200.vqvae import slice_runs
    off = torch.tensor([3, 1, 6])[:, None].expand(3, 25) * 256
    clip_run, run_l0, run_off = slice_runs(off, fq=8)
    assert clip_run.tolist() == [0, 1, 2, 3] and run_l0.tolist() == [0, 0, 0] and run_off.tolist() == [768, 256, 1536]
    # the same tiles as the per-clip kernels' own 128-row tiles of whole clips
    assert tiles_of((clip_run, run_l0, run_off), 200, 128) == [(b, l, min(128, 200 - l), o)
                                                              for b, o in enumerate([768, 256, 1536]) for l in (0, 128)]


# ---- C ABI ------------------------------------------------------------------------------------------------------------
def test_vq_runs_struct_mirrors_the_header():
    import ctypes as C
    from fdm_b200 import lib
    hdr = re.sub(r"/\*.*?\*/", "", open(HDR).read(), flags=re.S)
    body = re.search(r"typedef struct fdm_vq_runs \{(.*?)\} fdm_vq_runs;", hdr, flags=re.S).group(1)
    fields = []
    for decl in filter(None, (x.strip() for x in body.split(";"))):
        m = re.match(r"(const\s+)?(\w+)\s*(\*?)\s*(.*)", decl)
        fields.append((m.group(4).strip(), 8))
    assert [(n, C.sizeof(t)) for n, t in lib.VqRuns._fields_] == fields
    with tempfile.TemporaryDirectory() as td:
        src, exe = os.path.join(td, "s.c"), os.path.join(td, "s")
        with open(src, "w") as f:
            f.write('#include <stdio.h>\n#include "%s"\nint main(void){printf("%%zu\\n", sizeof(fdm_vq_runs));return 0;}\n' % HDR)
        subprocess.check_call(["gcc", "-o", exe, src])
        assert int(subprocess.check_output([exe])) == C.sizeof(lib.VqRuns)


def test_run_entry_points_are_bound():
    from fdm_b200 import lib
    handle = lib.load()
    for name in ("fdm_vq_quantize_runs", "fdm_vq_stats_runs", "fdm_vq_runs_workspace_bytes"):
        assert getattr(handle, name) is not None
    assert handle.fdm_abi_version() == 4
    # header + one 16-byte tile per started 64 rows and per run
    assert handle.fdm_vq_runs_workspace_bytes(2, 300, 4) == 16 + 16 * (10 + 4)
