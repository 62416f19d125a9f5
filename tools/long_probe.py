#!/usr/bin/env python
"""Long audio: sample_long against the serial continuation recipe, on the same audio (VOCASET, guidance 2.5, bf16, DDPM
over the preset's default range).

    python tools/long_probe.py [--out FILE.json] [--rounds R] [--seconds S] [--clips 1,16]

(a) sample_long: the windows (420 frames, 60 shared, default) of all clips as one batch, blended after every step.
(b) the continuation recipe of INTEGRATION.md: one sample() call per window, window w + 1 with window w's last 60 frames
    as known frames, windows one after another; its audio slices are the ones (a) uses.
Each job starts from a fresh copy of the audio tensor, so both arms run the audio encoder inside the job. A job is timed
with the host clock between two device synchronisations. Arms alternate round by round after one warm-up job each; the
figure is the median over rounds. ms per step is the job time over the denoising steps the job runs (arm (b) runs one
step list per window). The card's name and power limit are read in the same run."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "face-diffusion-model_b200"), os.path.join(ROOT, "tools")]
import torch  # noqa: E402

import bench  # noqa: E402
from fanout_probe import device_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the result to this JSON file")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=60.0)
    ap.add_argument("--clips", default="1,16")
    args = ap.parse_args()
    from fdm_b200 import lib
    from fdm_b200.presets import conv_out_len
    from fdm_b200.windows import plan_windows
    from utiles.classifierfree import ClassifierFreeSampleModel
    lib.require_device()
    dev = torch.device("cuda:0")
    res = dict(tool="tools/long_probe.py", device=device_info(), torch_device=torch.cuda.get_device_name(0), runs={})

    fdm, ae, diff = bench.build_models("vocaset", dev, "bf16")
    diff.denoise_fn = ClassifierFreeSampleModel(fdm, level=2.5)
    P = fdm.preset
    hi, lo = diff.default_range
    n_steps = hi - lo
    diff.seed, diff.clip_index0 = 20261022, 0
    for A in (int(c) for c in args.clips.split(",")):
        n_samples = int(16000 * args.seconds)
        T = conv_out_len(n_samples)
        shape = (A, T * P.fq, P.zdim)
        audio = bench.synthetic_audio(A, n_samples, 0).to(dev)
        ids = torch.eye(P.n_id)[[i % P.n_id for i in range(A)]].to(dev)
        plan = plan_windows(P, shape, A, n_samples)
        W, O, S, n_w = plan.W, plan.O, plan.S, plan.n_w
        wshape = (A, W * P.fq, P.zdim)
        mask = torch.arange(W, device=dev) < O

        def long_job(a):
            return diff.sample_long(a, shape, ids)

        def serial_job(a):
            slices = plan.window_audio(a).view(A, n_w, -1)
            pieces, prev = [], None
            for w in range(n_w):
                aw = slices[:, w].contiguous()
                if prev is None:
                    lat = diff.sample(aw, wshape, ids)
                else:
                    known = torch.zeros(wshape, device=dev)
                    known[:, :O * P.fq] = prev[:, -O * P.fq:]
                    lat = diff.sample(aw, wshape, ids, known=known, known_mask=mask)
                pieces.append(lat if w == n_w - 1 else lat[:, :S * P.fq])
                prev = lat
            return torch.cat(pieces, 1)[:, :T * P.fq]

        arms = {"sample_long": (long_job, n_steps), "serial_continuation": (serial_job, n_steps * n_w)}

        def timed(fn):
            a = audio.clone()  # a new tensor: the audio encoder runs inside the job
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = fn(a)
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) * 1e3, out

        for name, (fn, _) in arms.items():  # warm-up: graph capture, module loading, pooled buffers
            assert timed(fn)[1].shape == shape
        ms = {name: [] for name in arms}
        for _ in range(args.rounds):
            for name, (fn, _) in arms.items():
                ms[name].append(timed(fn)[0])
        row = dict(workload=f"VOCASET {A} clip(s) x {args.seconds:g} s ({T} frames), guidance 2.5, bf16, DDPM t = {hi - 1}..{lo} "
                            f"({n_steps} steps), windows of {W} frames sharing {O} ({n_w} per clip)")
        for name, (fn, steps) in arms.items():
            med = sorted(ms[name])[len(ms[name]) // 2]
            row[name] = dict(ms_per_job=round(med, 1), ms_per_job_all=[round(x, 1) for x in ms[name]],
                             denoising_steps=steps, ms_per_step=round(med / steps, 4),
                             frames_per_s=round(A * T / med * 1e3, 1))
        row["job_time_ratio_serial_over_long"] = round(row["serial_continuation"]["ms_per_job"] / row["sample_long"]["ms_per_job"], 3)
        res["runs"][f"{A}x{args.seconds:g}s"] = row
        print(json.dumps(row), flush=True)
    res["device_after"] = device_info()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
