#!/usr/bin/env python
"""Cost of known frames on the headline workload (BASELINE configs[1]: VOCASET 64 clips x 4 s, guidance 2.5, DDPM, bf16).

    python tools/known_probe.py [--out FILE.json] [--rounds R] [--ddpm-steps S] [--kernel-iters N]

Sampling arms, alternated round by round: no known frames, the first 25 % of every sequence's frames known (a
continuation prefix), all frames known. Each job runs p_sample_loop over S DDPM steps (t = 999 .. 1000 - S) and reads
the median device time per step from the CUDA events around every graph replay (diff.last_step_ms); the arm's figure is
the median over its jobs. The known_frames kernel is then timed on its own with CUDA events over N back-to-back launches
on the same (64, 3168, 64) state, Philox noise, with the bf16 copy, at 25 % and 100 % of the frames. The card's name and
power limit are read in the same run."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "face-diffusion-model_b200"), os.path.join(ROOT, "tools")]
import torch  # noqa: E402

import bench  # noqa: E402
from fanout_probe import device_info  # noqa: E402

ARMS = {"none": None, "25%": 0.25, "100%": 1.0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the result to this JSON file")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--ddpm-steps", type=int, default=100)
    ap.add_argument("--kernel-iters", type=int, default=200)
    args = ap.parse_args()
    from fdm_b200 import lib
    from fdm_b200.presets import conv_out_len
    from utiles.classifierfree import ClassifierFreeSampleModel
    lib.require_device()
    dev = torch.device("cuda:0")
    res = dict(tool="tools/known_probe.py", device=device_info(), torch_device=torch.cuda.get_device_name(0))

    fdm, ae, diff = bench.build_models("vocaset", dev, "bf16")
    diff.denoise_fn = ClassifierFreeSampleModel(fdm, level=2.5)
    P = fdm.preset
    A, n_samples = 64, 16000 * 4
    N = conv_out_len(n_samples)
    T = N - N % 2
    shape = (A, T * P.fq, P.zdim)
    audio = bench.synthetic_audio(A, n_samples, 0).to(dev)
    ids = torch.eye(P.n_id)[[i % P.n_id for i in range(A)]].to(dev)
    diff.seed, diff.clip_index0, diff.time_steps = 20261017, 0, True
    known = torch.randn(shape, generator=torch.Generator().manual_seed(1)).to(dev)
    masks = {k: None if f is None else (torch.arange(T, device=dev) < round(f * T)).expand(A, T).contiguous()
             for k, f in ARMS.items()}
    step_range = (1000, 1000 - args.ddpm_steps)

    def job(arm):
        kw = {} if masks[arm] is None else dict(known=known, known_mask=masks[arm])
        diff.p_sample_loop(shape, audio, ids, step_range=step_range, **kw)
        return diff.last_step_ms

    for arm in ARMS:  # warm-up: graph capture, module loading, pooled buffers
        job(arm)
    runs = {arm: [] for arm in ARMS}
    for _ in range(args.rounds):
        for arm in ARMS:
            runs[arm].append(job(arm))
    med = {arm: sorted(v)[len(v) // 2] for arm, v in runs.items()}
    base = med["none"]
    res["sampling"] = dict(workload=f"VOCASET {A} clips x 4 s ({T} frames), guidance 2.5, {args.ddpm_steps} DDPM steps, bf16",
                           ms_per_step=med, ms_per_step_all=runs,
                           overhead_frac={arm: round(med[arm] / base - 1, 5) for arm in ARMS if arm != "none"})

    # the kernel alone, on the sampler's own shapes
    x = torch.randn(shape, device=dev)
    xb = torch.empty(shape, device=dev, dtype=torch.bfloat16)
    ka = torch.full((2,), 0.5, device=dev)
    kb = torch.full((2,), 0.5, device=dev)
    index = torch.zeros(1, dtype=torch.int32, device=dev)
    seed_dev = torch.tensor([7], dtype=torch.int64, device=dev)
    t_dev = torch.tensor([500], dtype=torch.int32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # larger than L2: each timed pass starts cold
    kern = {}
    for arm in ("25%", "100%"):
        m = masks[arm].to(torch.uint8).reshape(-1).contiguous()
        rows = int(m.sum())
        for _ in range(3):
            lib.known_frames(x, known, m, ka, kb, index, x_bf16=xb, seed_dev=seed_dev, t_dev=t_dev)
        times = []
        for _ in range(args.kernel_iters):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            lib.known_frames(x, known, m, ka, kb, index, x_bf16=xb, seed_dev=seed_dev, t_dev=t_dev)
            e1.record()
            times.append((e0, e1))
        torch.cuda.synchronize()
        us = sorted(a.elapsed_time(b) * 1e3 for a, b in times)
        t_us = us[len(us) // 2]
        nbytes = rows * P.d * (4 + 4 + 2) + m.numel()  # known read, fp32 and bf16 state written, mask bytes
        kern[arm] = dict(known_rows=rows, median_us=round(t_us, 2), min_us=round(us[0], 2),
                         bytes=nbytes, gb_per_s=round(nbytes / t_us / 1e3, 1),
                         share_of_step=round(t_us / 1e3 / base, 5))
    res["kernel"] = dict(note="event-timed single launches, L2 flushed before each, Philox noise, bf16 copy on", **kern)
    res["device_after"] = device_info()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
