#!/usr/bin/env python
"""Cost of condition schedules on the MEAD configs[3] shape (256 clips x 8 s, guidance 2.5 on the emotion, bf16).

    python tools/schedule_probe.py [--out FILE.json] [--rounds R] [--ddpm-steps S] [--quant-iters N]

Quantise (tensor path, indices + z_q in the (B, D, L) layout, CUDA events over N calls each, arms alternated call by call):
the per-clip entry point with a per-clip emotion against fdm_vq_quantize_runs with a constant schedule, one switch per clip
(at the middle frame) and a switch every 16 frames. The run tables live on the device before timing; the timed call includes
the tile-table kernel. Sampling: p_sample_loop over S DDPM steps with per-sequence against per-frame (constant schedule)
conditions, alternated round by round; the figure is the median device ms per step (diff.last_step_ms). The card's name and
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the result to this JSON file")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--ddpm-steps", type=int, default=20)
    ap.add_argument("--quant-iters", type=int, default=30)
    args = ap.parse_args()
    from fdm_b200 import lib
    from fdm_b200.presets import conv_out_len
    from fdm_b200.vqvae import slice_runs
    from utiles.classifierfree import ClassifierFreeSampleModel
    lib.require_device()
    dev = torch.device("cuda:0")
    res = dict(tool="tools/schedule_probe.py", device=device_info(), torch_device=torch.cuda.get_device_name(0))

    fdm, ae, diff = bench.build_models("mead", dev, "bf16")
    diff.denoise_fn = ClassifierFreeSampleModel(fdm, level=2.5)
    P = fdm.preset
    A, n_samples = 256, 16000 * 8
    T = conv_out_len(n_samples) // (2 if P.pair_audio else 1)
    L = T * P.fq
    shape = (A, L, P.zdim)

    # ---- quantise ----
    g = torch.Generator(device=dev).manual_seed(5)
    z = torch.randn(shape, device=dev, generator=g) * 0.05
    cb = ae.quantize.embedding.weight.detach().float().contiguous()
    emo_clip = torch.arange(A, device=dev) % 7
    per_frame = {
        "constant": emo_clip[:, None].expand(A, T),
        "one_switch": torch.where(torch.arange(T, device=dev)[None] < T // 2, emo_clip[:, None], (emo_clip[:, None] + 3) % 7),
        "every_16_frames": (emo_clip[:, None] + torch.arange(T, device=dev)[None] // 16) % 7,
    }
    runs = {k: tuple(t.to(dev) for t in slice_runs(v * 256, P.fq)) for k, v in per_frame.items()}
    off = (emo_clip * 256).contiguous()
    arms = {"per_clip": lambda: lib.vq_quantize(z, cb, 256, code_offset=off, want_bdl=True, algo=lib.VQ_TENSOR)}
    for k, r in runs.items():
        arms[k] = (lambda r=r: lib.vq_quantize_runs(z, cb, 256, r, want_bdl=True, algo=lib.VQ_TENSOR))
    for f in arms.values():  # warm-up
        f()
    ev = {k: [] for k in arms}
    for _ in range(args.quant_iters):
        for k, f in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            ev[k].append((e0, e1))
    torch.cuda.synchronize()
    q = {}
    for k, v in ev.items():
        ms = sorted(a.elapsed_time(b) for a, b in v)
        q[k] = dict(median_ms=round(ms[len(ms) // 2], 4), min_ms=round(ms[0], 4),
                    runs=int(runs[k][1].numel()) if k in runs else A)
    base = q["per_clip"]["median_ms"]
    for k in runs:
        q[k]["vs_per_clip"] = round(q[k]["median_ms"] / base - 1, 4)
    ref = arms["per_clip"]()
    same = arms["constant"]()
    q["constant_equals_per_clip"] = bool(torch.equal(ref[0], same[0]) and torch.equal(ref[1], same[1]))
    res["quant"] = dict(workload=f"MEAD {A} clips x 8 s ({T} frames, {L} latent rows per clip), D = 64, tensor path, "
                                 "indices + z_q (B, D, L)", **q)
    del z, ref, same

    # ---- sampling ----
    audio = bench.synthetic_audio(A, n_samples, 0).to(dev)
    ids = torch.eye(P.n_id)[[i % P.n_id for i in range(A)]].to(dev)
    emo = torch.eye(7, device=dev)[emo_clip]
    conds = {"per_sequence": (emo, ids), "per_frame": (emo[:, None].expand(A, T, 7).contiguous(),
                                                       ids[:, None].expand(A, T, P.n_id).contiguous())}
    diff.seed, diff.clip_index0, diff.time_steps = 20261022, 0, True
    step_range = (1000, 1000 - args.ddpm_steps)

    def job(arm):
        out = diff.p_sample_loop(shape, audio, *conds[arm], step_range=step_range)
        return diff.last_step_ms, out

    outs = {arm: job(arm)[1] for arm in conds}  # warm-up: graph capture, module loading, pooled buffers
    runs_ms = {arm: [] for arm in conds}
    for _ in range(args.rounds):
        for arm in conds:
            runs_ms[arm].append(job(arm)[0])
    med = {arm: sorted(v)[len(v) // 2] for arm, v in runs_ms.items()}
    res["sampling"] = dict(workload=f"MEAD {A} clips x 8 s ({T} frames), guidance 2.5, {args.ddpm_steps} DDPM steps, bf16",
                           ms_per_step=med, ms_per_step_all=runs_ms,
                           per_frame_vs_per_sequence=round(med["per_frame"] / med["per_sequence"] - 1, 5),
                           same_latents=bool(torch.equal(outs["per_sequence"], outs["per_frame"])))
    res["device_after"] = device_info()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
