#!/usr/bin/env python
"""Fan-out sampling against the repeated audio batch on the sample scripts' own call shape: every audio clip sampled
under K conditions, no guidance, DDIM, bf16 (split-bf16 audio encoder and tail step), full-size models, random weights.

    python tools/fanout_probe.py [--out FILE.json] [--rounds R] [--workloads vocaset,mead]

  vocaset: 64 clips x 8 identities x 4 s, 100 DDIM steps (samples/sample_diffusion_vocaset.py loops over the 8 identities)
  mead:    32 clips x 7 emotions x 8 s, 50 DDIM steps

"repeated" passes audio.repeat_interleave(K, 0) (A*K audio rows), "fanout" the A clips. One job = encode_audio, the
step- and tail-engine prepare, ddim_sample, quant, decode, each bracketed by CUDA events; the inputs are fresh device
tensors per job (no cache carries over). Jobs run in rounds of (repeated, repeated, fanout, fanout); times are medians
over all timed jobs of an arm, peak allocated memory is taken on the second job of each pair (the cached features of
the previous job are then those of the same arm, as in a loop of identical jobs). The last latents and VQ indices of the
two arms are compared bit for bit."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "face-diffusion-model_b200")]
import torch  # noqa: E402

import bench  # noqa: E402

WORKLOADS = {
    "vocaset": dict(clips=64, k=8, seconds=4.0, ddim_steps=100, cond="identity"),
    "mead": dict(clips=32, k=7, seconds=8.0, ddim_steps=50, cond="emotion"),
}


def device_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30)
        fields = [f.strip() for f in r.stdout.strip().split(",")]
        return dict(zip(q.split(","), fields)) if len(fields) == 4 else {"nvidia-smi": r.stdout.strip()}
    except Exception as e:  # the timings stand without it
        return {"nvidia-smi": repr(e)}


def run_workload(name, w, rounds, dev):
    from fdm_b200.presets import conv_out_len
    fdm, ae, diff = bench.build_models(name, dev, "bf16")
    P = fdm.preset
    A, K = w["clips"], w["k"]
    B = A * K
    n_samples = int(16000 * w["seconds"])
    N = conv_out_len(n_samples)
    N -= N % 2
    T = N // 2 if P.pair_audio else N
    shape = (B, T * P.fq, P.zdim)
    audio_host = bench.synthetic_audio(A, n_samples, 0).pin_memory()
    # sequence a*K + k: condition k of clip a (identity k for VOCASET; emotion k, the clip's own identity for MEAD)
    if P.emotion:
        emo_host = torch.eye(7)[[b % K for b in range(B)]]
        ids_host = torch.eye(P.n_id)[[(b // K) % P.n_id for b in range(B)]]
    else:
        emo_host = None
        ids_host = torch.eye(P.n_id)[[b % K for b in range(B)]]
    diff.seed, diff.clip_index0, diff.time_steps = 20261017, 0, True
    tail = fdm.precision == "bf16" and fdm.hi_tail_steps > 0

    def job(arm):
        audio = audio_host.to(dev, non_blocking=True)
        if arm == "repeated":
            audio = audio.repeat_interleave(K, 0)
        ids = ids_host.to(dev, non_blocking=True)
        emo = emo_host.to(dev, non_blocking=True) if emo_host is not None else None
        conds = (emo, ids) if P.emotion else (ids,)
        k = B // audio.shape[0]
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        ev[0].record()
        fdm.encode_audio(audio)
        ev[1].record()
        fdm.prepare(audio, T, ids, emo, fanout=k)
        if tail:
            fdm.prepare(audio, T, ids, emo, tail=True, fanout=k)
        ev[2].record()
        lat = diff.ddim_sample(audio, shape, *conds, w["ddim_steps"])  # (prepare() above is its cache hit)
        ev[3].record()
        zq, _, (_, _, idx) = ae.quant(lat, emo) if P.emotion else ae.quant(lat)
        ae.decode(zq)
        ev[4].record()
        torch.cuda.synchronize()
        t = [ev[i].elapsed_time(ev[i + 1]) for i in range(4)]
        return dict(wall_ms=ev[0].elapsed_time(ev[4]), audio_encoder_ms=t[0], prepare_ms=t[1], sampling_ms=t[2],
                    quant_decode_ms=t[3], step_ms=diff.last_step_ms,
                    peak_alloc_gb=torch.cuda.max_memory_allocated() / 1e9), lat, idx

    for arm in ("repeated", "fanout"):  # warm-up: graph capture, kernel loading, pool buffers
        job(arm)
    runs = {"repeated": [], "fanout": []}
    peaks = {"repeated": [], "fanout": []}
    last = {}
    for _ in range(rounds):
        for arm in ("repeated", "fanout"):
            for i in range(2):
                r, lat, idx = job(arm)
                runs[arm].append(r)
                if i == 1:
                    peaks[arm].append(r["peak_alloc_gb"])
                last[arm] = (lat, idx)

    def med(arm, key):
        v = sorted(r[key] for r in runs[arm])
        return v[len(v) // 2]
    keys = ("wall_ms", "audio_encoder_ms", "prepare_ms", "sampling_ms", "quant_decode_ms", "step_ms")
    arms = {arm: dict({k: round(med(arm, k), 3) for k in keys}, peak_alloc_gb=round(max(peaks[arm]), 3),
                      audio_rows=A * K if arm == "repeated" else A, timed_jobs=len(runs[arm]),
                      wall_ms_all=[round(r["wall_ms"], 2) for r in runs[arm]])
            for arm in runs}
    rep, fan = arms["repeated"], arms["fanout"]
    out = dict(workload=f"{name.upper()} {A} clips x {K} {w['cond']} conditions x {w['seconds']:g} s, {w['ddim_steps']} DDIM "
                        f"steps, no guidance, bf16 ({fdm.audio_precision} audio encoder, {fdm.hi_tail_steps} x3 tail step)",
               sequences=B, frames=T, arms=arms,
               audio_encoder_saving_ms=round(rep["audio_encoder_ms"] - fan["audio_encoder_ms"], 3),
               prepare_saving_ms=round(rep["prepare_ms"] - fan["prepare_ms"], 3),
               job_saving_ms=round(rep["wall_ms"] - fan["wall_ms"], 3),
               job_saving_frac=round(1 - fan["wall_ms"] / rep["wall_ms"], 4),
               audio_encoder_share_of_repeated_job=round(rep["audio_encoder_ms"] / rep["wall_ms"], 4),
               peak_alloc_gb_saving=round(rep["peak_alloc_gb"] - fan["peak_alloc_gb"], 3),
               outputs_bit_equal=bool(torch.equal(last["repeated"][0], last["fanout"][0])
                                      and torch.equal(last["repeated"][1], last["fanout"][1])))
    del fdm, ae, diff, last
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the result to this JSON file")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--workloads", default="vocaset,mead")
    args = ap.parse_args()
    from fdm_b200 import lib
    lib.require_device()
    dev = torch.device("cuda:0")
    res = dict(tool="tools/fanout_probe.py", device=device_info(), torch_device=torch.cuda.get_device_name(0),
               workloads={})
    for name in args.workloads.split(","):
        res["workloads"][name] = run_workload(name, WORKLOADS[name], args.rounds, dev)
        print(json.dumps({name: res["workloads"][name]}), flush=True)
    res["device_after"] = device_info()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
