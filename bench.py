#!/usr/bin/env python
"""bench.py - LG-LDM sampling throughput on B200 (BASELINE.json metric: animated frames/s over the full DDPM loop).

A "step" is one complete sampling job over one batch of synthetic clips: audio encoder (once) -> 1000-step DDPM
loop with classifier-free guidance (CUDA-graph replay of the fused step) -> EVQ-VAE quantise -> decode to
vertices (-> NCCL all-gather of the vertex sequences, overlapped with the decode, when N > 1).

Headline workload (the top-level `value`): BASELINE.json configs[1], "VOCASET LG-LDM sampling, batch 64 clips x 4 s with
classifier-free guidance on 1 B200"; for N > 1 every rank runs that workload on its own shard of clips (weak scaling).
`named_configs` adds, in the same JSON line, the configurations BASELINE.json names for several GPUs, STRONG-sharded:
configs[2] BIWI 128 clips x 6 s over N GPUs and configs[3] MEAD 256 clips x 8 s over N GPUs (both also at N = 1 as the
anchor of the strong-scaling curve). `microbench` (N = 1) is configs[4]: EVQ-VAE quantise / decode and HuBERT encode at
1024 clips x 10 s with a roofline per stage.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

--dump-outputs DIR writes the vertices the last timed job of the headline workload returned to DIR/vertices.npy (see
dump_vertices); inputs, weights and sampling noise are seeded, so two builds run with the same arguments can be compared
output for output.

--impl reference times the REAL reference modules (copied unmodified by __graft_entry__.build() into the git-ignored
oracle/_ref, run by oracle/ref_runner.py in a subprocess) on the host cores; without oracle/_ref it falls back to the
oracle port and says so (`cpu_baseline.kind`). build() fills oracle/_ref only when FDM_B200_REFERENCE_DIR names a
checkout of the reference, so set it there to time the reference itself.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "face-diffusion-model_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

METRIC = "animated frames/sec (full DDPM loop)"
UNIT = "frames/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--clips", type=int, default=64, help="clips per GPU of the headline workload")
    ap.add_argument("--seconds", type=float, default=4.0)
    ap.add_argument("--ddpm-steps", type=int, default=1000)
    ap.add_argument("--preset", default="vocaset", choices=["vocaset", "mead", "biwi"])
    ap.add_argument("--no-cfg", action="store_true")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--ref-sample-steps", type=int, default=20, help="DDPM steps per bounded CPU sample (extrapolation <= 50x)")
    ap.add_argument("--named", default="auto", choices=["auto", "none"], help="also run BASELINE configs[2] / configs[3], strong-sharded")
    ap.add_argument("--microbench", default="auto", choices=["auto", "none"], help="also run BASELINE configs[4] (N = 1 only)")
    ap.add_argument("--gather-chunks", type=int, default=0, help="decode / all-gather chunks (0 = automatic)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the vertices of the last timed job to DIR/vertices.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def workload_config(args, world):
    """`config` of the JSON line - shared by both arms (--impl b200 / reference) so the driver compares like with like."""
    use_cfg = not args.no_cfg
    return {"workload": (f"{args.preset.upper()} LG-LDM sampling, batch {args.clips} clips x {args.seconds:g} s "
                         f"{'with' if use_cfg else 'without'} classifier-free guidance, {args.ddpm_steps} DDPM steps, per GPU"),
            "global_clips": world * args.clips, "ddpm_steps": args.ddpm_steps, "guidance": 2.5 if use_cfg else None,
            "parallelism": f"dp{world} (clips sharded, one all-gather of vertices)"}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sustained=p["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


def build_models(preset, device, precision):
    import warnings
    warnings.simplefilter("ignore")
    torch.manual_seed(0)
    os.environ["FDM_B200_RANDOM_AUDIO_ENCODER"] = "1"  # synthetic benchmark: no checkpoint, architecture with random weights
    if preset == "vocaset":
        from models.fdm_vocaset import FDM
        from models.vq_vae_vocaset import VQAutoEncoder
        from models.utils.config import vocaset_vq_vae_args as vargs
        from video_diffusion_pytorch.diffusion_BIWI_encoder_decoder import GaussianDiffusion
        fdm = FDM(feature_dim=1024)
    elif preset == "mead":
        from models.fdm_vqvae_mead import FDM
        from models.vq_vae_emotion import VQAutoEncoder
        from utiles.args import vq_vae_args as vargs
        from video_diffusion_pytorch.diffusion_mead_encoder_decoder import GaussianDiffusion
        fdm = FDM(feature_dim=512, vertice_dim=5023 * 3, struct="Dec")
    else:
        from models.fdm import FDM
        from models.vq_vae import VQAutoEncoder
        from models.utils.config import biwi_vq_vae_args as vargs
        from video_diffusion_pytorch.diffusion_BIWI_encoder_decoder import GaussianDiffusion
        fdm = FDM(feature_dim=1024, struct="Dec")
    torch.nn.init.normal_(fdm.latent_decoder.weight, std=0.02)  # reference zero-init would make x0_hat == 0
    ae = VQAutoEncoder(vargs())
    torch.nn.init.normal_(ae.quantize.embedding.weight)
    diff = GaussianDiffusion(fdm, timesteps=1000, loss_type="l2")
    if device is not None:
        fdm.set_precision(precision)
        ae.set_precision(precision)
        diff.to(device)
        ae.to(device)
    return fdm.eval(), ae.eval(), diff.eval()


def synthetic_audio(n_clips, n_samples, clip0):
    out = torch.empty(n_clips, n_samples)
    for i in range(n_clips):
        g = torch.Generator(device="cpu").manual_seed(1234 + clip0 + i)
        a = torch.randn(n_samples, generator=g)
        out[i] = (a - a.mean()) / a.std()
    return out


DUMP_BYTES = 64_000_000


def dump_vertices(out_dir, verts):
    """verts (clips, frames, V * 3) -> out_dir/vertices.npy, float32 (c, frames, n, 3): all of it when it fits in
    DUMP_BYTES, else a fixed, seeded subset of n vertices, the same for every clip and frame (the headline workload's
    64 clips x 198 frames keep 420 of the 5023 vertices), and of c clips too when one vertex of every clip would not fit."""
    import numpy as np
    clips, frames, v3 = verts.shape
    budget = DUMP_BYTES - 1024  # room for the .npy header
    track = frames * 3 * 4  # bytes of one vertex over one clip's frames
    if track > budget:
        raise ValueError(f"--dump-outputs: one vertex of one clip over {frames} frames exceeds {DUMP_BYTES} bytes")
    g = torch.Generator().manual_seed(0)
    v = verts.view(clips, frames, v3 // 3, 3)
    c = min(clips, budget // track)
    if c < clips:
        v = v[torch.randperm(clips, generator=g)[:c].sort().values.to(v.device)]
    n = min(v3 // 3, budget // (c * track))
    if n < v3 // 3:
        v = v[:, :, torch.randperm(v3 // 3, generator=g)[:n].sort().values.to(v.device)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "vertices.npy"), v.float().cpu().numpy())


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                       "-i", str(self.idx)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons, pw = [], [], set(), []
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2])); pw.append(float(c[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = sorted(s for s, p in zip(sm, pw) if p > 0.5 * max(pw)) or sorted(sm)
        return {"sm_mhz": busy[len(busy) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                "power_w_max": max(pw)}


# --------------------------------------------------------------------------------------------------
# per-kernel timing of one eager denoiser step (roofline evidence)
# --------------------------------------------------------------------------------------------------
def profile_step(eng, sampler_args, repeats=3):
    """Times every library launch of one denoiser evaluation + fused update with CUDA events on the launching
    stream (eager, not under the graph) and aggregates by kernel class."""
    from fdm_b200 import lib
    records = []
    orig = {n: getattr(lib, n) for n in ("gemm", "layernorm", "self_attention", "ddpm_step")}

    def wrap(name):
        fn = orig[name]

        def inner(*a, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a, **k)
            e1.record()
            work = 0.0
            if name == "gemm":
                aa, w = a[0], a[1]
                M = k.get("M") or aa.shape[0]
                work = 2.0 * M * w.shape[0] * w.shape[1]
                cls = "gemm_bf16_tcgen05" if aa.dtype == torch.bfloat16 else "gemm_f32"
            elif name == "ddpm_step":
                cls = "ddpm_step"
            else:
                cls = name
            records.append((cls, work, e0, e1))
            return r
        return inner

    x_in, t_dev, ddpm = sampler_args
    lanes = getattr(eng, "lanes", 1)
    eng.lanes = 1  # serial launches on one stream: the per-kernel events must not overlap another lane's kernels
    try:
        for n in orig:
            setattr(lib, n, wrap(n))
        for _ in range(repeats):
            x0 = eng.denoise(x_in, t_dev)
            ddpm(x0)
        torch.cuda.synchronize()
    finally:
        eng.lanes = lanes
        for n, fn in orig.items():
            setattr(lib, n, fn)
    agg = {}
    for cls, work, e0, e1 in records:
        a = agg.setdefault(cls, dict(ms=0.0, work=0.0, launches=0))
        a["ms"] += e0.elapsed_time(e1)
        a["work"] += work
        a["launches"] += 1
    for a in agg.values():
        a["ms"] /= repeats
        a["work"] /= repeats
        a["launches"] //= repeats
    return agg


# --------------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the reference's own PyTorch path on the host cores
# --------------------------------------------------------------------------------------------------
def cpu_reference_real(args, n_ddpm_steps, samples, warmup_samples):
    """The REAL reference modules (oracle/_ref, copied unmodified by build()) in a subprocess - its packages have the same
    names as the drop-in's, so it gets its own interpreter. Returns the list of per-sample dicts, or None when oracle/_ref
    is absent."""
    from oracle import ref_runner
    if not ref_runner.available():
        return None
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "ref_runner.py"), args.preset, str(args.seconds), str(n_ddpm_steps),
           str(args.ddpm_steps), "0" if args.no_cfg else "1", str(os.cpu_count() or 1), str(samples), str(warmup_samples)]
    env = {k: v for k, v in os.environ.items() if k not in ("PYTHONPATH",)}
    env["CUDA_VISIBLE_DEVICES"] = ""  # the baseline is the reference's CPU path
    r = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=ROOT)
    if r.returncode != 0:
        raise RuntimeError("oracle/ref_runner.py failed:\n" + r.stderr[-2000:])
    return json.loads(r.stdout.strip().splitlines()[-1])


def cpu_reference_port(args, n_ddpm_steps, hoisted_only=False):
    """The oracle port (oracle/reference_ops.py) run the way the reference runs (B = 1, audio encoder re-evaluated inside
    every denoiser call, two denoiser calls per step with guidance) for `n_ddpm_steps` steps of one clip, plus one
    quantise + decode, extrapolated to the full chain; and the same with the audio encoder hoisted out of the loop."""
    from oracle import reference_ops as R
    torch.set_num_threads(os.cpu_count() or 1)
    fdm, ae, diff = build_models(args.preset, None, "fp32")
    P = R.PRESETS[args.preset]
    sd = {k: v.detach() for k, v in fdm.state_dict().items()}
    from transformers import HubertModel, Wav2Vec2Model
    kind = P["audio"]
    hf = (HubertModel if kind == "hubert" else Wav2Vec2Model)(R.audio_encoder_config(kind, False)).eval()
    hf.load_state_dict({k[len("audio_encoder."):]: v for k, v in sd.items() if k.startswith("audio_encoder.")})
    n_samples = int(16000 * args.seconds)
    audio = synthetic_audio(1, n_samples, 0)[0]
    idh = torch.eye(P["n_id"])[0][None]
    emo = torch.eye(7)[4][None] if P["emotion"] else None
    tabs = R.diffusion_tables(1000)
    with torch.no_grad():
        hidden = R.audio_encode(hf, audio)
        T = hidden.shape[0] // (2 if P["pair"] else 1)
        x = torch.randn(T * P["fq"], P["zdim"])

        def denoise_as_is(z, t, idh_, emo_):
            h = R.audio_encode(hf, audio)  # the reference re-runs the audio encoder in every forward
            return R.fdm_forward(sd, args.preset, h, t, z, idh_, emo_)

        def denoise_hoisted(z, t, idh_, emo_):  # the same port with the encoder run once per clip
            return R.fdm_forward(sd, args.preset, hidden, t, z, idh_, emo_)

        def step(z, t, den):
            if args.no_cfg:
                x0 = den(z, t, idh, emo)
            elif P["emotion"]:
                x0 = R.cfg_forward(lambda oh: den(z, t, idh, oh), emo, 2.5)
            else:
                x0 = R.cfg_forward(lambda oh: den(z, t, oh, None), idh, 2.5)
            return R.p_sample(tabs, x0, z, t, torch.randn_like(z))

        per_step = None
        if not hoisted_only:
            step(x, 999, denoise_as_is)  # warm-up
            t0 = time.perf_counter()
            for i in range(n_ddpm_steps):
                x = step(x, 998 - i, denoise_as_is)
            per_step = (time.perf_counter() - t0) / n_ddpm_steps
        step(x, 999, denoise_hoisted)
        t0 = time.perf_counter()
        for i in range(n_ddpm_steps):
            x = step(x, 998 - n_ddpm_steps - i, denoise_hoisted)
        per_step_hoisted = (time.perf_counter() - t0) / n_ddpm_steps
        t0 = time.perf_counter()
        enc_s = None
        R.audio_encode(hf, audio)
        enc_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        idx, zq, _ = R.vq_quantize(x, ae.quantize.embedding.weight.detach(), 4 if P["emotion"] else None)
        R.vq_decode({k: v.detach() for k, v in ae.state_dict().items()}, args.preset, zq)
        tail = time.perf_counter() - t0
    out = dict(frames=T, cores=torch.get_num_threads(), quant_decode_s=tail, s_per_step_hoisted=per_step_hoisted,
               fps_hoisted=T / (per_step_hoisted * args.ddpm_steps + tail + enc_s), sampled_steps=n_ddpm_steps)
    if per_step is not None:
        out.update(s_per_step=per_step, fps=T / (per_step * args.ddpm_steps + tail))
    return out


def cpu_baseline_block(args, n_steps, samples=1, warmup_samples=0):
    """-> (per-sample fps list, cpu_baseline dict, measured seconds per sample)."""
    use_cfg = not args.no_cfg
    how = (f"1 clip x {args.seconds:g} s, {n_steps} of {args.ddpm_steps} DDPM steps through the reference's p_sample as its sample "
           f"scripts run them (B = 1, audio encoder re-run in every denoiser call, {'2 calls/step for guidance' if use_cfg else '1 call/step'}) "
           f"+ quantise + decode, loop time extrapolated x{args.ddpm_steps / n_steps:g}")
    real = cpu_reference_real(args, n_steps, samples, warmup_samples)
    if real is not None:
        fps = [r["fps"] for r in real]
        d = real[-1]
        base = {"value": sum(fps) / len(fps), "unit": UNIT, "cores": d["cores"], "kind": "reference",
                "sample": "REAL reference modules (oracle/_ref, unmodified): " + how + f"; {d['s_per_step']:.3f} s/step",
                "s_per_ddpm_step": d["s_per_step"], "quant_decode_s": d["quant_decode_s"], "frames_per_clip": d["frames"]}
        secs = [r["sample_s"] for r in real]
    else:
        res = [cpu_reference_port(args, n_steps) for _ in range(warmup_samples + samples)][warmup_samples:]
        fps = [r["fps"] for r in res]
        d = res[-1]
        base = {"value": sum(fps) / len(fps), "unit": UNIT, "cores": d["cores"], "kind": "port",
                "sample": "oracle port (oracle/_ref absent): " + how + f"; {d['s_per_step']:.3f} s/step",
                "s_per_ddpm_step": d["s_per_step"], "quant_decode_s": d["quant_decode_s"], "frames_per_clip": d["frames"]}
        secs = [r["s_per_step"] * n_steps + r["quant_decode_s"] for r in res]
    return fps, base, secs


# --------------------------------------------------------------------------------------------------
# one sampling workload on this rank's shard
# --------------------------------------------------------------------------------------------------
class Workload:
    def __init__(self, preset, clips_local, seconds, args, rank, world, dev):
        from fdm_b200.presets import conv_out_len
        from utiles.classifierfree import ClassifierFreeSampleModel
        self.preset, self.B, self.seconds, self.args, self.rank, self.world, self.dev = preset, clips_local, seconds, args, rank, world, dev
        self.use_cfg = not args.no_cfg
        self.fdm, self.ae, self.diff = build_models(preset, dev, args.precision)
        P = self.P = self.fdm.preset
        if self.use_cfg:
            self.diff.denoise_fn = ClassifierFreeSampleModel(self.fdm, level=2.5)
        B = self.B
        n_samples = int(16000 * seconds)
        clip0 = self.clip0 = rank * B
        self.audio_host = synthetic_audio(B, n_samples, clip0).pin_memory()
        self.ids_host = torch.eye(P.n_id)[[(clip0 + i) % P.n_id for i in range(B)]].pin_memory()
        self.emo_host = torch.eye(7)[[(clip0 + i) % 7 for i in range(B)]].pin_memory() if P.emotion else None
        N = conv_out_len(n_samples)
        N -= N % 2
        self.T = T = N // 2 if P.pair_audio else N
        self.shape = (B, T * P.fq, P.zdim)
        self.diff.seed, self.diff.clip_index0, self.diff.noise_source = 20261017, clip0, "philox"
        self.diff.time_steps = True
        self.step_range = (1000, 1000 - args.ddpm_steps)
        self.V3 = V3 = self.ae.args.in_dim
        from fdm_b200.parallel import OverlappedDecodeGather
        # chunks of >= 8 clips keep the decoder's GEMMs filled; two chunks already halve the exposed tail of a 16-clip shard
        # (BIWI 128 / 8: 12.6 ms exposed with one chunk for 5.35 GB gathered)
        chunks = args.gather_chunks or max(1, min(4, B // 8))
        self.gather = OverlappedDecodeGather(chunks=chunks)
        self.gathered = torch.empty(world, B, T, V3, device=dev)  # (world = 1: simply the output buffer)
        self.verts_host = None  # pinned (B, T, V3) buffer of the end-to-end leg, allocated when that leg runs
        self.h2d_bytes = int(self.audio_host.numel() * 4 + self.ids_host.numel() * 4 + (self.emo_host.numel() * 4 if P.emotion else 0))

    def fresh_inputs(self):
        # new device tensors per job so nothing is served from the per-clip caches of a previous job
        a = self.audio_host.to(self.dev, non_blocking=True)
        i = self.ids_host.to(self.dev, non_blocking=True)
        e = self.emo_host.to(self.dev, non_blocking=True) if self.emo_host is not None else None
        return a, i, e

    def job(self, audio_dev, ids_dev, emo_dev, time_gather=False):
        P = self.P
        conds = (emo_dev, ids_dev) if P.emotion else (ids_dev,)
        lat = self.diff.sample(audio_dev, self.shape, *conds, step_range=self.step_range)
        zq, _, _ = self.ae.quant(lat, emo_dev) if P.emotion else self.ae.quant(lat)
        # decode in clip chunks straight into this rank's region of the gathered buffer; the path's only collective (one
        # NCCL all-gather per chunk) runs on a side stream while the next chunk decodes
        self.gather.run(lambda k0, k1, dst: self.ae.decode(zq, out=dst, clips=(k0, k1)), self.gathered, time_it=time_gather)
        return self.gathered[self.rank]

    def measure(self, steps, warmup, e2e=True, dump_dir=None):
        from fdm_b200 import lib
        world, dev = self.world, self.dev

        def barrier():
            if world > 1:
                import torch.distributed as dist
                dist.barrier()
            torch.cuda.synchronize()

        for _ in range(warmup):
            self.job(*self.fresh_inputs())
        barrier()
        inputs = [self.fresh_inputs() for _ in range(steps)]
        barrier()
        launches0 = lib.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        samplers = []
        for k in range(steps):
            self.job(*inputs[k], time_gather=True)
            samplers.append(self.diff.__dict__["_last_sampler"])
        e1.record()
        barrier()
        launches = lib.launch_count - launches0
        ms_dev = e0.elapsed_time(e1)
        den_ms = [s.step_ms() for s in samplers]
        gather_ms = self.gather.exposed_gather_ms()
        if dump_dir:  # before the end-to-end leg reuses the buffer; after the all-gather it holds every rank's clips
            dump_vertices(dump_dir, self.gathered.flatten(0, 1))
        ms_e2e = None
        if e2e:
            self.verts_host = torch.empty(self.B, self.T, self.V3).pin_memory()
            barrier()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            for k in range(steps):
                v = self.job(*self.fresh_inputs())
                self.verts_host.copy_(v, non_blocking=True)
            f1.record()
            barrier()
            ms_e2e = f0.elapsed_time(f1)
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms_dev, ms_e2e or 0.0, gather_ms or 0.0], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_dev, m2, gather_ms = t.tolist()
            ms_e2e = m2 if e2e else None
        frames = world * self.B * self.T * steps
        den = sorted(d for d in den_ms if d)
        return dict(value=frames / (ms_dev / 1e3), e2e=(frames / (ms_e2e / 1e3)) if ms_e2e else None, ms_per_job=ms_dev / steps,
                    ms_per_denoise_step=den[len(den) // 2] if den else None, launches=int(launches),
                    exposed_gather_ms=gather_ms if world > 1 else None)

    def roofline(self):
        """Per-kernel event timing of one eager denoiser step (rank 0)."""
        from fdm_b200 import lib
        fdm, diff, P, B, T, dev = self.fdm, self.diff, self.P, self.B, self.T, self.dev
        pk = peaks()
        eng = fdm.engine()
        a_dev, i_dev, e_dev = self.fresh_inputs()
        fdm.prepare(a_dev, T, i_dev, e_dev, guidance=(diff.denoise_fn.guidance_cond if self.use_cfg else None))
        x = torch.randn(B, T * P.d, device=dev)
        xin = x.view(B * T, P.d).to(eng.dtype)
        xbf = torch.empty(B * T, P.d, device=dev, dtype=torch.bfloat16)
        t_dev = torch.tensor([500], dtype=torch.int32, device=dev)
        use_cfg = self.use_cfg

        def ddpm(x0):
            lib.ddpm_step(x0[0], x, x, diff.posterior_mean_coef1, diff.posterior_mean_coef2, diff._sigma_table(),
                          x0_uncond=x0[1] if use_cfg else None, guidance=2.5, noise=None, out_bf16=xbf, t_dev=t_dev,
                          seed=1, clip_index0=0)
        agg = profile_step(eng, (xin, t_dev, ddpm))
        tot_ms = sum(a["ms"] for a in agg.values())
        shares = {k: round(a["ms"] / tot_ms, 4) for k, a in agg.items()}
        g = agg.get("gemm_bf16_tcgen05") or agg.get("gemm_f32")
        tf = g["work"] / (g["ms"] / 1e3) / 1e12
        traffic, traffic_note = None, None
        tpath = os.path.join(ROOT, "profiles", "gemm_traffic.json")
        if os.path.exists(tpath) and "gemm_bf16_tcgen05" in agg and self.preset == "vocaset":
            with open(tpath) as f:
                tj = json.load(f)
            traffic, traffic_note = tj["mean_dram_bytes_per_launch"], tj["source"]
        roof = {"bound": "tensor", "kernel": "gemm_tc_kernel (fdm_gemm_bf16)" if "gemm_bf16_tcgen05" in agg else "gemm_f32_kernel",
                "achieved": tf, "peak": pk["tf_sustained"], "unit": "TFLOP/s", "frac": tf / pk["tf_sustained"],
                "peak_source": f"{pk['src']} sustained bf16 cuBLAS (kernel timed inside the step)", "traffic": traffic,
                "traffic_unit": "DRAM bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)", "traffic_source": traffic_note,
                "flops_per_launch": g["work"] / max(g["launches"], 1),
                "launches_per_denoise_step": g["launches"], "ms_per_denoise_step_in_kernel": g["ms"]}
        d = agg["ddpm_step"]
        elems = B * T * P.d
        bytes_alg = elems * ((4 * 4 if use_cfg else 3 * 4) + 2)  # x0c,(x0u),x_t reads + fp32 write + bf16 copy; noise in-kernel
        extra = {"ddpm_step_kernel": {"bound": "hbm", "achieved": bytes_alg / (d["ms"] / 1e3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                                      "frac": bytes_alg / (d["ms"] / 1e3) / 1e9 / pk["hbm"], "bytes_per_launch": bytes_alg},
                 "kernel_time_shares_eager_step": shares, "eager_step_ms": tot_ms,
                 "kernel_ms_eager_step": {k: round(a["ms"], 4) for k, a in agg.items()}}
        return roof, extra, eng.flops_per_step()

    def free(self):
        for n in ("fdm", "ae", "diff", "gathered", "verts_host", "audio_host"):
            setattr(self, n, None)
        import gc
        gc.collect()
        torch.cuda.empty_cache()


# --------------------------------------------------------------------------------------------------
# BASELINE configs[4]: once-per-clip stages at 1024 clips x 10 s (N = 1)
# --------------------------------------------------------------------------------------------------
def microbench(dev, args):
    from fdm_b200 import lib
    from fdm_b200.presets import conv_out_len
    pk = peaks()
    clips, batch, seconds = 1024, 64, 10.0
    fdm, ae, diff = build_models("vocaset", dev, "bf16")
    P = fdm.preset
    n_samples = int(16000 * seconds)
    N = conv_out_len(n_samples)
    N -= N % 2
    T = N

    def timed(fn, n, warm=1):
        for i in range(warm):
            fn(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    out = {"workload": f"configs[4]: {clips} clips x 10 s, VOCASET preset ({T} frames, {T * P.fq} latent rows per clip)"}
    # ---- EVQ-VAE quantise: all 8 159 232 rows in one launch, tensor-core filter + exact recheck ----
    L, D, codes = T * P.fq, P.zdim, 256
    cb = ae.quantize.embedding.weight.detach().float().contiguous()
    z = torch.randn(clips, L, D, device=dev)
    rows = clips * L
    vq = {}
    for name, want_zq in (("indices_only", False), ("indices_and_zq", True)):
        ms = timed(lambda i: lib.vq_quantize(z, cb, codes, want_bdl=want_zq, algo=lib.VQ_TENSOR), 10, warm=2) / 10
        alg = rows * (4 * D + 8 + (4 * D if want_zq else 0))
        vq[name] = {"ms": ms, "algorithmic_bytes": alg, "achieved": alg / ms / 1e6, "unit": "GB/s", "peak": pk["hbm"],
                    "frac": alg / ms / 1e6 / pk["hbm"], "bound": "hbm"}
    cnt = torch.zeros(1, dtype=torch.int64, device=dev)
    idx_t, _, _ = lib.vq_quantize(z, cb, codes, want_bdl=False, algo=lib.VQ_TENSOR, recheck_rows=cnt)
    idx_f, _, _ = lib.vq_quantize(z, cb, codes, want_bdl=False, algo=lib.VQ_FFMA)
    vq["tensor_equals_ffma_all_rows"] = bool(torch.equal(idx_t, idx_f))  # (the FFMA kernel is held to the CPU oracle by the tests)
    vq["recheck_row_fraction"] = cnt.item() / rows
    vq["rows"] = rows
    sweep = []
    for n in (16, 64, 256, 1024):
        zs = z[:n]
        ms = timed(lambda i: lib.vq_quantize(zs, cb, codes, want_bdl=True, algo=lib.VQ_TENSOR), 20, warm=3) / 20
        alg = n * L * (8 * D + 8)
        sweep.append({"clips": n, "ms": ms, "GBps": alg / ms / 1e6, "frac": alg / ms / 1e6 / pk["hbm"]})
    vq["sweep_indices_and_zq"] = sweep
    del idx_t, idx_f
    # ---- through the public API: quant() (indices + z_q (B,D,L) + rows for the decoder + loss / perplexity by-products) ----
    lat = z[:batch]
    keep = []

    def run_quant(i):
        keep[:] = [ae.quant(lat)[0]]
    ms = timed(run_quant, clips // batch)
    alg = rows * (4 * D + 8 + 2 * 4 * D)
    vq["quant_api"] = {"ms": ms, "achieved": alg / ms / 1e6, "unit": "GB/s", "frac": alg / ms / 1e6 / pk["hbm"]}
    out["vq_quantize"] = vq
    # ---- EVQ-VAE decode ----
    ms = timed(lambda i: ae.decode(keep[0]), clips // batch)
    fl = 71.6e9 * clips  # SURVEY section 8(a) D1 at T = 498
    out["vq_decode"] = {"ms": ms, "clips_per_s": clips / ms * 1e3, "achieved": fl / ms / 1e9, "unit": "TFLOP/s", "peak": pk["tf_sustained"],
                        "frac": fl / ms / 1e9 / pk["tf_sustained"], "bound": "tensor"}
    del z, keep
    # ---- the BIWI latent width (D = 128, models/utils/config.py:44-60): 1024 clips x 6 s x 8 latent rows per frame ----
    B2, L2, D2 = 1024, 149 * 8, 128
    g2 = torch.Generator(device="cpu").manual_seed(7)
    cb2 = (torch.randn(codes, D2, generator=g2) * 0.5).to(dev)
    z2 = torch.randn(B2, L2, D2, device=dev)
    d128 = {"rows": B2 * L2}
    for name, algo, reps in (("tensor", lib.VQ_TENSOR, 10), ("ffma", lib.VQ_FFMA, 2)):
        ms = timed(lambda i: lib.vq_quantize(z2, cb2, codes, want_bdl=True, algo=algo), reps, warm=1) / reps
        alg = B2 * L2 * (8 * D2 + 8)
        d128[name] = {"ms": ms, "achieved": alg / ms / 1e6, "unit": "GB/s", "peak": pk["hbm"], "frac": alg / ms / 1e6 / pk["hbm"],
                      "bound": "hbm"}
    i_t, _, _ = lib.vq_quantize(z2, cb2, codes, want_bdl=False, algo=lib.VQ_TENSOR)
    i_f, _, _ = lib.vq_quantize(z2, cb2, codes, want_bdl=False, algo=lib.VQ_FFMA)
    d128["tensor_equals_ffma_all_rows"] = bool(torch.equal(i_t, i_f))
    out["vq_quantize"]["biwi_d128_indices_and_zq"] = d128
    del z2, i_t, i_f
    # ---- HuBERT-large encode (bf16 throughput mode; and the split-bf16 mode the sampler uses by default) ----
    audios = [synthetic_audio(batch, n_samples, 0).to(dev) for _ in range(2)]
    fl = 383.1e9  # per clip at 10 s (SURVEY section 8(a) A1)
    for mode, n_clips in (("bf16", clips), ("x3", 256)):
        fdm.audio_precision = mode
        ms = timed(lambda i: fdm.encode_audio(audios[i % 2].clone()), n_clips // batch)
        eff = fl * n_clips * (3 if mode == "x3" else 1)
        out[f"hubert_encode_{mode}"] = {"ms": ms, "clips": n_clips, "clips_per_s": n_clips / ms * 1e3, "achieved": fl * n_clips / ms / 1e9,
                                        "executed_tensor_TFLOPs": eff / ms / 1e9, "unit": "TFLOP/s", "peak": pk["tf_sustained"],
                                        "frac": fl * n_clips / ms / 1e9 / pk["tf_sustained"], "bound": "tensor"}
    return out


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    use_cfg = not args.no_cfg
    config = workload_config(args, world)

    if args.impl == "reference":
        if rank != 0:
            return
        fps, base, secs = cpu_baseline_block(args, args.ref_sample_steps, samples=args.steps, warmup_samples=args.warmup)
        v = sum(fps) / len(fps)
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sum(secs) / len(secs), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "note": "a step = one bounded sample of the workload (see cpu_baseline.sample); ms_per_step is its measured time, "
                    "value the frames/s of a full job extrapolated from it",
            "cpu_baseline": base,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return

    from fdm_b200 import lib
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    lib.require_device()
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    wl = Workload(args.preset, args.clips, args.seconds, args, rank, world, dev)
    m = wl.measure(args.steps, args.warmup, e2e=True, dump_dir=args.dump_outputs if rank == 0 else None)
    clocks = sampler.stop() if rank == 0 else None
    roof, extra, flops = (None, {}, None)
    if rank == 0:
        roof, extra, flops = wl.roofline()
        extra["denoiser_tflops_in_loop"] = flops / (m["ms_per_denoise_step"] / 1e3) / 1e12 if m["ms_per_denoise_step"] else None
    d2h = int(wl.verts_host.numel() * 4)
    h2d = wl.h2d_bytes
    T_main = wl.T
    lanes = wl.fdm.engine().lanes if use_cfg else 1
    tail_steps, audio_mode = wl.fdm.hi_tail_steps, wl.fdm._audio_mode()
    wl.free()

    # ---- BASELINE configs[2] / configs[3], strong-sharded over the N ranks --------------------------------------------
    named = []
    if args.named == "auto" and args.preset == "vocaset" and args.clips == 64 and args.ddpm_steps == 1000:
        for label, preset, total, seconds in (("configs[2]: BIWI LG-LDM sampling (23370-vertex mesh), batch 128 clips x 6 s", "biwi", 128, 6.0),
                                              ("configs[3]: 3D MEAD emotional LG-LDM sampling (7 emotions, local+global codebooks), batch 256 clips x 8 s", "mead", 256, 8.0)):
            if total % world != 0:
                continue
            w2 = Workload(preset, total // world, seconds, args, rank, world, dev)
            r = w2.measure(2 if world > 1 else 1, 1, e2e=False)
            blk = {"config": f"{label}, sharded over {world} GPU(s): {total // world} clips per GPU, guidance 2.5, 1000 DDPM steps",
                   "scaling": "strong", "n_gpus": world, "global_clips": total, "frames_per_clip": w2.T, "value": r["value"], "unit": UNIT,
                   "ms_per_job": r["ms_per_job"], "ms_per_denoise_step": r["ms_per_denoise_step"], "exposed_gather_ms": r["exposed_gather_ms"],
                   "gather_bytes_per_rank": int(w2.B * w2.T * w2.V3 * 4)}
            if rank == 0:
                rf, ex, fl = w2.roofline()
                blk["gemm_roofline_frac"] = rf["frac"]
                blk["gemm_TFLOPs"] = rf["achieved"]
                blk["kernel_time_shares_eager_step"] = ex["kernel_time_shares_eager_step"]
                blk["denoiser_tflops_in_loop"] = fl / (r["ms_per_denoise_step"] / 1e3) / 1e12 if r["ms_per_denoise_step"] else None
            named.append(blk)
            w2.free()

    micro = None
    if rank == 0 and world == 1 and args.microbench == "auto" and args.preset == "vocaset":
        micro = microbench(dev, args)

    cpu_base = None
    if rank == 0 and world == 1 and not args.skip_cpu_baseline:
        _, cpu_base, _ = cpu_baseline_block(args, args.ref_sample_steps, samples=1, warmup_samples=0)
        try:
            port = cpu_reference_port(args, 4, hoisted_only=True)
            cpu_base["audio_encoder_hoisted"] = {"value": port["fps_hoisted"], "unit": UNIT, "s_per_ddpm_step": port["s_per_step_hoisted"],
                                                 "kind": "port", "note": "oracle port with the audio encoder run once per clip instead of in every "
                                                                         "denoiser call (4 DDPM steps, extrapolated)"}
        except Exception as e:  # the headline baseline above stands on its own
            cpu_base["audio_encoder_hoisted"] = {"error": str(e)[:200]}

    if rank == 0:
        detail = dict(config)
        detail.update({"frames_per_clip": T_main, "noise": "in-kernel Philox4x32-10 keyed by global clip index",
                       "denoiser_lanes": lanes, "high_precision_tail_steps": tail_steps, "audio_encoder_precision": audio_mode,
                       "l2": "inputs larger than L2: every denoise step streams > 1.4 GB of activations, weights and cross-attention "
                             "caches through the 126 MB L2, each job starts from fresh input tensors and ends with a 764 MB vertex "
                             "write; no explicit flush is needed between timed jobs"})
        line = {
            "metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": m["ms_per_job"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.precision, "data": "synthetic", "config": config, "config_detail": detail,
            "ms_per_denoise_step": m["ms_per_denoise_step"], "exposed_gather_ms": m["exposed_gather_ms"],
            "clocks": clocks,
            "e2e": {"value": m["e2e"], "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": m["launches"],
            "roofline": roof, "cpu_baseline": cpu_base, "named_configs": named, "microbench": micro,
        }
        line.update(extra)
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
