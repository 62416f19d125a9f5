"""Sampling-loop engine: the DDPM ancestral loop (and DDIM) as a CUDA-graph replay of one fused step.

Replaces GaussianDiffusion.p_sample_loop / p_sample / p_mean_variance / q_posterior (reference
video_diffusion_pytorch/diffusion_mead_encoder_decoder.py:632-671, diffusion_BIWI_encoder_decoder.py:632-710).
One step = DenoiserEngine.denoise (all layers) + ONE fused update kernel (CFG combine + posterior mean + noise
add, csrc/ddpm.cu) + a 1-thread kernel that advances the device-resident step counter; nothing in a step
touches the host, so the whole step is captured once and replayed for every t.
"""
from __future__ import annotations

import os
from typing import Callable, NamedTuple, Optional, Sequence, Union

import torch

from . import lib
from .denoiser import DenoiserEngine

NoiseSpec = Union[None, str, Callable[[int], torch.Tensor]]


class KnownFrames(NamedTuple):
    """Known frames of a sampling call, in pooled buffers of the denoiser engine (stable addresses: new known data of the
    same shape is no reason to capture new step graphs). Rows whose mask is set take ka[s] * latent + kb[s] * z at state s
    (0 = start, s + 1 = after step s; the last entry is (1, 0)), see fdm_known_frames."""
    latent: torch.Tensor  # (B, fq*T, zdim) fp32
    mask: torch.Tensor    # (B*T,) uint8, one entry per frame (denoiser row)
    ka: torch.Tensor      # (len(steps) + 1,) fp32
    kb: torch.Tensor


def pool_known(den: DenoiserEngine, latent: torch.Tensor, mask: torch.Tensor, ka: torch.Tensor, kb: torch.Tensor) -> KnownFrames:
    """Copy a call's known frames (latent broadcastable to (den.B, fq*T, zdim), mask to (den.B, den.T), host tables)
    into the engine's pooled buffers."""
    B, T, d = den.B, den.T, den.P.d
    dev = den.dev
    lat = den.buf("smp_known", (B, T * den.P.fq, d // den.P.fq), torch.float32, dev)
    lat.copy_(latent)
    m = den.buf("smp_known_mask", (B * T,), torch.uint8, dev)
    m.view(B, T).copy_(mask)
    kab = den.buf("smp_known_ab", (2, ka.numel()), torch.float32, dev)
    kab.copy_(torch.stack([ka, kb]).to(torch.float32))
    return KnownFrames(lat, m, kab[0], kab[1])


class SamplerEngine:
    def __init__(self, denoiser: DenoiserEngine, c1: torch.Tensor, c2: torch.Tensor, sigma: torch.Tensor,
                 guidance_level: Optional[float] = None):
        self.den = denoiser
        self.c1, self.c2, self.sigma = c1, c2, sigma
        self.level = guidance_level
        self.last_step_ms = None
        self._step_events = None
        self.steps_per_graph = int(os.environ.get("FDM_B200_STEPS_PER_GRAPH", "10"))

    def step_ms(self):
        """Median device time of one denoising step of the last run(time_steps=True), from the CUDA events recorded around
        every graph replay (waits for the last of them)."""
        if self._step_events is not None:
            evs, unroll = self._step_events
            evs[-1].synchronize()
            ms = sorted(evs[i].elapsed_time(evs[i + 1]) / unroll for i in range(len(evs) - 1))
            self.last_step_ms = ms[len(ms) // 2]
            self._step_events = None
        return self.last_step_ms

    @torch.no_grad()
    def run(self, x_T: torch.Tensor, steps: Sequence[int], noise: NoiseSpec = "philox", seed: int = 0,
            clip_index0: int = 0, graph: bool = True, tap: Optional[Callable[[int, torch.Tensor], None]] = None,
            time_steps: bool = False, ddim: Optional[dict] = None, tail=None,
            known: Optional[KnownFrames] = None) -> torch.Tensor:
        """x_T (B, fq*T, zdim) fp32 on device; steps: the t values in execution order (e.g. 999..0).
        noise: "philox" (in-kernel counter-based generator), or a callable t -> tensor (host- or device-side,
        same shape as x_T) that is copied in before every step with t > 0 (parity runs).
        ddim: None for the ancestral (DDPM) update, or per-step device tables {a_recip, a_recipm1, sqrt_an, c} (one
        entry per element of `steps`) for the deterministic DDIM update (eta = 0, no noise).
        tail: None, or (DenoiserEngine prepared for the same clip batch, n): the LAST n steps evaluate the denoiser on that
        (high-precision, fp32-activation) engine, eagerly, after the graph-replayed bf16 steps - the final latent is the
        last denoiser output, so its precision is what the quantiser sees (profiles/r02_precision_probe.json).
        known: None, or KnownFrames (pool_known): the start state and the state after every step are replaced on the known
        rows (one fdm_known_frames launch after each step's update). Its z is the draw the update used at that element:
        the host noise buffer, or Philox at (seed, clip_index0 + b, t); after the last step the known rows hold
        `known.latent` bit for bit."""
        den = self.den
        B, T, d, S = den.B, den.T, den.P.d, den.passes
        assert x_T.is_cuda and x_T.dtype == torch.float32 and x_T.numel() == B * T * d, "x_T does not match prepare()"
        assert (S == 2) == (self.level is not None), "guidance passes and guidance level disagree"
        dev = x_T.device
        steps = list(steps)
        # loop state lives in the denoiser engine's persistent buffers: same shapes -> same addresses -> cached graphs
        x = den.buf("smp_x", tuple(x_T.shape), torch.float32, dev)
        xin_bf = den.buf("smp_xin_bf", (B * T, d), torch.bfloat16, dev) if den.dtype == torch.bfloat16 else None
        xin = xin_bf if xin_bf is not None else x.view(B * T, d)
        sched = den.buf("smp_sched", (len(steps),), torch.int32, dev)
        sched.copy_(torch.tensor(steps, dtype=torch.int32), non_blocking=False)
        cursor = den.buf("smp_cursor", (1,), torch.int32, dev)
        t_dev = den.buf("smp_t", (1,), torch.int32, dev)
        seed_dev = den.buf("smp_seed", (1,), torch.int64, dev)  # Philox seed in device memory: the cached graphs survive a new seed
        seed_dev.fill_(int(seed))
        tail_den, n_tail = tail if tail is not None else (None, 0)
        n_tail = min(n_tail, len(steps))
        if tail_den is not None:
            assert (tail_den.B, tail_den.T, tail_den.passes) == (B, T, S) and tail_den.dtype == torch.float32
        host_noise = callable(noise) and ddim is None
        noise_buf = den.buf("smp_noise", tuple(x_T.shape), torch.float32, dev) if host_noise else None
        assert host_noise or ddim is not None or noise in (None, "philox")
        if known is not None:
            assert known.latent.shape == x.shape and known.mask.numel() == B * T and known.ka.numel() == len(steps) + 1

        def replace_known(offset: int, z=None):
            lib.known_frames(x, known.latent, known.mask, known.ka, known.kb, cursor, offset=offset, noise=z, x_bf16=xin_bf,
                             seed_dev=seed_dev, t_dev=t_dev, clip_index0=clip_index0)

        def step_body(hi: bool = False):
            x0 = tail_den.denoise(x.view(B * T, d), t_dev) if hi else den.denoise(xin, t_dev)
            if ddim is None:
                lib.ddpm_step(x0[0], x, x, self.c1, self.c2, self.sigma, x0_uncond=x0[1] if S == 2 else None,
                              guidance=float(self.level) if S == 2 else 0.0, noise=noise_buf, out_bf16=xin_bf, t_dev=t_dev,
                              seed_dev=seed_dev, clip_index0=clip_index0)
            else:
                lib.ddim_step(x0[0], x, x, ddim["a_recip"], ddim["a_recipm1"], ddim["sqrt_an"], ddim["c"], cursor,
                              x0_uncond=x0[1] if S == 2 else None, guidance=float(self.level) if S == 2 else 0.0,
                              out_bf16=xin_bf)
            if known is not None:  # state after step `cursor`: table entry cursor + 1
                replace_known(1, noise_buf)
            lib.advance_cursor(cursor, sched, t_dev)

        def reset():
            x.copy_(x_T.reshape(x.shape))
            if xin_bf is not None:
                lib.cast(x, xin_bf.view(x.shape))
            cursor.zero_()
            t_dev.copy_(sched[:1])
            if known is not None:  # start state at the first step's noise level, from x_T's own values
                replace_known(0, x)

        def feed_noise(t):
            if host_noise and t > 0:
                n = noise(t)
                noise_buf.copy_(n.reshape(noise_buf.shape), non_blocking=True)

        main_steps = steps[: len(steps) - n_tail]
        tail_steps = steps[len(steps) - n_tail:]
        all_steps, steps = steps, main_steps  # (the device schedule holds every step; the graph loop runs the main ones)
        use_graph = graph and tap is None
        if use_graph and not steps:
            reset()
        elif use_graph:
            # Steps per graph: the step body is the same for every t (t and the schedule cursor live on the device), so
            # when no host data is fed per step several steps are captured back to back in one graph: a slow or busy host
            # then costs one launch per `unroll` steps instead of one per step (measured on a shared box: 880 ms of
            # launch gaps per 1000-step job with one step per replay).
            unroll = 1 if host_noise else max(1, min(int(self.steps_per_graph), len(steps)))
            n_rep, rem = divmod(len(steps), unroll)
            # Captured graphs are cached on the denoiser engine, keyed by every address and scalar baked into their nodes
            # (instantiating a 740-node graph costs tens of ms: 18 % of a MEAD job, 3 % of a VOCASET job).
            ddim_key = None if ddim is None else tuple(sorted((k, v.data_ptr()) for k, v in ddim.items()))
            key = (unroll, S, B, T, seed_dev.data_ptr(), clip_index0, self.level, den.pack_serial, den.lanes, host_noise, ddim_key,
                   x.data_ptr(), xin.data_ptr(), sched.data_ptr(), cursor.data_ptr(), t_dev.data_ptr(),
                   None if noise_buf is None else noise_buf.data_ptr(), self.c1.data_ptr(), self.c2.data_ptr(),
                   self.sigma.data_ptr(), den.x.data_ptr(), den.qkv.data_ptr(), den.att.data_ptr(), den.proj.data_ptr(),
                   den.ffn.data_ptr(), den.x0.data_ptr(), tuple(c.data_ptr() for c in den.cross),
                   tuple(a.data_ptr() for a in den.addend))
            if known is not None:
                key += (known.latent.data_ptr(), known.mask.data_ptr(), known.ka.data_ptr(), known.kb.data_ptr())
            hit = den.graph_cache.get(key)
            if hit is None:
                reset()
                if host_noise:
                    noise_buf.zero_()
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    step_body()  # warm-up outside capture (function attributes, lazy module loading)
                torch.cuda.current_stream().wait_stream(side)
                reset()
                n_before = lib.launch_count
                g1 = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g1):
                    step_body()
                per_step = lib.launch_count - n_before
                gk = g1
                if unroll > 1:
                    reset()
                    gk = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(gk):
                        for _ in range(unroll):
                            step_body()
                if len(den.graph_cache) >= 4:
                    den.graph_cache.pop(next(iter(den.graph_cache)))
                hit = den.graph_cache[key] = (g1, gk, per_step, ddim)  # (ddim tables are kept alive with their graph)
            g1, gk, per_step, _ = hit
            reset()
            evs = None
            if time_steps:
                evs = [torch.cuda.Event(enable_timing=True) for _ in range(n_rep + 1)]
                evs[0].record()
            for i in range(n_rep):
                if host_noise:
                    feed_noise(steps[i])
                gk.replay()
                lib._launched(per_step * unroll)
                if evs is not None:
                    evs[i + 1].record()
            for i in range(rem):
                g1.replay()
                lib._launched(per_step)
            if evs is not None and n_rep > 0:
                self._step_events = (evs, unroll)  # read lazily (step_ms): no synchronisation inside the sampling job
        else:
            reset()
            for t in steps:
                feed_noise(t)
                if tap is not None:
                    x0 = den.denoise(xin, t_dev)
                    tap(t, x0.clone())
                step_body()  # (recomputes the denoiser when tapping: taps are a debugging aid)
        for t in tail_steps:  # high-precision tail: eager launches on the same loop state, schedule cursor and seed
            if lib.NVTX:
                torch.cuda.nvtx.range_push("fdm/tail_step")
            feed_noise(t)
            if tap is not None:
                tap(t, tail_den.denoise(x.view(B * T, d), t_dev).clone())
            step_body(hi=True)
            if lib.NVTX:
                torch.cuda.nvtx.range_pop()
        return x.view(x_T.shape).clone()  # the loop state buffer is reused by the next call
