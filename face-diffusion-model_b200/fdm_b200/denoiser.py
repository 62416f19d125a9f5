"""FDM denoiser engine: the per-step transformer of the LG-LDM sampler on libfdm_b200 kernels.

Replaces the body of FDM.forward (reference models/fdm_vocaset.py:54-91, models/fdm_vqvae_mead.py:65-104,
models/fdm.py:65-98). What changes against the reference, per SURVEY.md §0:
  * everything that does not depend on the step t is computed ONCE per clip batch (`prepare`): the audio
    encoder, audio_extract, style/emotion embeddings, positional encoding, and — because enc_dec_mask only
    keeps the diagonal (models/fdm_vocaset.py:118-127), so softmax has one live entry — the whole
    cross-attention block, which collapses to out_proj(v_proj(memory_i)) with memory = audio_feature + time(t):
    the audio part is cached per clip and layer, the time part is a 1000-row table per layer;
  * a step is 4 GEMMs + 1 attention + 2 fused residual/LayerNorm kernels per layer, launched on the current
    stream with no host synchronisation (t is read from device memory), so a step can be graph-captured;
  * clips are batched (the reference is B = 1 only); every clip follows the reference's B = 1 semantics.
"""
from __future__ import annotations

import math
import os
from typing import Optional

import torch

from . import lib
from .presets import Preset, alibi_slopes
from .vqvae import check_frame_cond


def _sin_table(n: int, d: int) -> torch.Tensor:
    pe = torch.zeros(n, d)
    pos = torch.arange(0, n, dtype=torch.float).unsqueeze(1)
    div = torch.exp(torch.arange(0, d, 2).float() * (-math.log(10000.0) / d))
    pe[:, 0::2] = torch.sin(pos * div)
    pe[:, 1::2] = torch.cos(pos * div)
    return pe


class DenoiserEngine:
    def __init__(self, module: torch.nn.Module, preset: Preset, precision: str = "bf16"):
        # "bf16": bf16 operands and activations (throughput mode); "fp32": FFMA GEMMs, exact fp32 attention (parity mode);
        # "x3": fp32 activations, GEMMs on the tensor cores with split-bf16 operands (A_lo W + A W_lo + A W, 2^-17 relative):
        # the high-precision tail steps of the bf16 sampler
        assert precision in ("bf16", "fp32", "x3")
        self.module = module
        self.P = preset
        self.precision = precision
        self.dtype = torch.bfloat16 if precision == "bf16" else torch.float32
        self._packed_key = None
        self.pack_serial = 0
        self.w = {}
        self.B = 0
        self.T = 0
        self.passes = 1
        self.lanes = int(os.environ.get("FDM_B200_LANES", "1"))
        if self.lanes == 2:
            lib.splitk_enabled = False  # two streams run GEMMs concurrently: they must not share the (opt-in) tail split-K workspace
        self._side = None
        self.fold = False
        # bf16 mode: residual adds inside the LayerNorm kernels (FDM_B200_RES_IN_LN=0: in the GEMM epilogues, as in fp32 / x3 mode)
        self.res_in_ln = self.dtype == torch.bfloat16 and os.environ.get("FDM_B200_RES_IN_LN", "1") != "0"
        self._pool = {}          # name -> persistent device buffer (stable addresses keep captured step graphs valid)
        self.graph_cache = {}    # sampler step graphs, keyed by every address / scalar baked into them

    # ---- weights ---------------------------------------------------------------------------------
    def _params(self):
        return {k: v for k, v in self.module.state_dict().items() if not k.startswith("audio_encoder.")}

    def pack(self, force: bool = False) -> None:
        sd = self._params()
        key = (self.precision,) + tuple((k, v.data_ptr(), v._version) for k, v in sd.items())
        if not force and key == self._packed_key:
            return
        P, d = self.P, self.P.d
        dev = next(iter(sd.values())).device
        assert dev.type == "cuda", "FDM must live on a CUDA device (no CPU fallback)"
        if self.precision == "x3":
            Wt = lambda t: lib.split(t.detach().float().contiguous())
        else:
            Wt = lambda t: t.detach().to(self.dtype).contiguous()
        W = lambda k: Wt(sd[k])
        Bv = lambda k: sd[k].detach().float().contiguous()
        w = {}
        w["ae0_w"], w["ae0_b"] = W("audio_extract.0.weight"), Bv("audio_extract.0.bias")
        w["ae2_w"], w["ae2_b"] = W("audio_extract.2.weight"), Bv("audio_extract.2.bias")
        le = "latent_encoder.0." if P.latent_mish else "latent_encoder."
        w["le_w"], w["le_b"] = W(le + "weight"), Bv(le + "bias")
        st = "style_embedd.0." if P.style_mish else "style_embedd."
        w["st_w"], w["st_b"] = Bv(st + "weight"), Bv(st + "bias")
        if P.emotion:
            w["em_w"], w["em_b"] = Bv("emotion_embedd.weight"), Bv("emotion_embedd.bias")
        w["ld_w"], w["ld_b"] = W("latent_decoder.weight"), Bv("latent_decoder.bias")
        # time table: Mish(Linear(one_hot(t))) for every t, via an fp32 GEMM against the identity
        n_t = sd["time_embedd.0.weight"].shape[1]
        eye = torch.eye(n_t, device=dev)
        tt = torch.empty(n_t, d, device=dev)
        lib.gemm(eye, Bv("time_embedd.0.weight"), tt, bias=Bv("time_embedd.0.bias"), act=lib.ACT_MISH)
        w["time_table"] = tt
        tmp = torch.empty(n_t, d, device=dev)
        for l in range(P.layers):
            p = f"transformer_decoder.layers.{l}."
            L = {}
            L["qkv_w"], L["qkv_b"] = W(p + "self_attn.in_proj_weight"), Bv(p + "self_attn.in_proj_bias")
            L["o_w"], L["o_b"] = W(p + "self_attn.out_proj.weight"), Bv(p + "self_attn.out_proj.bias")
            ipw, ipb = sd[p + "multihead_attn.in_proj_weight"].detach(), sd[p + "multihead_attn.in_proj_bias"].detach()
            L["cv_w"], L["cv_b"] = Wt(ipw[2 * d:]), ipb[2 * d:].float().contiguous()
            L["co_w"], L["co_b"] = W(p + "multihead_attn.out_proj.weight"), Bv(p + "multihead_attn.out_proj.bias")
            L["f1_w"], L["f1_b"] = W(p + "linear1.weight"), Bv(p + "linear1.bias")
            L["f2_w"], L["f2_b"] = W(p + "linear2.weight"), Bv(p + "linear2.bias")
            for n in (1, 2, 3):
                L[f"n{n}_w"], L[f"n{n}_b"] = Bv(p + f"norm{n}.weight"), Bv(p + f"norm{n}.bias")
            # time part of the collapsed cross-attention: out_proj(v_proj(time_table)) without biases, fp32
            lib.gemm(tt, ipw[2 * d:].float().contiguous(), tmp)
            L["time_cross"] = torch.empty(n_t, d, device=dev)
            lib.gemm(tmp, Bv(p + "multihead_attn.out_proj.weight"), L["time_cross"])
            w[l] = L
        # LayerNorm folding (bf16 mode): norm3 of layer l-1 is never materialised. The FFN2 GEMM writes u = x + FFN(x) and its
        # row statistics; the next QKV projection (or the latent decoder after the last layer) runs on u with
        # W' = W diag(gamma3), colsum(W') and bias' = bias + W beta3, and the out-projection rebuilds LN3(u) for its residual.
        # Opt-in (FDM_B200_FOLD_LN=1): it removes 0.23 ms of LayerNorm kernels per step but the extra epilogue work (per-column
        # gamma / beta on a row-per-thread layout, row statistics) costs the GEMMs the same 0.23 ms - 4.64 vs 4.47 ms per step.
        self.fold = self.dtype == torch.bfloat16 and os.environ.get("FDM_B200_FOLD_LN", "0") == "1"
        if self.fold:
            def folded(weight_f32, bias_f32, gamma, beta):
                wp = (weight_f32 * gamma[None]).to(self.dtype).contiguous()
                return wp, wp.float().sum(-1).contiguous(), (bias_f32 + weight_f32 @ beta).contiguous()
            for l in range(1, P.layers):
                p = f"transformer_decoder.layers.{l}."
                g3, b3 = w[l - 1]["n3_w"], w[l - 1]["n3_b"]
                w[l]["qkv_wf"], w[l]["qkv_cs"], w[l]["qkv_bf"] = folded(sd[p + "self_attn.in_proj_weight"].detach().float(),
                                                                      w[l]["qkv_b"], g3, b3)
            g3, b3 = w[P.layers - 1]["n3_w"], w[P.layers - 1]["n3_b"]
            w["ld_wf"], w["ld_cs"], w["ld_bf"] = folded(sd["latent_decoder.weight"].detach().float(), w["ld_b"], g3, b3)
        w["slopes"] = torch.tensor(alibi_slopes(P.heads), dtype=torch.float32, device=dev)
        if P.periodic_pe:
            w["pe"] = _sin_table(P.period, d).to(dev)
        else:
            w["pe"] = None  # built per T in prepare
        self.w = w
        self.dev = dev
        self._packed_key = key
        self.pack_serial += 1

    def buf(self, name: str, shape, dtype, device=None) -> torch.Tensor:
        """Persistent buffer: the same tensor is returned while name / shape / dtype / device do not change, so that a
        new clip batch of the same shape reuses the addresses the cached CUDA graphs were captured with."""
        device = device if device is not None else self.dev
        t = self._pool.get(name)
        if t is None or tuple(t.shape) != tuple(shape) or t.dtype != dtype or t.device != device:
            with torch.inference_mode(False):  # a normal tensor: it is updated in place inside and outside inference mode
                t = torch.empty(tuple(shape), device=device, dtype=dtype)
            self._pool[name] = t
        return t

    # ---- per-clip-batch state ---------------------------------------------------------------------
    def prepare(self, audio_hidden: torch.Tensor, n_frames: int, id_one_hot: torch.Tensor,
                emo_one_hot: Optional[torch.Tensor] = None, guidance: Optional[str] = None, fanout: int = 1) -> None:
        """audio_hidden: (A, N, audio_dim) audio-encoder output in the compute dtype; n_frames: latent frames T.
        fanout: K sequences per audio clip, B = A*K sequences, sequence a*K + k on clip a; the one-hots have B rows or 1,
        or are per frame, (B | 1, T, n): frame f of sequence b is conditioned on row [b, f] (any values, e.g. a cross-fade).
        guidance: None, or the name of the condition the unconditional pass zeroes ("id" | "emotion")."""
        self.pack()
        P, w, d = self.P, self.w, self.P.d
        A, N, Ca = audio_hidden.shape
        assert Ca == P.audio_dim and audio_hidden.dtype == self.dtype and audio_hidden.is_contiguous() and fanout >= 1
        B = A * fanout
        Ta = N // 2 if P.pair_audio else N
        if n_frames > Ta:
            raise ValueError(f"latent has {n_frames} frames but the audio only yields {Ta} (the reference fails here too)")
        for oh, n in ((id_one_hot, P.n_id), (emo_one_hot, 7)):  # checked before any buffer changes, so a refused call keeps
            if oh is not None and oh.dim() == 3:                 # the prepared state
                check_frame_cond(oh, B, n_frames, n)
                continue
            rows = 1 if oh is None or oh.dim() == 1 else oh.shape[0]
            if rows not in (1, B):
                raise ValueError(f"a condition has {rows} rows; the call has {B} sequences (give {B} rows or 1)")
        T = n_frames
        if P.pair_audio:
            a = audio_hidden[:, : 2 * T].reshape(A, T, 2 * Ca)
        else:
            a = audio_hidden[:, :T]
        a = a.reshape(A * T, P.audio_in) if a.is_contiguous() else a.contiguous().view(A * T, P.audio_in)
        dev, dt = self.dev, self.dtype
        AT, BT = A * T, B * T
        h = self.buf("prep_h", (AT, d), dt)
        af = self.buf("prep_af", (AT, d), dt)
        lib.gemm(a, w["ae0_w"], h, bias=w["ae0_b"], act=lib.ACT_MISH)
        lib.gemm(h, w["ae2_w"], af, bias=w["ae2_b"])
        af_op = lib.split(af) if self.precision == "x3" else af  # (operand of eight GEMMs: split once)
        # audio part of the collapsed cross-attention, per layer and clip; with fan-out each clip's block is then copied
        # to its K sequences, so the step reads the same (B*T, d) caches as for the repeated audio batch
        cc = self.buf("prep_cross", (AT, d), dt) if fanout > 1 else None
        self.cross = []
        for l in range(P.layers):
            L = w[l]
            c = self.buf(f"cross{l}", (BT, d), dt)
            lib.gemm(af_op, L["cv_w"], h, bias=L["cv_b"])
            if cc is None:
                lib.gemm(h, L["co_w"], c, bias=L["co_b"])
            else:
                lib.gemm(h, L["co_w"], cc, bias=L["co_b"])
                c.view(A, fanout, T, d).copy_(cc.view(A, 1, T, d).expand(A, fanout, T, d))  # setup-time broadcast
            self.cross.append(c)
        # style (+ emotion) per sequence (or per frame) and pass, plus positional encoding -> one addend tensor per pass. With a
        # per-frame condition both GEMMs run over the B*T frame rows; the FFMA GEMM's rows do not depend on M, so a constant
        # schedule gives the per-sequence call's bits.
        per_frame = any(oh is not None and oh.dim() == 3 for oh in (id_one_hot, emo_one_hot))
        def expand(oh, n):
            oh = oh.to(dev, torch.float32)
            if oh.dim() == 3:
                return oh.expand(B, T, n).reshape(BT, n).contiguous()
            if oh.dim() == 1:
                oh = oh[None]
            assert oh.shape[-1] == n
            oh = oh.expand(B, n) if oh.shape[0] == 1 else oh
            return oh.repeat_interleave(T, dim=0) if per_frame else oh.contiguous()
        ids = expand(id_one_hot, P.n_id)
        emo = expand(emo_one_hot, 7) if P.emotion else None
        passes = [(ids, emo)]
        if guidance == "id":
            passes.append((torch.zeros_like(ids), emo))
        elif guidance == "emotion":
            assert P.emotion
            passes.append((ids, torch.zeros_like(emo)))
        elif guidance is not None:
            raise ValueError(guidance)
        pe = w["pe"][torch.arange(T, device=dev) % P.period] if P.periodic_pe else _sin_table(T, d).to(dev)
        addends = []
        for (i_oh, e_oh) in passes:
            sty = torch.empty(i_oh.shape[0], d, device=dev)
            lib.gemm(i_oh, w["st_w"], sty, bias=w["st_b"], act=lib.ACT_MISH if P.style_mish else lib.ACT_NONE)
            if P.emotion:
                lib.gemm(e_oh, w["em_w"], sty, bias=w["em_b"], residual=sty)
            ad = self.buf(f"addend{len(addends)}", (BT, d), dt)
            ad.copy_((sty.view(B, -1, d) + pe[None]).reshape(BT, d))  # setup-time broadcast (+ cast)
            addends.append(ad)
        self.addend = addends
        # guidance: both passes share Mish(latent_encoder(x_t)); the second pass is the first plus (addend_1 - addend_0)
        self.addend_delta = None
        if len(addends) == 2:
            self.addend_delta = self.buf("addend_delta", (BT, d), dt)
            self.addend_delta.copy_(addends[1].float() - addends[0].float())
        S = len(passes)
        self.B, self.T, self.passes = B, T, S
        self.x = self.buf("x", (S * BT, d), dt)
        self.qkv = self.buf("qkv", (S * BT, 3 * d), dt)
        self.att = self.buf("att", (S * BT, d), dt)
        self.proj = self.buf("proj", (S * BT, d), dt)
        self.ffn = self.buf("ffn", (S * BT, 2 * d), dt)
        self.x0 = self.buf("x0", (S, B, T * d), torch.float32)
        if self.fold:
            self.ln_parts = self.buf("ln_parts", (S * BT, d // 64, 2), torch.float32)
            self.ln_mr = self.buf("ln_mr", (S * BT, 2), torch.float32)

    # ---- one denoiser evaluation ------------------------------------------------------------------------
    def denoise(self, x_in: torch.Tensor, t_dev: torch.Tensor) -> torch.Tensor:
        """x_in: (B*T, d) noisy latent regrouped per frame, compute dtype; t_dev: int32[1] on device.
        Returns x0_hat (passes, B, T*d) fp32 (pass 0 = conditional, pass 1 = unconditional).

        With guidance the two passes are independent until the fused update, so they can run as two LANES on two
        streams (fork / join with events, capturable in a CUDA graph): the HBM-bound residual/LayerNorm kernels of one
        lane then overlap the power-bound tcgen05 GEMMs of the other instead of queueing behind them. `self.lanes`
        (env FDM_B200_LANES = 2) selects it; per-row results do not depend on the split. Off by default: measured
        4.44 vs 4.41 ms per step - the step sits at the 1 kW power cap, overlap only lowers the SM clock further."""
        B, T, S = self.B, self.T, self.passes
        assert x_in.shape == (B * T, self.P.d) and x_in.dtype == self.dtype
        if S == 2 and self.lanes == 2:
            cur = torch.cuda.current_stream()
            if self._side is None or self._side.device != x_in.device:
                self._side = torch.cuda.Stream(device=x_in.device)
            self._side.wait_stream(cur)
            with torch.cuda.stream(self._side):
                self._run_passes(x_in, t_dev, 1, 2)
            self._run_passes(x_in, t_dev, 0, 1)
            cur.wait_stream(self._side)
        else:
            self._run_passes(x_in, t_dev, 0, S)
        return self.x0

    def _run_passes(self, x_in: torch.Tensor, t_dev: torch.Tensor, s0: int, s1: int) -> None:
        """The transformer stack for passes [s0, s1) = rows [s0*B*T, s1*B*T) of every activation buffer."""
        P, w, d = self.P, self.w, self.P.d
        B, T = self.B, self.T
        BT = B * T
        r0, r1, n = s0 * BT, s1 * BT, s1 - s0
        x, qkv, att, proj, ffn = self.x[r0:r1], self.qkv[r0:r1], self.att[r0:r1], self.proj[r0:r1], self.ffn[r0:r1]
        if n == 2 and self.addend_delta is not None and self.dtype == torch.bfloat16:
            # one latent-encoder GEMM for both guidance passes (its Mish epilogue is MUFU-bound: 55 us per pass) + one add
            lib.gemm(x_in, w["le_w"], x[:BT], bias=w["le_b"], act=lib.ACT_MISH if P.latent_mish else lib.ACT_NONE,
                     residual=self.addend[0])
            lib.layernorm(x[:BT], x[BT:], r1=self.addend_delta)  # no gamma: a plain row-wise add
        else:
            x_op = lib.split(x_in) if self.precision == "x3" else x_in
            for s in range(n):
                lib.gemm(x_op, w["le_w"], x[s * BT:(s + 1) * BT], bias=w["le_b"],
                         act=lib.ACT_MISH if P.latent_mish else lib.ACT_NONE, residual=self.addend[s0 + s])
        scale = 1.0 / math.sqrt(P.dh)
        rows = r1 - r0
        if not self.fold:
            for l in range(P.layers):
                L = w[l]
                lib.gemm(x, L["qkv_w"], qkv, bias=L["qkv_b"])
                lib.self_attention(qkv[:, 0:], qkv[:, d:], qkv[:, 2 * d:], att, n * B, T, T, P.heads, P.dh, scale,
                                   slopes=w["slopes"], period=P.period)
                if self.res_in_ln:
                    # the residual adds x + f(x) happen inside the LayerNorm kernels, in fp32: the sums are never rounded to
                    # bf16 (two of the seven bf16 roundings per layer gone) and the GEMMs lose their residual epilogue
                    lib.gemm(att, L["o_w"], proj, bias=L["o_b"])
                    lib.layernorm(proj, x, r1=x, g1=L["n1_w"], b1=L["n1_b"], r2=self.cross[l], vec2=L["time_cross"],
                                  vec_index_dev=t_dev, g2=L["n2_w"], b2=L["n2_b"])
                    lib.gemm(x, L["f1_w"], ffn, bias=L["f1_b"], act=lib.ACT_RELU)
                    lib.gemm(ffn, L["f2_w"], proj, bias=L["f2_b"])
                    lib.layernorm(proj, x, r1=x, g1=L["n3_w"], b1=L["n3_b"])
                    continue
                lib.gemm(att, L["o_w"], proj, bias=L["o_b"], residual=x)
                lib.layernorm(proj, x, g1=L["n1_w"], b1=L["n1_b"], r2=self.cross[l], vec2=L["time_cross"],
                              vec_index_dev=t_dev, g2=L["n2_w"], b2=L["n2_b"])
                lib.gemm(x, L["f1_w"], ffn, bias=L["f1_b"], act=lib.ACT_RELU)
                lib.gemm(ffn, L["f2_w"], proj, bias=L["f2_b"], residual=x)
                lib.layernorm(proj, x, g1=L["n3_w"], b1=L["n3_b"])
            lib.gemm(x, w["ld_w"], self.x0.view(self.passes * BT, d)[r0:r1], bias=w["ld_b"])
            return
        # ---- norm3 folded into the neighbouring GEMMs: `proj` carries u = x + FFN(x) between layers, `mr` its (mean, rstd) ----
        parts, mr = self.ln_parts[r0:r1], self.ln_mr[r0:r1]
        for l in range(P.layers):
            L = w[l]
            if l == 0:
                lib.gemm(x, L["qkv_w"], qkv, bias=L["qkv_b"])
            else:
                lib.gemm(proj, L["qkv_wf"], qkv, bias=L["qkv_bf"], a_ln=mr, w_colsum=L["qkv_cs"])
            lib.self_attention(qkv[:, 0:], qkv[:, d:], qkv[:, 2 * d:], att, n * B, T, T, P.heads, P.dh, scale,
                               slopes=w["slopes"], period=P.period)
            if l == 0:
                lib.gemm(att, L["o_w"], proj, bias=L["o_b"], residual=x)
                u1 = proj
            else:  # residual = LN3(u) of the previous layer, rebuilt in the epilogue from `proj`
                lib.gemm(att, L["o_w"], x, bias=L["o_b"], residual=proj, res_ln=mr, res_gamma=w[l - 1]["n3_w"],
                         res_beta=w[l - 1]["n3_b"])
                u1 = x
            lib.layernorm(u1, x, g1=L["n1_w"], b1=L["n1_b"], r2=self.cross[l], vec2=L["time_cross"],
                          vec_index_dev=t_dev, g2=L["n2_w"], b2=L["n2_b"])
            lib.gemm(x, L["f1_w"], ffn, bias=L["f1_b"], act=lib.ACT_RELU)
            lib.gemm(ffn, L["f2_w"], proj, bias=L["f2_b"], residual=x, stats_out=parts)
            lib.ln_stats_finalize(parts, rows, d // 64, d, mr)
        lib.gemm(proj, w["ld_wf"], self.x0.view(self.passes * BT, d)[r0:r1], bias=w["ld_bf"], a_ln=mr, w_colsum=w["ld_cs"])

    def kernels_per_step(self) -> int:
        return (self.passes + 2 * (7 * self.P.layers + 1)) if (self.passes == 2 and self.lanes == 2) else (self.passes + 7 * self.P.layers + 1)

    def flops_per_step(self) -> float:
        """FLOPs actually executed by one denoise() call (GEMMs + dense attention)."""
        d, T, S, B = self.P.d, self.T, self.passes, self.B
        per_seq = self.P.layers * (16 * T * d * d + 4 * T * T * d) + 4 * T * d * d
        return float(S * B * per_seq)
