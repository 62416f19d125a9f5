"""EVQ-VAE quantise + decode engine on libfdm_b200 kernels.

Replaces VectorQuantizer.forward (reference models/lib/quantizer.py:35-64, models/vq_vae_emotion.py:221-252,
models/vq_vae.py:219-248) and TransformerDecoder.forward (models/vq_vae_vocaset.py:245-258,
models/vq_vae_emotion.py:335-352) with the blocks of models/lib/base_models.py:37-174.
Per-clip (B = 1) semantics of the reference are kept for every clip of the batch: the positional encoding adds
row 0 of the sinusoid table to every frame (base_models.py:300 adds pe[:B]) and the emotion codebook slice is
chosen per clip.
"""
from __future__ import annotations

import math
from typing import Optional

import torch

from . import lib


class VQDecoderEngine:
    def __init__(self, module: torch.nn.Module, precision: str = "bf16"):
        assert precision in ("bf16", "fp32")
        self.m = module
        self.args = module.args
        self.precision = precision
        self.dtype = torch.bfloat16 if precision == "bf16" else torch.float32
        self._packed_key = None

    def pack(self, force: bool = False) -> None:
        sd = {k: v for k, v in self.m.state_dict().items() if k.startswith("decoder.")}
        key = (self.precision,) + tuple((k, v.data_ptr(), v._version) for k, v in sd.items())
        if not force and key == self._packed_key:
            return
        a = self.args
        if a.quant_factor != 0:
            raise NotImplementedError("only quant_factor == 0 (the reference's shipped configuration) is implemented")
        dev = next(iter(sd.values())).device
        assert dev.type == "cuda", "VQAutoEncoder must live on a CUDA device (no CPU fallback)"
        W = lambda k: sd["decoder." + k].detach().to(self.dtype).contiguous()
        Fv = lambda k: sd["decoder." + k].detach().float().contiguous()
        w = {}
        self.pre_linear = "decoder.decoder_linear_embedding_pre.net.weight" in sd
        if self.pre_linear:
            w["pre_w"], w["pre_b"] = W("decoder_linear_embedding_pre.net.weight"), Fv("decoder_linear_embedding_pre.net.bias")
        cw = sd["decoder.expander.0.0.weight"].detach()  # [C, C, 5] -> [Cout, tap, Cin]
        w["conv_w"] = cw.permute(0, 2, 1).reshape(cw.shape[0], -1).to(self.dtype).contiguous()
        w["conv_b"] = Fv("expander.0.0.bias")
        self.conv_k = cw.shape[2]
        d = a.hidden_size
        pe0 = torch.zeros(d, device=dev)
        pe0[1::2] = 1.0  # sin(0) = 0 on even channels, cos(0) = 1 on odd channels
        w["emb_w"] = W("decoder_linear_embedding.net.weight")
        w["emb_b"] = (Fv("decoder_linear_embedding.net.bias") + pe0).contiguous()
        w["blocks"] = []
        for l in range(a.num_hidden_layers):
            p, q = f"decoder_transformer.net.{2 * l}.fn.", f"decoder_transformer.net.{2 * l + 1}.fn."
            w["blocks"].append(dict(
                ln1_g=Fv(p + "norm.weight"), ln1_b=Fv(p + "norm.bias"), qkv_w=W(p + "fn.to_qkv.weight"),
                o_w=W(p + "fn.to_out.weight"), o_b=Fv(p + "fn.to_out.bias"),
                ln2_g=Fv(q + "norm.weight"), ln2_b=Fv(q + "norm.bias"),
                f1_w=W(q + "fn.l1.weight"), f1_b=Fv(q + "fn.l1.bias"), f2_w=W(q + "fn.l2.weight"), f2_b=Fv(q + "fn.l2.bias")))
        w["out_w"] = W("vertice_map_reverse.weight")
        w["out_b"] = Fv("vertice_map_reverse.bias") if "decoder.vertice_map_reverse.bias" in sd else None
        self.w, self.dev, self._packed_key = w, dev, key

    @torch.no_grad()
    def decode_rows(self, z_rows: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """z_rows: (B, T, fq*zdim) quantised latent per frame (fp32 or compute dtype) -> (B, T, in_dim) fp32."""
        self.pack()
        a, w, dev, dt = self.args, self.w, self.dev, self.dtype
        B, T, Cin = z_rows.shape
        assert Cin == a.face_quan_num * a.zquant_dim
        d = a.hidden_size
        x = z_rows.reshape(B * T, Cin)
        if x.dtype != dt:
            x = lib.cast(x.contiguous(), torch.empty(B * T, Cin, device=dev, dtype=dt))
        if self.pre_linear:
            y = torch.empty(B * T, d, device=dev, dtype=dt)
            lib.gemm(x, w["pre_w"], y, bias=w["pre_b"])
            x = y
        else:
            assert Cin == d
        k = self.conv_k
        pad = k // 2
        Tp = T + 2 * pad
        xp = torch.empty(B * Tp, d, device=dev, dtype=dt)
        lib.pad_time(x, xp, B, T, d, pad, pad, 1)  # Conv1d padding_mode='replicate'
        h = torch.zeros(B * Tp, d, device=dev, dtype=dt)
        lib.gemm(xp, w["conv_w"], h, bias=w["conv_b"], M=B * Tp - (k - 1), lda=d, a_rows=B * Tp, taps=k, tap_k=d, tap_row_shift=1)
        hc = torch.empty(B * T, d, device=dev, dtype=dt)
        lib.leaky_instnorm(h, hc, B, T, Tp, d, slope=0.2, eps=1e-5, out_t_stride=T)
        x = torch.empty(B * T, d, device=dev, dtype=dt)
        lib.gemm(hc, w["emb_w"], x, bias=w["emb_b"])
        H = a.num_attention_heads
        dh = d // H
        qkv = torch.empty(B * T, 3 * d, device=dev, dtype=dt)
        y = torch.empty(B * T, d, device=dev, dtype=dt)
        att = torch.empty(B * T, d, device=dev, dtype=dt)
        ffn = torch.empty(B * T, a.intermediate_size, device=dev, dtype=dt)
        for Lw in w["blocks"]:
            lib.layernorm(x, y, g1=Lw["ln1_g"], b1=Lw["ln1_b"])
            lib.gemm(y, Lw["qkv_w"], qkv)
            lib.self_attention(qkv[:, 0:], qkv[:, d:], qkv[:, 2 * d:], att, B, T, T, H, dh, d ** -0.5)
            lib.gemm(att, Lw["o_w"], x, bias=Lw["o_b"], residual=x)
            lib.layernorm(x, y, g1=Lw["ln2_g"], b1=Lw["ln2_b"])
            lib.gemm(y, Lw["f1_w"], ffn, bias=Lw["f1_b"], act=lib.ACT_GELU_TANH)
            lib.gemm(ffn, Lw["f2_w"], x, bias=Lw["f2_b"], residual=x)
        V3 = w["out_w"].shape[0]
        if out is None:
            out = torch.empty(B, T, V3, device=dev, dtype=torch.float32)
        lib.gemm(x, w["out_w"], out.view(B * T, V3), bias=w["out_b"])
        return out


    # ---- encoder (SURVEY section 8(f) item 3: VQAutoEncoder.encode, the stage-1 reconstruction path) -------------------
    def pack_encoder(self, force: bool = False) -> None:
        sd = {k: v for k, v in self.m.state_dict().items() if k.startswith("encoder.")}
        key = (self.precision,) + tuple((k, v.data_ptr(), v._version) for k, v in sd.items())
        if not force and key == getattr(self, "_enc_key", None):
            return
        a = self.args
        if a.quant_factor != 0:
            raise NotImplementedError("only quant_factor == 0 (the reference's shipped configuration) is implemented")
        dev = next(iter(sd.values())).device
        assert dev.type == "cuda", "VQAutoEncoder must live on a CUDA device (no CPU fallback)"
        dt = self.dtype
        W = lambda k: sd["encoder." + k].detach().to(dt).contiguous()
        Fv = lambda k: sd["encoder." + k].detach().float().contiguous()
        w = {}
        vm = sd["encoder.vertice_mapping.0.weight"].detach()
        K = vm.shape[1]
        Kp = (K + 7) // 8 * 8  # TMA needs 16-byte row pitches: in_dim = 15069 / 70110 are padded with zero columns
        vmp = torch.zeros(vm.shape[0], Kp, device=dev, dtype=dt)
        vmp[:, :K] = vm.to(dt)
        w["vm_w"], w["vm_b"], w["K"], w["Kp"] = vmp, Fv("vertice_mapping.0.bias"), K, Kp
        if "encoder.emotion_mapping.0.weight" in sd:
            w["emo_w"], w["emo_b"] = Fv("emotion_mapping.0.weight"), Fv("emotion_mapping.0.bias")
        cw = sd["encoder.squasher.0.0.weight"].detach()  # [C, C, 5] -> [Cout, tap, Cin]
        w["conv_w"] = cw.permute(0, 2, 1).reshape(cw.shape[0], -1).to(dt).contiguous()
        w["conv_b"] = Fv("squasher.0.0.bias")
        w["conv_k"] = cw.shape[2]
        d = a.hidden_size
        pe0 = torch.zeros(d, device=dev)
        pe0[1::2] = 1.0  # pe[:B] at B = 1: sin(0) on even, cos(0) on odd channels, for every frame
        w["emb_w"] = W("encoder_linear_embedding.net.weight")
        w["emb_b"] = (Fv("encoder_linear_embedding.net.bias") + pe0).contiguous()
        w["blocks"] = []
        for l in range(a.num_hidden_layers):
            p, q = f"encoder_transformer.net.{2 * l}.fn.", f"encoder_transformer.net.{2 * l + 1}.fn."
            w["blocks"].append(dict(
                ln1_g=Fv(p + "norm.weight"), ln1_b=Fv(p + "norm.bias"), qkv_w=W(p + "fn.to_qkv.weight"),
                o_w=W(p + "fn.to_out.weight"), o_b=Fv(p + "fn.to_out.bias"),
                ln2_g=Fv(q + "norm.weight"), ln2_b=Fv(q + "norm.bias"),
                f1_w=W(q + "fn.l1.weight"), f1_b=Fv(q + "fn.l1.bias"), f2_w=W(q + "fn.l2.weight"), f2_b=Fv(q + "fn.l2.bias")))
        # models/vq_vae_vocaset.py:181-191 never applies encoder_linear_embedding_post; vq_vae.py / vq_vae_emotion.py do
        self.enc_post = self.pre_linear_enc = "encoder.encoder_linear_embedding_post.net.weight" in sd and type(self.m).pre_linear
        if self.enc_post:
            w["post_w"], w["post_b"] = W("encoder_linear_embedding_post.net.weight"), Fv("encoder_linear_embedding_post.net.bias")
        self.we, self.dev, self._enc_key = w, dev, key

    @torch.no_grad()
    def encode_rows(self, verts: torch.Tensor, emo_one_hot: Optional[torch.Tensor] = None) -> torch.Tensor:
        """verts (B, T, in_dim) motion -> latent (B, fq*T, zquant_dim) fp32 (per-clip B = 1 semantics for every clip)."""
        self.pack_encoder()
        a, w, dev, dt = self.args, self.we, self.dev, self.dtype
        B, T, K = verts.shape
        assert K == w["K"]
        d = a.hidden_size
        xin = torch.empty(B * T, w["Kp"], device=dev, dtype=dt)
        lib.cast_rows(verts.detach().float().contiguous().view(B * T, K), xin)
        res = None
        if "emo_w" in w:
            if emo_one_hot is None:
                raise TypeError("encode() of the emotion EVQ-VAE needs the emotion one-hot")
            oh = emo_one_hot.to(dev).float()
            if oh.dim() == 3:  # per frame: (B | 1, T, 7), the emotion_mapping output of frame f is added to frame f
                oh = oh.expand(B, T, -1).reshape(B * T, -1).contiguous()
                e = torch.empty(B * T, d, device=dev, dtype=torch.float32)
                lib.gemm(oh, w["emo_w"], e, bias=w["emo_b"], act=lib.ACT_LEAKY02)
                res = e.to(dt)
            else:
                oh = (oh[None] if oh.dim() == 1 else oh).expand(B, -1).contiguous()
                e = torch.empty(B, d, device=dev, dtype=torch.float32)
                lib.gemm(oh, w["emo_w"], e, bias=w["emo_b"], act=lib.ACT_LEAKY02)
                res = e.to(dt).repeat_interleave(T, dim=0)  # emotion_mapping output is added to every frame of its clip
        x = torch.empty(B * T, d, device=dev, dtype=dt)
        lib.gemm(xin, w["vm_w"], x, bias=w["vm_b"], act=lib.ACT_LEAKY02, residual=res)
        k = w["conv_k"]
        pad = k // 2
        Tp = T + 2 * pad
        xp = torch.empty(B * Tp, d, device=dev, dtype=dt)
        lib.pad_time(x, xp, B, T, d, pad, pad, 1)  # Conv1d padding_mode='replicate'
        h = torch.zeros(B * Tp, d, device=dev, dtype=dt)
        lib.gemm(xp, w["conv_w"], h, bias=w["conv_b"], M=B * Tp - (k - 1), lda=d, a_rows=B * Tp, taps=k, tap_k=d, tap_row_shift=1)
        hc = torch.empty(B * T, d, device=dev, dtype=dt)
        lib.leaky_instnorm(h, hc, B, T, Tp, d, slope=0.2, eps=1e-5, out_t_stride=T)
        lib.gemm(hc, w["emb_w"], x, bias=w["emb_b"])
        x = self._blocks(x, w["blocks"], B, T)
        if self.enc_post:
            out = torch.empty(B * T, a.face_quan_num * a.zquant_dim, device=dev, dtype=torch.float32)
            lib.gemm(x, w["post_w"], out, bias=w["post_b"])
        else:
            out = x.float() if x.dtype != torch.float32 else x
        return out.view(B, T * a.face_quan_num, a.zquant_dim)

    def _blocks(self, x: torch.Tensor, blocks, B: int, T: int) -> torch.Tensor:
        a, dev, dt = self.args, self.dev, self.dtype
        d = a.hidden_size
        H = a.num_attention_heads
        dh = d // H
        qkv = torch.empty(B * T, 3 * d, device=dev, dtype=dt)
        y = torch.empty(B * T, d, device=dev, dtype=dt)
        att = torch.empty(B * T, d, device=dev, dtype=dt)
        ffn = torch.empty(B * T, a.intermediate_size, device=dev, dtype=dt)
        for Lw in blocks:
            lib.layernorm(x, y, g1=Lw["ln1_g"], b1=Lw["ln1_b"])
            lib.gemm(y, Lw["qkv_w"], qkv)
            lib.self_attention(qkv[:, 0:], qkv[:, d:], qkv[:, 2 * d:], att, B, T, T, H, dh, d ** -0.5)
            lib.gemm(att, Lw["o_w"], x, bias=Lw["o_b"], residual=x)
            lib.layernorm(x, y, g1=Lw["ln2_g"], b1=Lw["ln2_b"])
            lib.gemm(y, Lw["f1_w"], ffn, bias=Lw["f1_b"], act=lib.ACT_GELU_TANH)
            lib.gemm(ffn, Lw["f2_w"], x, bias=Lw["f2_b"], residual=x)
        return x


def slice_runs(offsets: torch.Tensor, fq: int):
    """(B, T) int64 codebook offset per frame -> the CSR run table of fdm_vq_runs over the (B, fq*T) latent rows, as host
    tensors (clip_run (B+1), run_l0, run_offset): a run starts at a clip's first frame and wherever the offset changes."""
    offsets = offsets.to("cpu", torch.int64)
    B, T = offsets.shape
    start = torch.ones(B, T, dtype=torch.bool)
    start[:, 1:] = offsets[:, 1:] != offsets[:, :-1]
    b, f = start.nonzero(as_tuple=True)
    clip_run = torch.zeros(B + 1, dtype=torch.int64)
    clip_run[1:] = start.sum(1).cumsum(0)
    return clip_run, f * fq, offsets[b, f].contiguous()


def check_frame_cond(oh, B: int, T: int, n: int, what: str = "a condition") -> None:
    """ValueError unless the per-frame condition `oh` is (B or 1, T, n)."""
    if oh.shape[0] not in (1, B):
        raise ValueError(f"{what} has {oh.shape[0]} rows; the call has {B} sequences (give {B} rows or 1)")
    if oh.shape[1] != T:
        raise ValueError(f"{what} has {oh.shape[1]} frames; the call has {T} (a per-frame condition is (B | 1, T, n))")
    if oh.shape[2] != n:
        raise ValueError(f"{what} has rows of {oh.shape[2]} entries; it needs {n}")


def quantize(z: torch.Tensor, codebook: torch.Tensor, n_local: int, emo_one_hot: Optional[torch.Tensor] = None,
             want_bdl: bool = True, want_rows: bool = False, want_stats: bool = False, fq: int = 1):
    """z (B, L, D) fp32. Per-clip emotion slice: offset = n_local * argmax(one_hot[b]) (the reference takes a
    global argmax because it only ever sees B = 1, models/vq_vae_emotion.py:223). A per-frame one-hot (B | 1, L / fq, n)
    gives frame f's fq latent rows the slice n_local * argmax(one_hot[b, f]) (fdm_vq_quantize_runs). want_stats: also the
    by-products of the reference forward (sum of squared quantisation errors as a 0-d fp64 tensor, code histogram) from one
    more pass over z."""
    z = z.contiguous().float()
    B = z.shape[0]
    if emo_one_hot is not None and emo_one_hot.dim() == 3:
        T = z.shape[1] // fq
        pos = torch.argmax(emo_one_hot, dim=-1).to(torch.int64).expand(B, T)
        runs = slice_runs(pos * n_local, fq)
        cb = codebook.detach().float().contiguous()
        idx, zq, zr = lib.vq_quantize_runs(z, cb, n_local, runs, want_bdl=want_bdl, want_rows=want_rows)
        if want_stats:
            sq, hist = lib.vq_stats_runs(z, cb, idx.view(-1), n_local, runs)
            return idx, zq, zr, sq, hist
        return idx, zq, zr
    off = None
    if emo_one_hot is not None:
        oh = emo_one_hot.to(z.device)
        if oh.dim() == 1:
            oh = oh[None]
        pos = torch.argmax(oh, dim=-1).to(torch.int64)
        if pos.numel() == 1 and B > 1:
            pos = pos.expand(B)
        off = (pos * n_local).contiguous()
    cb = codebook.detach().float().contiguous()
    idx, zq, zr = lib.vq_quantize(z, cb, n_local, code_offset=off, want_bdl=want_bdl, want_rows=want_rows)
    if want_stats:
        sq, hist = lib.vq_stats(z, cb, idx.view(-1), n_local, code_offset=off)
        return idx, zq, zr, sq, hist
    return idx, zq, zr
