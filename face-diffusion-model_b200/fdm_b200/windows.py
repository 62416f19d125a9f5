"""Window plan of long-audio sampling (GaussianDiffusion.sample_long), host side and device-free.

A long sequence of T frames is cut into n_w windows of W frames, window w covering absolute frames [w*S, w*S + W) with
stride S = W - O: neighbouring windows share O frames. All windows of all clips are sampled as one batch, and after every
step fdm_window_blend mixes each shared frame's two rows. Window sequence (a*n_w + w)*K + k holds window w of clip a's
fan-out sequence k. The last window may run past T: its extra frames are sampled on zero audio and dropped (self-attention
is causal and everything else is per frame, so they cannot change a real frame).
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional, Tuple

import torch

from .presets import Preset, conv_out_len

HOP = 320          # audio samples per audio-encoder frame (16 kHz: conv strides 5 * 2^6)
RECEPTIVE = 400    # audio samples the first encoder frame needs
MAX_WINDOW = 600   # longest clip the model was trained on, in frames


def default_window(P: Preset) -> Tuple[int, int]:
    """(window, overlap) in frames: 14 and 2 periods (420 / 60 for VOCASET and MEAD, 350 / 50 for BIWI)."""
    return 14 * P.period, 2 * P.period


@dataclass(frozen=True)
class WindowPlan:
    A: int   # audio clips
    K: int   # sequences per clip (fan-out)
    T: int   # frames of the long sequences
    W: int   # frames per window
    O: int   # frames shared by neighbouring windows
    r: int   # audio-encoder frames per latent frame (2 for pair_audio presets)

    @property
    def S(self) -> int:
        return self.W - self.O

    @property
    def n_w(self) -> int:
        return max(1, math.ceil((self.T - self.O) / self.S))

    @property
    def T_pad(self) -> int:
        """Frames the windows cover: T rounded up to the end of the last window."""
        return (self.n_w - 1) * self.S + self.W

    @property
    def n_seq(self) -> int:
        return self.A * self.n_w * self.K

    def starts(self):
        return [w * self.S for w in range(self.n_w)]

    def seq(self, a: int, w: int, k: int) -> int:
        return (a * self.n_w + w) * self.K + k

    # -- audio ------------------------------------------------------------------------------------------
    @property
    def audio_len(self) -> int:
        """Samples per window: exactly W*r encoder frames."""
        return HOP * (self.W * self.r - 1) + RECEPTIVE

    def audio_bounds(self, w: int) -> Tuple[int, int]:
        lo = w * self.S * self.r * HOP
        return lo, lo + self.audio_len

    def window_audio(self, audio: torch.Tensor) -> torch.Tensor:
        """(A, L) -> (A*n_w, audio_len): row a*n_w + w is window w's slice of clip a, zero past the end of the clip."""
        step = self.S * self.r * HOP
        need = (self.n_w - 1) * step + self.audio_len
        a = audio[:, :need]
        if a.shape[1] < need:
            a = torch.nn.functional.pad(a, (0, need - a.shape[1]))
        return a.unfold(1, self.audio_len, step).reshape(self.A * self.n_w, self.audio_len).contiguous()

    # -- sequences ----------------------------------------------------------------------------------------
    def repeat_rows(self, cond: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
        """A condition of A*K rows (sequence a*K + k) -> one row per window sequence; one row (or 1-D) is kept."""
        if cond is None or cond.dim() == 1 or cond.shape[0] == 1:
            return cond
        n = cond.shape[-1]
        return cond.reshape(self.A, 1, self.K, n).expand(self.A, self.n_w, self.K, n).reshape(self.n_seq, n)

    def gather_frames(self, cond: torch.Tensor) -> torch.Tensor:
        """A per-frame condition (A*K or 1, T, n) -> (A*n_w*K, W, n): window w's rows are frames [w*S, w*S + W), frames at
        or past T (sampled on zero audio and dropped) take frame T - 1's row."""
        n = cond.shape[-1]
        f = self.frame_index().clamp(max=self.T - 1).to(cond.device)
        x = cond.expand(self.A * self.K, self.T, n).reshape(self.A, self.K, self.T, n)[:, :, f]  # (A, K, n_w, W, n)
        return x.permute(0, 2, 1, 3, 4).reshape(self.n_seq, self.W, n).contiguous()

    def window_rows(self, cond: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
        """The condition of the window sequences: gather_frames for a per-frame (3-D) condition, else repeat_rows."""
        if cond is not None and cond.dim() == 3:
            return self.gather_frames(cond)
        return self.repeat_rows(cond)

    def frame_index(self) -> torch.Tensor:
        """(n_w, W) absolute frame of every window row."""
        return torch.arange(self.n_w)[:, None] * self.S + torch.arange(self.W)[None, :]

    def gather(self, x: torch.Tensor) -> torch.Tensor:
        """Full-length (A*K, fq*T_pad, zdim) -> windows (A*n_w*K, fq*W, zdim)."""
        B, L, z = x.shape
        d = L // self.T_pad * z
        xf = x.reshape(self.A, self.K, self.T_pad, d)[:, :, self.frame_index().to(x.device)]  # (A, K, n_w, W, d)
        return xf.permute(0, 2, 1, 3, 4).reshape(self.n_seq, -1, z).contiguous()

    def assembly_index(self) -> Tuple[torch.Tensor, torch.Tensor]:
        """(window, row) of every absolute frame f < T: window w gives its rows [0, S), the last window all its rows."""
        f = torch.arange(self.T)
        w = torch.clamp(f // self.S, max=self.n_w - 1)
        return w, f - w * self.S

    def assemble(self, xw: torch.Tensor) -> torch.Tensor:
        """Windows (A*n_w*K, fq*W, zdim) -> (A*K, fq*T, zdim)."""
        n, L, z = xw.shape
        d = L // self.W * z
        w, row = (i.to(xw.device) for i in self.assembly_index())
        x = xw.reshape(self.A, self.n_w, self.K, self.W, d).permute(0, 2, 1, 3, 4)[:, :, w, row]  # (A, K, T, d)
        return x.reshape(self.A * self.K, -1, z).contiguous()

    # -- device tables ------------------------------------------------------------------------------------
    def weights(self) -> torch.Tensor:
        """Blend weight of window w + 1 at overlap row j: (j + 1) / (O + 1), fp32."""
        return (torch.arange(1, self.O + 1, dtype=torch.float64) / (self.O + 1)).to(torch.float32)

    def noise_keys(self, clip_index0: int, d: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """(clip, e4_offset) int64 per window sequence (fdm_noise_keys): the long sequence's global index, and the first
        float4 of the window within it, so every window covering a frame draws the same noise for it."""
        a = torch.arange(self.A)[:, None, None]
        w = torch.arange(self.n_w)[None, :, None]
        k = torch.arange(self.K)[None, None, :]
        clip = (clip_index0 + a * self.K + k).expand(self.A, self.n_w, self.K)
        e4 = (w * self.S * d // 4).expand(self.A, self.n_w, self.K)
        return clip.reshape(-1).to(torch.int64), e4.reshape(-1).to(torch.int64)


def plan_windows(P: Preset, shape, n_audio: int, n_samples: int, window: Optional[int] = None,
                 overlap: Optional[int] = None) -> WindowPlan:
    """The plan of a sample_long call with latent `shape` (B, fq*T, zdim) and (n_audio, n_samples) audio. Raises ValueError
    for a window the model cannot use or audio too short for T frames."""
    if len(shape) != 3 or shape[1] % P.fq or shape[2] != P.zdim or shape[1] <= 0:
        raise ValueError(f"latent shape {tuple(shape)} is not (B, {P.fq}*T, {P.zdim})")
    B, T = int(shape[0]), int(shape[1]) // P.fq
    if n_audio < 1 or B % n_audio:
        raise ValueError(f"{B} sequences do not split evenly over {n_audio} audio clips")
    dw, do = default_window(P)
    W = dw if window is None else window
    O = do if overlap is None else overlap
    for name, v in (("window", W), ("overlap", O)):
        if not isinstance(v, int) or isinstance(v, bool):
            raise ValueError(f"{name} must be an int number of frames, got {v!r}")
    if W > MAX_WINDOW:
        raise ValueError(f"window {W} is longer than the {MAX_WINDOW} frames the model was trained on")
    if not 1 <= O <= W // 2:
        raise ValueError(f"overlap {O} must lie in [1, window // 2 = {W // 2}] (a frame lies in at most two windows)")
    if (W - O) % P.period:
        raise ValueError(f"window - overlap = {W - O} must be a multiple of the period {P.period}, so that every window's "
                         "periodic positional encoding is in phase with absolute time")
    r = 2 if P.pair_audio else 1
    have = conv_out_len(int(n_samples)) // r
    if have < T:
        raise ValueError(f"latent has {T} frames but the audio only yields {have}")
    return WindowPlan(A=int(n_audio), K=B // int(n_audio), T=T, W=W, O=O, r=r)
