"""ctypes binding of libfdm_b200.so (C ABI declared in include/fdm_b200.h).

PyTorch is used only for device memory and streams: every wrapper takes torch CUDA tensors, passes
``data_ptr()`` + explicit sizes/strides to the library and launches on torch's current stream.
There is no CPU or eager fallback: a missing library or a non-sm_100 device is a hard error.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FDM_B200_LIB") or os.path.join(_HERE, "libfdm_b200.so")  # override: instrumented builds (tools/)

F32, BF16 = 0, 1
ACT_NONE, ACT_RELU, ACT_MISH, ACT_GELU_ERF, ACT_GELU_TANH, ACT_LEAKY02 = range(6)

_vp, _i64, _i32, _f32, _u64 = C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_uint64


class GemmArgs(C.Structure):
    _fields_ = [("A", _vp), ("lda", _i64), ("a_rows", _i64), ("W", _vp), ("ldw", _i64), ("bias", _vp),
                ("residual", _vp), ("ldr", _i64), ("res_dtype", _i32), ("out_dtype", _i32), ("C", _vp),
                ("ldc", _i64), ("M", _i64), ("N", _i64), ("K", _i64), ("act", _i32), ("taps", _i32),
                ("tap_k", _i64), ("tap_row_shift", _i64), ("a_ln", _vp), ("w_colsum", _vp), ("res_ln", _vp),
                ("res_gamma", _vp), ("res_beta", _vp), ("stats_out", _vp), ("A_lo", _vp), ("W_lo", _vp),
                ("a_group_cols", _i64), ("splitk_ws", _vp), ("splitk_ws_bytes", _i64)]


class NormArgs(C.Structure):
    _fields_ = [("x", _vp), ("ldx", _i64), ("x_dtype", _i32), ("r1", _vp), ("ldr1", _i64), ("r1_dtype", _i32),
                ("g1", _vp), ("b1", _vp), ("act1", _i32), ("r2", _vp), ("ldr2", _i64), ("r2_dtype", _i32),
                ("r2_rows", _i64), ("vec2", _vp), ("vec_index_dev", _vp), ("g2", _vp), ("b2", _vp), ("out", _vp), ("ldo", _i64),
                ("out_dtype", _i32), ("out2", _vp), ("ldo2", _i64), ("out2_dtype", _i32), ("rows", _i64),
                ("d", _i64), ("eps", _f32)]


class AttnArgs(C.Structure):
    _fields_ = [("Q", _vp), ("K", _vp), ("V", _vp), ("ldq", _i64), ("ldk", _i64), ("ldv", _i64), ("O", _vp),
                ("ldo", _i64), ("dtype", _i32), ("B", _i64), ("T", _i64), ("t_stride", _i64), ("H", _i64),
                ("dh", _i64), ("scale", _f32), ("bias_mode", _i32), ("period", _i32), ("slopes", _vp)]


class DdpmArgs(C.Structure):
    _fields_ = [("x0_cond", _vp), ("x0_uncond", _vp), ("guidance", _f32), ("x_t", _vp), ("noise", _vp),
                ("out", _vp), ("out_bf16", _vp), ("c1", _vp), ("c2", _vp), ("sigma", _vp), ("t_per_clip", _vp),
                ("t_dev", _vp), ("B", _i64), ("elems_per_clip", _i64), ("seed", _u64),
                ("clip_index0", _i64), ("seed_dev", _vp)]


class DdimArgs(C.Structure):
    _fields_ = [("x0_cond", _vp), ("x0_uncond", _vp), ("guidance", _f32), ("x_t", _vp), ("out", _vp), ("out_bf16", _vp),
                ("a_recip", _vp), ("a_recipm1", _vp), ("sqrt_an", _vp), ("c", _vp), ("index_dev", _vp), ("n", _i64)]


class KnownArgs(C.Structure):
    _fields_ = [("x", _vp), ("x_bf16", _vp), ("known", _vp), ("mask", _vp), ("noise", _vp), ("ka", _vp), ("kb", _vp),
                ("index_dev", _vp), ("offset", _i32), ("seed_dev", _vp), ("t_dev", _vp), ("clip_index0", _i64),
                ("B", _i64), ("T", _i64), ("d", _i64)]


EXPORTS = {
    "fdm_last_error": (C.c_char_p, []),
    "fdm_device_info": (C.c_int, [C.POINTER(_i32)] * 3),
    "fdm_abi_version": (C.c_int, []),
    "fdm_gemm_set_option": (C.c_int, [C.c_char_p, _i32]),
    "fdm_gemm_bf16": (C.c_int, [C.POINTER(GemmArgs), _vp]),
    "fdm_gemm_f32": (C.c_int, [C.POINTER(GemmArgs), _vp]),
    "fdm_ln_stats_finalize": (C.c_int, [_vp, _i64, _i64, _i64, _f32, _vp, _vp]),
    "fdm_layernorm": (C.c_int, [C.POINTER(NormArgs), _vp]),
    "fdm_leaky_instnorm": (C.c_int, [_vp, _i32, _vp, _i32, _i64, _i64, _i64, _i64, _i64, _f32, _f32, _vp, _vp, _i32, _vp]),
    "fdm_self_attention": (C.c_int, [C.POINTER(AttnArgs), _vp]),
    "fdm_ddpm_step": (C.c_int, [C.POINTER(DdpmArgs), _vp]),
    "fdm_ddim_step": (C.c_int, [C.POINTER(DdimArgs), _vp]),
    "fdm_known_frames": (C.c_int, [C.POINTER(KnownArgs), _vp]),
    "fdm_advance_cursor": (C.c_int, [_vp, _vp, _i32, _vp, _vp]),
    "fdm_philox_normal": (C.c_int, [_vp, _i64, _i64, _u64, _i64, _i32, _vp]),
    "fdm_vq_quantize": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _i64, _i64, _vp, _vp, _vp, _vp]),
    "fdm_vq_quantize_ex": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _i64, _i64, _vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    "fdm_vq_stats": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _vp, _i64, _vp, _vp]),
    "fdm_split_bf16x2": (C.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "fdm_cast": (C.c_int, [_vp, _i32, _vp, _i32, _i64, _vp]),
    "fdm_cast_rows": (C.c_int, [_vp, _i64, _vp, _i32, _i64, _i64, _i64, _vp]),
    "fdm_audio_normalize_pad": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _f32, _vp]),
    "fdm_resample_poly": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _vp, _i64, _i64, _i64, _i64, _vp]),
    "fdm_vertex_error": (C.c_int, [_vp, _vp, _i64, _i64, _vp, _i64, _i32, _vp, _vp]),
    "fdm_transpose_bcl_to_blc": (C.c_int, [_vp, _vp, _i32, _i64, _i64, _i64, _vp]),
    "fdm_pad_time": (C.c_int, [_vp, _i64, _vp, _i32, _i64, _i64, _i64, _i64, _i64, _i32, _vp]),
    "fdm_hubert_conv0": (C.c_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i64, _i64, _vp]),
}

_lib = None
_device_checked = False


class FdmError(RuntimeError):
    pass


ABI_VERSION = 4  # fdm_abi_version() of the library these ctypes structs mirror


def load() -> C.CDLL:
    """dlopen the library and bind every symbol include/fdm_b200.h declares (no GPU needed)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FdmError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in EXPORTS.items():
            try:
                fn = getattr(lib, name)
            except AttributeError:  # a library built from older sources
                raise FdmError(f"{LIB_PATH} does not export {name}: rebuild it "
                               "(`python -c 'import __graft_entry__ as g; g.build()'`)") from None
            fn.restype, fn.argtypes = res, args
        if lib.fdm_abi_version() != ABI_VERSION:  # a stale build would read the argument structs with another layout
            raise FdmError(f"{LIB_PATH} has ABI version {lib.fdm_abi_version()}, this binding needs {ABI_VERSION}: rebuild it "
                           "(`python -c 'import __graft_entry__ as g; g.build()'`)")
        _lib = lib
    return _lib


class _NullRange:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


class _NvtxRange:
    def __init__(self, name: str):
        self.name = name

    def __enter__(self):
        torch.cuda.nvtx.range_push(self.name)
        return self

    def __exit__(self, *exc):
        torch.cuda.nvtx.range_pop()
        return False


NVTX = os.environ.get("FDM_B200_NVTX", "0") == "1"
_NULL_RANGE = _NullRange()


def nvtx_range(name: str):
    """NVTX range around one stage of the sampling job (audio encoder, prepare, sampling loop, tail, quantise, decode,
    gather) when FDM_B200_NVTX=1: `ncu --nvtx --nvtx-include "fdm/decode/"` then profiles exactly that stage. Off by
    default (a no-op context manager)."""
    return _NvtxRange("fdm/" + name) if NVTX else _NULL_RANGE


def require_device() -> C.CDLL:
    """Library + an sm_100 device, or raise."""
    global _device_checked
    lib = load()
    if not _device_checked:
        if not torch.cuda.is_available():
            raise FdmError("libfdm_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        sm, mj, mn = _i32(), _i32(), _i32()
        _check(lib.fdm_device_info(C.byref(sm), C.byref(mj), C.byref(mn)))
        _device_checked = True
    return lib


def _check(rc: int) -> None:
    if rc != 0:
        raise FdmError(load().fdm_last_error().decode())


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise FdmError(f"unsupported dtype {t.dtype}")


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None:
        return None
    assert t.is_cuda, "libfdm_b200 operates on CUDA tensors only"
    return t.data_ptr()


launch_count = 0  # number of library kernels launched by this process (bench.py reports it)


def _launched(n: int = 1) -> None:
    global launch_count
    launch_count += n


# ------------------------------------------------------------------------------------------------
class Split:
    """A tensor as a bf16 pair x = hi + lo (split-bf16 / "bf16x3" operand of the tcgen05 GEMM): fp32-grade products
    (2^-17 relative) at three tensor-core passes. `hi` and `lo` have identical shapes / strides; indexing slices both."""
    __slots__ = ("hi", "lo")

    def __init__(self, hi: torch.Tensor, lo: torch.Tensor):
        assert hi.dtype == lo.dtype == torch.bfloat16 and hi.shape == lo.shape and hi.stride() == lo.stride()
        self.hi, self.lo = hi, lo

    def __getitem__(self, idx) -> "Split":
        return Split(self.hi[idx], self.lo[idx])

    shape = property(lambda self: self.hi.shape)
    dtype = property(lambda self: "bf16x2")

    def dim(self):
        return self.hi.dim()

    def stride(self, *a):
        return self.hi.stride(*a)

    def float(self) -> torch.Tensor:
        return self.hi.float() + self.lo.float()


def split(x: torch.Tensor) -> Split:
    """fp32 tensor (contiguous) -> Split(hi, lo) of the same shape."""
    assert x.dtype == torch.float32 and x.is_contiguous() and x.is_cuda
    hi = torch.empty_like(x, dtype=torch.bfloat16)
    lo = torch.empty_like(x, dtype=torch.bfloat16)
    _check(require_device().fdm_split_bf16x2(_ptr(x), _ptr(hi), _ptr(lo), x.numel(), _stream()))
    _launched()
    return Split(hi, lo)


_SPLITK_WS = {}
SPLITK_WS_BYTES = 20 << 20
# Off by default: measured slower than the plain schedule in its current form (the finalising warp's dependent global
# round trips cost 7-14 us per GEMM against 3-6 us saved, profiles/README.md r02_h), and per-element summation order then
# depends on the tile schedule, i.e. on the batch size. FDM_B200_GEMM_TAILK=1 (or lib.splitk_enabled = True) turns it on.
splitk_enabled = os.environ.get("FDM_B200_GEMM_TAILK", "0") == "1"


def _splitk_workspace(device) -> Optional[torch.Tensor]:
    """Per-device workspace of the GEMM's tail split-K (fdm_gemm_args.splitk_ws). Kernels ordered on one stream or graph
    share it; code that runs GEMMs CONCURRENTLY on several streams sets lib.splitk_enabled = False. Never allocated during
    stream capture (a capture that starts before any eager GEMM on the device simply runs without the split)."""
    if not splitk_enabled:
        return None
    idx = device.index if device.index is not None else torch.cuda.current_device()
    ws = _SPLITK_WS.get(idx)
    if ws is None:
        if torch.cuda.is_current_stream_capturing():
            return None
        ws = _SPLITK_WS[idx] = torch.zeros(SPLITK_WS_BYTES, dtype=torch.uint8, device=device)
    return ws


def gemm(a: torch.Tensor, w: torch.Tensor, out: torch.Tensor, bias: Optional[torch.Tensor] = None,
         act: int = ACT_NONE, residual: Optional[torch.Tensor] = None, *, M: Optional[int] = None,
         lda: Optional[int] = None, a_rows: Optional[int] = None, taps: int = 1, tap_k: int = 0,
         tap_row_shift: int = 0, K: Optional[int] = None, a_ln: Optional[torch.Tensor] = None,
         w_colsum: Optional[torch.Tensor] = None, res_ln: Optional[torch.Tensor] = None,
         res_gamma: Optional[torch.Tensor] = None, res_beta: Optional[torch.Tensor] = None,
         stats_out: Optional[torch.Tensor] = None, a_group_cols: int = 0) -> torch.Tensor:
    """out[M,N] = act(a[M,K] @ w[N,K]^T + bias) + residual; bf16 operands -> tcgen05, f32 -> FFMA.
    a_group_cols > 0: grouped (block-diagonal) mode of fdm_gemm_bf16, see fdm_gemm_args.a_group_cols.

    `a` may be any tensor whose storage holds the rows (lda/a_rows/M override the 2-D view for implicit
    convolutions); `out`/`residual` are 2-D with unit inner stride."""
    lib = require_device()
    a_lo = w_lo = None
    if isinstance(w, Split):  # split-bf16 operands: A_lo W^T + A W_lo^T + A W^T in one accumulator (fdm_gemm_args.A_lo / W_lo)
        if not isinstance(a, Split):
            a = split(a)
        assert a.hi.data_ptr() % 16 == 0 and a.lo.data_ptr() % 16 == 0
        a, a_lo, w, w_lo = a.hi, a.lo, w.hi, w.lo
        assert a_lo.stride() == a.stride() and w_lo.stride() == w.stride()
    assert a.dtype == w.dtype and w.dim() == 2 and w.stride(1) == 1 and out.dim() == 2 and out.stride(1) == 1
    N = w.shape[0]
    Kk = K if K is not None else w.shape[1]
    g = GemmArgs()
    g.A, g.W, g.C = _ptr(a), _ptr(w), _ptr(out)
    g.lda = lda if lda is not None else a.stride(0)
    g.M = M if M is not None else a.shape[0]
    g.a_rows = a_rows if a_rows is not None else (a.shape[0] if a.dim() == 2 else g.M)
    g.ldw = w.stride(0)
    g.bias = _ptr(bias)
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.numel() == N
    g.residual = _ptr(residual)
    g.ldr = residual.stride(0) if residual is not None else 0
    g.res_dtype = _dt(residual) if residual is not None else F32
    g.out_dtype = _dt(out)
    g.ldc = out.stride(0)
    g.N, g.K = N, Kk
    g.act, g.taps, g.tap_k, g.tap_row_shift = act, taps, tap_k, tap_row_shift
    # LayerNorm folding (bf16 path; see fdm_gemm_args)
    g.a_ln, g.w_colsum, g.res_ln = _ptr(a_ln), _ptr(w_colsum), _ptr(res_ln)
    g.res_gamma, g.res_beta, g.stats_out = _ptr(res_gamma), _ptr(res_beta), _ptr(stats_out)
    g.A_lo, g.W_lo = _ptr(a_lo), _ptr(w_lo)
    g.a_group_cols = a_group_cols
    ws = _splitk_workspace(a.device) if (a.dtype == torch.bfloat16 and a_lo is None) else None
    if ws is not None:
        g.splitk_ws, g.splitk_ws_bytes = _ptr(ws), ws.numel()
    if stats_out is not None:
        assert stats_out.dtype == torch.float32 and stats_out.numel() >= g.M * (N // 64) * 2
    assert out.shape[0] >= g.M and out.shape[1] == N
    fn = lib.fdm_gemm_bf16 if a.dtype == torch.bfloat16 else lib.fdm_gemm_f32
    _check(fn(C.byref(g), _stream()))
    _launched()
    return out


def gemm_set_option(name: str, value: int) -> None:
    """Process-wide kernel-selection switch of fdm_gemm_bf16 (see include/fdm_b200.h), e.g. ("resmma", 1)."""
    _check(load().fdm_gemm_set_option(name.encode(), int(value)))


def ln_stats_finalize(partials: torch.Tensor, M: int, parts: int, d: int, out: torch.Tensor, eps: float = 1e-5) -> torch.Tensor:
    """(mean, rstd) per row [M, 2] from the [M, parts, 2] partial statistics written by gemm(..., stats_out=...)."""
    assert partials.dtype == torch.float32 and out.dtype == torch.float32 and out.numel() >= 2 * M
    _check(require_device().fdm_ln_stats_finalize(_ptr(partials), M, parts, d, eps, _ptr(out), _stream()))
    _launched()
    return out


def layernorm(x: torch.Tensor, out: torch.Tensor, g1=None, b1=None, r1=None, act1: int = ACT_NONE, r2=None,
              vec2=None, vec_index_dev=None, g2=None, b2=None, out2=None, eps: float = 1e-5) -> torch.Tensor:
    lib = require_device()
    n = NormArgs()
    d = x.shape[-1]
    x2 = x.reshape(-1, d) if x.is_contiguous() else x
    assert x2.dim() == 2 and x2.stride(1) == 1
    n.x, n.ldx, n.x_dtype = _ptr(x2), x2.stride(0), _dt(x2)

    def two_d(t):
        t2 = t.reshape(-1, d) if t.is_contiguous() else t
        assert t2.dim() == 2 and t2.stride(1) == 1 and t2.shape[0] >= x2.shape[0]
        return t2

    if r1 is not None:
        r = two_d(r1); n.r1, n.ldr1, n.r1_dtype = _ptr(r), r.stride(0), _dt(r)
    if r2 is not None:
        r = r2.reshape(-1, d) if r2.is_contiguous() else r2
        assert r.dim() == 2 and r.stride(1) == 1 and x2.shape[0] % r.shape[0] == 0
        n.r2, n.ldr2, n.r2_dtype = _ptr(r), r.stride(0), _dt(r)
        n.r2_rows = 0 if r.shape[0] == x2.shape[0] else r.shape[0]
    n.g1, n.b1, n.g2, n.b2 = _ptr(g1), _ptr(b1), _ptr(g2), _ptr(b2)
    n.act1 = act1
    n.vec2, n.vec_index_dev = _ptr(vec2), _ptr(vec_index_dev)
    o = two_d(out); n.out, n.ldo, n.out_dtype = _ptr(o), o.stride(0), _dt(o)
    if out2 is not None:
        o2 = two_d(out2); n.out2, n.ldo2, n.out2_dtype = _ptr(o2), o2.stride(0), _dt(o2)
    n.rows, n.d, n.eps = x2.shape[0], d, eps
    _check(lib.fdm_layernorm(C.byref(n), _stream()))
    _launched()
    return out


def leaky_instnorm(x: torch.Tensor, out: torch.Tensor, B: int, T: int, t_stride: int, Cn: int,
                   slope: float = 0.2, eps: float = 1e-5, out_t_stride: Optional[int] = None, gamma=None, beta=None,
                   post_act: int = ACT_NONE) -> torch.Tensor:
    lib = require_device()
    _check(lib.fdm_leaky_instnorm(_ptr(x), _dt(x), _ptr(out), _dt(out), B, T, t_stride,
                                  out_t_stride if out_t_stride is not None else t_stride, Cn, slope, eps,
                                  _ptr(gamma), _ptr(beta), post_act, _stream()))
    _launched()
    return out


def self_attention(q, k, v, out, B: int, T: int, t_stride: int, H: int, dh: int, scale: float,
                   slopes: Optional[torch.Tensor] = None, period: int = 0) -> torch.Tensor:
    """q/k/v/out: 2-D row views (row = b*t_stride + t) whose column 0 is head 0 of the respective operand."""
    lib = require_device()
    a = AttnArgs()
    a.Q, a.K, a.V, a.O = _ptr(q), _ptr(k), _ptr(v), _ptr(out)
    a.ldq, a.ldk, a.ldv, a.ldo = q.stride(0), k.stride(0), v.stride(0), out.stride(0)
    a.dtype = _dt(q)
    assert q.dtype == k.dtype == v.dtype == out.dtype
    a.B, a.T, a.t_stride, a.H, a.dh, a.scale = B, T, t_stride, H, dh, scale
    a.bias_mode = 1 if slopes is not None else 0
    a.period = period
    a.slopes = _ptr(slopes)
    _check(lib.fdm_self_attention(C.byref(a), _stream()))
    _launched()
    return out


def ddpm_step(x0_cond, x_t, out, c1, c2, sigma, *, x0_uncond=None, guidance: float = 0.0, noise=None,
              out_bf16=None, t_per_clip=None, t_dev=None, seed: int = 0,
              clip_index0: int = 0, seed_dev: Optional[torch.Tensor] = None) -> torch.Tensor:
    lib = require_device()
    a = DdpmArgs()
    B = x_t.shape[0]
    for t in (x0_cond, x_t, out, x0_uncond, noise):
        assert t is None or (t.dtype == torch.float32 and t.is_contiguous() and t.numel() == x_t.numel())
    a.x0_cond, a.x0_uncond, a.guidance = _ptr(x0_cond), _ptr(x0_uncond), guidance
    a.x_t, a.noise, a.out, a.out_bf16 = _ptr(x_t), _ptr(noise), _ptr(out), _ptr(out_bf16)
    a.c1, a.c2, a.sigma = _ptr(c1), _ptr(c2), _ptr(sigma)
    if t_per_clip is not None:
        assert t_per_clip.dtype == torch.int64 and t_per_clip.numel() == B
    a.t_per_clip, a.t_dev = _ptr(t_per_clip), _ptr(t_dev)
    a.B, a.elems_per_clip = B, x_t.numel() // B
    a.seed, a.clip_index0 = seed, clip_index0
    if seed_dev is not None:  # Philox seed read from device memory (int64[1]): replayable graphs, fresh seed per call
        assert seed_dev.dtype == torch.int64 and seed_dev.numel() == 1
    a.seed_dev = _ptr(seed_dev)
    _check(lib.fdm_ddpm_step(C.byref(a), _stream()))
    _launched()
    return out


def ddim_step(x0_cond, x_t, out, a_recip, a_recipm1, sqrt_an, c, index_dev, *, x0_uncond=None, guidance: float = 0.0,
              out_bf16=None) -> torch.Tensor:
    lib = require_device()
    a = DdimArgs()
    for t in (x0_cond, x_t, out, x0_uncond):
        assert t is None or (t.dtype == torch.float32 and t.is_contiguous() and t.numel() == x_t.numel())
    a.x0_cond, a.x0_uncond, a.guidance = _ptr(x0_cond), _ptr(x0_uncond), guidance
    a.x_t, a.out, a.out_bf16 = _ptr(x_t), _ptr(out), _ptr(out_bf16)
    a.a_recip, a.a_recipm1, a.sqrt_an, a.c = _ptr(a_recip), _ptr(a_recipm1), _ptr(sqrt_an), _ptr(c)
    assert index_dev.dtype == torch.int32
    a.index_dev, a.n = _ptr(index_dev), x_t.numel()
    _check(lib.fdm_ddim_step(C.byref(a), _stream()))
    _launched()
    return out


def known_frames(x, known, mask, ka, kb, index_dev, *, offset: int = 0, noise=None, x_bf16=None,
                 seed_dev: Optional[torch.Tensor] = None, t_dev: Optional[torch.Tensor] = None, clip_index0: int = 0) -> torch.Tensor:
    """Known-frame replacement in place (fdm_known_frames): x (B, ...) fp32 holds B sequences of mask.numel() / B rows;
    rows whose uint8 mask is set become ka[i] * known + kb[i] * z with i = index_dev[0] + offset, z from `noise` (may be
    x itself) or, when noise is None, the Philox draw of (seed_dev[0], clip_index0 + b, t_dev[0], element)."""
    lib = require_device()
    a = KnownArgs()
    B, rows = x.shape[0], mask.numel()
    for t in (x, known, noise):
        assert t is None or (t.dtype == torch.float32 and t.is_contiguous() and t.numel() == x.numel())
    assert mask.dtype == torch.uint8 and mask.is_contiguous() and rows % B == 0 and x.numel() % rows == 0
    assert ka.dtype == kb.dtype == torch.float32 and index_dev.dtype == torch.int32
    if x_bf16 is not None:
        assert x_bf16.dtype == torch.bfloat16 and x_bf16.is_contiguous() and x_bf16.numel() == x.numel()
    if seed_dev is not None:
        assert seed_dev.dtype == torch.int64 and seed_dev.numel() == 1
    if t_dev is not None:
        assert t_dev.dtype == torch.int32 and t_dev.numel() == 1
    a.x, a.x_bf16, a.known, a.mask, a.noise = _ptr(x), _ptr(x_bf16), _ptr(known), _ptr(mask), _ptr(noise)
    a.ka, a.kb, a.index_dev, a.offset = _ptr(ka), _ptr(kb), _ptr(index_dev), offset
    a.seed_dev, a.t_dev, a.clip_index0 = _ptr(seed_dev), _ptr(t_dev), clip_index0
    a.B, a.T, a.d = B, rows // B, x.numel() // rows
    _check(lib.fdm_known_frames(C.byref(a), _stream()))
    _launched()
    return x


def advance_cursor(cursor: torch.Tensor, t_sched: torch.Tensor, t_dev: torch.Tensor) -> None:
    assert cursor.dtype == t_sched.dtype == t_dev.dtype == torch.int32
    _check(require_device().fdm_advance_cursor(_ptr(cursor), _ptr(t_sched), t_sched.numel(), _ptr(t_dev), _stream()))
    _launched()


def philox_normal(out: torch.Tensor, seed: int, clip_index0: int, t: int) -> torch.Tensor:
    B = out.shape[0]
    _check(require_device().fdm_philox_normal(_ptr(out), B, out.numel() // B, seed, clip_index0, t, _stream()))
    _launched()
    return out


VQ_AUTO, VQ_FFMA, VQ_TENSOR = 0, 1, 2


def vq_quantize(z: torch.Tensor, codebook: torch.Tensor, n_codes: int, code_offset=None, want_bdl=True,
                want_rows=False, algo: int = VQ_AUTO, recheck_rows: Optional[torch.Tensor] = None,
                dbg_acc: Optional[torch.Tensor] = None):
    """z (B, L, D) f32 -> (indices (B*L, 1) int64, z_q (B, D, L) or None, z_q rows (B, L, D) or None).
    algo: VQ_AUTO (tensor-core filter + exact recheck when D = 64 / 128), VQ_FFMA, VQ_TENSOR; identical indices either way.
    recheck_rows: optional zeroed int64[1] device counter of rows that took the exact pass (tensor path);
    dbg_acc: optional (B*L, n_codes) f32 dump of the tensor-core dot products (tests)."""
    lib = require_device()
    assert z.dtype == torch.float32 and z.is_contiguous() and codebook.dtype == torch.float32 and codebook.is_contiguous()
    B, L, D = z.shape
    idx = torch.empty((B * L, 1), dtype=torch.int64, device=z.device)
    zq = torch.empty((B, D, L), dtype=torch.float32, device=z.device) if want_bdl else None
    zr = torch.empty((B, L, D), dtype=torch.float32, device=z.device) if want_rows else None
    if code_offset is not None:
        assert code_offset.dtype == torch.int64 and code_offset.numel() == B
    if recheck_rows is not None:
        assert recheck_rows.dtype == torch.int64 and recheck_rows.numel() == 1
    if dbg_acc is not None:
        assert dbg_acc.dtype == torch.float32 and dbg_acc.is_contiguous() and dbg_acc.numel() == B * L * n_codes
    _check(lib.fdm_vq_quantize_ex(_ptr(z), _ptr(codebook), _ptr(code_offset), B, L, D, n_codes, _ptr(idx), _ptr(zq),
                                  _ptr(zr), algo, _ptr(recheck_rows), _ptr(dbg_acc), _stream()))
    _launched()
    return idx, zq, zr


def cast_rows(src: torch.Tensor, dst: torch.Tensor) -> torch.Tensor:
    """dst[r, :] = cast(src[r, :]) zero-padded to dst's row length (f32 source, f32 / bf16 destination)."""
    assert src.dtype == torch.float32 and src.dim() == 2 and dst.dim() == 2 and src.stride(1) == 1 and dst.stride(1) == 1
    assert dst.shape[0] == src.shape[0] and dst.shape[1] >= src.shape[1]
    _check(require_device().fdm_cast_rows(_ptr(src), src.stride(0), _ptr(dst), _dt(dst), dst.stride(0), src.shape[0],
                                          src.shape[1], _stream()))
    _launched()
    return dst


def audio_normalize_pad(audio: torch.Tensor, pad_samples: int = 0, eps: float = 1e-7) -> torch.Tensor:
    """Wav2Vec2Processor normalisation + zero tail on device (demo/demo_3d_mead.py:85-97). audio (B, L) f32."""
    assert audio.dtype == torch.float32 and audio.dim() == 2 and audio.is_contiguous()
    B, L = audio.shape
    out = torch.empty(B, L + pad_samples, device=audio.device, dtype=torch.float32)
    _check(require_device().fdm_audio_normalize_pad(_ptr(audio), B, L, _ptr(out), L + pad_samples, eps, _stream()))
    _launched()
    return out


def vq_stats(z: torch.Tensor, codebook: torch.Tensor, indices: torch.Tensor, n_codes: int,
             code_offset: Optional[torch.Tensor] = None):
    """(sum of (e_idx - z)^2 over all elements as a 0-d fp64 tensor, code histogram int64[n_codes]) in one pass over z."""
    assert z.dtype == torch.float32 and z.dim() == 3 and z.is_contiguous() and codebook.dtype == torch.float32 and codebook.is_contiguous()
    assert indices.dtype == torch.int64 and indices.is_contiguous() and indices.numel() == z.shape[0] * z.shape[1]
    B, L, D = z.shape
    n_part = int(min(8 * 148, max(1, (B * L + 63) // 64)))
    partials = torch.empty(n_part, device=z.device, dtype=torch.float32)
    hist = torch.zeros(n_codes, device=z.device, dtype=torch.int64)
    _check(require_device().fdm_vq_stats(_ptr(z), _ptr(codebook), _ptr(code_offset), _ptr(indices), B, L, D, n_codes,
                                         _ptr(partials), n_part, _ptr(hist), _stream()))
    _launched()
    return partials.double().sum(), hist


def resample_poly(audio: torch.Tensor, taps: torch.Tensor, up: int, down: int, pre: int, n_out: int) -> torch.Tensor:
    """Polyphase FIR resampling on device (scipy.signal.resample_poly semantics; see fdm_resample_poly). audio (B, L) f32."""
    assert audio.dtype == torch.float32 and audio.dim() == 2 and audio.is_contiguous()
    assert taps.dtype == torch.float32 and taps.is_contiguous() and taps.device == audio.device
    B, L = audio.shape
    out = torch.empty(B, n_out, device=audio.device, dtype=torch.float32)
    _check(require_device().fdm_resample_poly(_ptr(audio), B, L, _ptr(out), n_out, _ptr(taps), taps.numel(), up, down, pre, _stream()))
    _launched()
    return out


def vertex_error(pred: torch.Tensor, gt: Optional[torch.Tensor], vertex_idx: Optional[torch.Tensor] = None,
                 mode: str = "max") -> torch.Tensor:
    """Per-frame max / mean over a vertex subset of the squared L2 error (metric/metric.py:115-138).
    pred, gt: (frames, V*3) or (frames, V, 3) f32; returns (frames,) f32 — the metric is its mean."""
    assert pred.dtype == torch.float32 and pred.is_contiguous()
    F_ = pred.shape[0]
    V = pred.numel() // F_ // 3
    if gt is not None:
        assert gt.dtype == torch.float32 and gt.is_contiguous() and gt.numel() == pred.numel()
    if vertex_idx is not None:
        assert vertex_idx.dtype == torch.int64 and vertex_idx.is_contiguous()
    out = torch.empty(F_, device=pred.device, dtype=torch.float32)
    _check(require_device().fdm_vertex_error(_ptr(pred), _ptr(gt), F_, V, _ptr(vertex_idx),
                                             vertex_idx.numel() if vertex_idx is not None else 0,
                                             0 if mode == "max" else 1, _ptr(out), _stream()))
    _launched()
    return out


def cast(src: torch.Tensor, dst: torch.Tensor) -> torch.Tensor:
    assert src.is_contiguous() and dst.is_contiguous() and src.numel() == dst.numel()
    _check(require_device().fdm_cast(_ptr(src), _dt(src), _ptr(dst), _dt(dst), src.numel(), _stream()))
    _launched()
    return dst


def transpose_bcl_to_blc(src: torch.Tensor, dst: torch.Tensor) -> torch.Tensor:
    B, Cn, L = src.shape
    assert src.dtype == torch.float32 and src.is_contiguous() and dst.is_contiguous() and dst.numel() == src.numel()
    _check(require_device().fdm_transpose_bcl_to_blc(_ptr(src), _ptr(dst), _dt(dst), B, Cn, L, _stream()))
    _launched()
    return dst


def pad_time(src: torch.Tensor, dst: torch.Tensor, B: int, T: int, Cn: int, pad_l: int, pad_r: int, mode: int,
             src_t_stride: Optional[int] = None) -> torch.Tensor:
    assert src.dtype == dst.dtype and dst.numel() >= B * (pad_l + T + pad_r) * Cn
    _check(require_device().fdm_pad_time(_ptr(src), src_t_stride or T, _ptr(dst), _dt(src), B, T, Cn, pad_l, pad_r,
                                         mode, _stream()))
    _launched()
    return dst


def hubert_conv0(audio, w, bias, ln_g, ln_b, out, Lout: int, out_t_stride: int, Cn: int) -> torch.Tensor:
    B, L = audio.shape
    assert audio.dtype == torch.float32 and audio.is_contiguous()
    _check(require_device().fdm_hubert_conv0(_ptr(audio), B, L, _ptr(w), _ptr(bias), _ptr(ln_g), _ptr(ln_b),
                                             _ptr(out), _dt(out), Lout, out_t_stride, Cn, _stream()))
    _launched()
    return out
