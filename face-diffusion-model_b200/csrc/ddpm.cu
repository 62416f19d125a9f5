// fdm_ddpm_step: the fused diffusion-step update (SURVEY K7): classifier-free-guidance combine, DDPM posterior
// mean, and noise add in ONE vectorised, HBM-bound pass. 16 B/element (20 B with CFG) of algorithmic traffic
// when noise is streamed from HBM, 12/16 B when it is drawn in-kernel from Philox4x32-10.
#include "common.cuh"

namespace {

struct Philox {
  // Philox4x32-10 (Salmon et al. 2011); counter = (elem/4 lo, elem/4 hi, step t, clip), key = seed
  static __host__ __device__ __forceinline__ void mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
    const uint64_t p = static_cast<uint64_t>(a) * b;
    hi = static_cast<uint32_t>(p >> 32);
    lo = static_cast<uint32_t>(p);
  }
  static __host__ __device__ __forceinline__ void generate(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                                           uint32_t k1, uint32_t (&out)[4]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      uint32_t hi0, lo0, hi1, lo1;
      mulhilo(0xD2511F53u, c0, hi0, lo0);
      mulhilo(0xCD9E8D57u, c2, hi1, lo1);
      const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
      c0 = n0; c1 = n1; c2 = n2; c3 = n3;
      k0 += 0x9E3779B9u;
      k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
  }
};

// four standard normals for elements [4*e4, 4*e4+4) of clip `clip` at step `t`
__device__ __forceinline__ float4 philox_normal4(uint64_t seed, uint32_t clip, uint32_t t, uint64_t e4) {
  uint32_t r[4];
  Philox::generate(static_cast<uint32_t>(e4), static_cast<uint32_t>(e4 >> 32), t, clip, static_cast<uint32_t>(seed),
                   static_cast<uint32_t>(seed >> 32), r);
  const float inv24 = 5.9604644775390625e-08f;  // 2^-24
  const float u0 = static_cast<float>((r[0] >> 8) + 1u) * inv24;  // (0, 1]
  const float u1 = static_cast<float>(r[1] >> 8) * inv24;         // [0, 1)
  const float u2 = static_cast<float>((r[2] >> 8) + 1u) * inv24;
  const float u3 = static_cast<float>(r[3] >> 8) * inv24;
  const float ra = sqrtf(-2.f * logf(u0)), rb = sqrtf(-2.f * logf(u2));
  float sa, ca, sb, cb;
  sincospif(2.f * u1, &sa, &ca);  // sin / cos of 2 pi u without the range reduction of sincosf
  sincospif(2.f * u3, &sb, &cb);
  return make_float4(ra * ca, ra * sa, rb * cb, rb * sb);
}

// grid = (chunks, clips): a block walks one clip's float4 elements, two per thread and iteration (six 16-byte loads in
// flight before the Philox / Box-Muller arithmetic), so no 64-bit division sits in the loop and t / c1 / c2 / sigma are
// per-block constants.
__device__ __forceinline__ float4 ddpm_update(const fdm_ddpm_args& a, float4 x0, const float4& u, const float4& xt, float c1, float c2) {
  if (a.x0_uncond) {
    // u + s*(c - u), each op rounded separately (utiles/classifierfree.py:20-21)
    x0.x = __fadd_rn(u.x, __fmul_rn(a.guidance, __fsub_rn(x0.x, u.x)));
    x0.y = __fadd_rn(u.y, __fmul_rn(a.guidance, __fsub_rn(x0.y, u.y)));
    x0.z = __fadd_rn(u.z, __fmul_rn(a.guidance, __fsub_rn(x0.z, u.z)));
    x0.w = __fadd_rn(u.w, __fmul_rn(a.guidance, __fsub_rn(x0.w, u.w)));
  }
  float4 o;
  o.x = __fadd_rn(__fmul_rn(c1, x0.x), __fmul_rn(c2, xt.x));
  o.y = __fadd_rn(__fmul_rn(c1, x0.y), __fmul_rn(c2, xt.y));
  o.z = __fadd_rn(__fmul_rn(c1, x0.z), __fmul_rn(c2, xt.z));
  o.w = __fadd_rn(__fmul_rn(c1, x0.w), __fmul_rn(c2, xt.w));
  return o;
}
__device__ __forceinline__ void ddpm_store(const fdm_ddpm_args& a, int64_t i, float4 o, const float4& z, float sg, bool add_noise) {
  if (add_noise) {
    o.x = __fadd_rn(o.x, __fmul_rn(sg, z.x));
    o.y = __fadd_rn(o.y, __fmul_rn(sg, z.y));
    o.z = __fadd_rn(o.z, __fmul_rn(sg, z.z));
    o.w = __fadd_rn(o.w, __fmul_rn(sg, z.w));
  }
  reinterpret_cast<float4*>(a.out)[i] = o;
  if (a.out_bf16) {
    uint2 u;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
    h[0] = __floats2bfloat162_rn(o.x, o.y);
    h[1] = __floats2bfloat162_rn(o.z, o.w);
    reinterpret_cast<uint2*>(a.out_bf16)[i] = u;
  }
}

__global__ void __launch_bounds__(256) ddpm_step_kernel(const fdm_ddpm_args a, const int64_t e4_per_clip) {
  pdl_trigger();
  pdl_wait();
  const int64_t b = blockIdx.y;
  const int t = a.t_per_clip ? static_cast<int>(a.t_per_clip[b]) : *a.t_dev;
  const float c1 = a.c1[t], c2 = a.c2[t], sg = a.sigma[t];
  const bool add_noise = t > 0;
  const uint32_t clip = static_cast<uint32_t>(a.clip_index0 + b);
  const uint64_t seed = a.seed_dev ? *a.seed_dev : a.seed;  // device-resident seed: one captured graph, a fresh seed per call
  const int64_t base = b * e4_per_clip;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int64_t e0 = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; e0 < e4_per_clip; e0 += 2 * stride) {
    const int64_t e1 = e0 + stride;
    const bool two = e1 < e4_per_clip;
    const int64_t i0 = base + e0, i1 = base + (two ? e1 : e0);
    const float4 xa = reinterpret_cast<const float4*>(a.x0_cond)[i0];
    const float4 xb = reinterpret_cast<const float4*>(a.x0_cond)[i1];
    const float4 ua = a.x0_uncond ? reinterpret_cast<const float4*>(a.x0_uncond)[i0] : zero;
    const float4 ub = a.x0_uncond ? reinterpret_cast<const float4*>(a.x0_uncond)[i1] : zero;
    const float4 ta = reinterpret_cast<const float4*>(a.x_t)[i0];
    const float4 tb = reinterpret_cast<const float4*>(a.x_t)[i1];
    float4 za = zero, zb = zero;
    if (add_noise) {
      if (a.noise) {
        za = reinterpret_cast<const float4*>(a.noise)[i0];
        zb = reinterpret_cast<const float4*>(a.noise)[i1];
      } else {
        za = philox_normal4(seed, clip, static_cast<uint32_t>(t), static_cast<uint64_t>(e0));
        if (two) zb = philox_normal4(seed, clip, static_cast<uint32_t>(t), static_cast<uint64_t>(e1));
      }
    }
    ddpm_store(a, i0, ddpm_update(a, xa, ua, ta, c1, c2), za, sg, add_noise);
    if (two) ddpm_store(a, i1, ddpm_update(a, xb, ub, tb, c1, c2), zb, sg, add_noise);
  }
}

__global__ void __launch_bounds__(256) ddim_step_kernel(const fdm_ddim_args a, const int64_t n4) {
  pdl_trigger();
  pdl_wait();
  const int i0 = *a.index_dev;
  const float A = a.a_recip[i0], Bm = a.a_recipm1[i0], sa = a.sqrt_an[i0], c = a.c[i0];
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float4 x0 = reinterpret_cast<const float4*>(a.x0_cond)[i];
    if (a.x0_uncond) {
      const float4 u = reinterpret_cast<const float4*>(a.x0_uncond)[i];
      x0.x = __fadd_rn(u.x, __fmul_rn(a.guidance, __fsub_rn(x0.x, u.x)));
      x0.y = __fadd_rn(u.y, __fmul_rn(a.guidance, __fsub_rn(x0.y, u.y)));
      x0.z = __fadd_rn(u.z, __fmul_rn(a.guidance, __fsub_rn(x0.z, u.z)));
      x0.w = __fadd_rn(u.w, __fmul_rn(a.guidance, __fsub_rn(x0.w, u.w)));
    }
    const float4 xt = reinterpret_cast<const float4*>(a.x_t)[i];
    float4 o;
#define FDM_DDIM(X0, XT) __fadd_rn(__fmul_rn(X0, sa), __fmul_rn(c, __fdiv_rn(__fsub_rn(__fmul_rn(A, XT), X0), Bm)))
    o.x = FDM_DDIM(x0.x, xt.x);
    o.y = FDM_DDIM(x0.y, xt.y);
    o.z = FDM_DDIM(x0.z, xt.z);
    o.w = FDM_DDIM(x0.w, xt.w);
#undef FDM_DDIM
    reinterpret_cast<float4*>(a.out)[i] = o;
    if (a.out_bf16) {
      uint2 u;
      __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
      h[0] = __floats2bfloat162_rn(o.x, o.y);
      h[1] = __floats2bfloat162_rn(o.z, o.w);
      reinterpret_cast<uint2*>(a.out_bf16)[i] = u;
    }
  }
}

// grid = rows (one CTA per (sequence, frame) row). The mask is written by host copies before the sampling loop, never by
// the kernels this one follows, so a CTA may read it before pdl_wait(), and a CTA of an unknown row exits without waiting,
// except CTA 0: the grid must not complete before its predecessor has, or the next kernel's pdl_wait() (advance_cursor
// rewriting t_dev / cursor) would no longer order it after the step update, e.g. when no row is known.
__global__ void __launch_bounds__(128) known_frames_kernel(const fdm_known_args a, const int64_t d4) {
  pdl_trigger();
  const int64_t row = blockIdx.x;
  const bool known = a.mask[row] != 0;
  if (!known && row != 0) return;
  pdl_wait();
  if (!known) return;
  const int i = *a.index_dev + a.offset;
  const float ka = a.ka[i], kb = a.kb[i];
  const bool draw = kb != 0.f;
  const bool philox = draw && a.noise == nullptr;
  const int64_t b = row / a.T;
  const uint32_t clip = static_cast<uint32_t>(a.clip_index0 + b);
  const uint64_t seed = philox ? *a.seed_dev : 0;
  const uint32_t t = philox ? static_cast<uint32_t>(*a.t_dev) : 0u;
  const int64_t e4_0 = (row - b * a.T) * d4;  // first float4 of the row within its sequence (the Philox element counter)
  for (int64_t j = threadIdx.x; j < d4; j += blockDim.x) {
    const int64_t i4 = row * d4 + j;
    const float4 k = reinterpret_cast<const float4*>(a.known)[i4];
    float4 o = make_float4(__fmul_rn(ka, k.x), __fmul_rn(ka, k.y), __fmul_rn(ka, k.z), __fmul_rn(ka, k.w));
    if (draw) {
      const float4 z = philox ? philox_normal4(seed, clip, t, static_cast<uint64_t>(e4_0 + j))
                              : reinterpret_cast<const float4*>(a.noise)[i4];
      o.x = __fadd_rn(o.x, __fmul_rn(kb, z.x));
      o.y = __fadd_rn(o.y, __fmul_rn(kb, z.y));
      o.z = __fadd_rn(o.z, __fmul_rn(kb, z.z));
      o.w = __fadd_rn(o.w, __fmul_rn(kb, z.w));
    }
    reinterpret_cast<float4*>(a.x)[i4] = o;
    if (a.x_bf16) {
      uint2 u;
      __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
      h[0] = __floats2bfloat162_rn(o.x, o.y);
      h[1] = __floats2bfloat162_rn(o.z, o.w);
      reinterpret_cast<uint2*>(a.x_bf16)[i4] = u;
    }
  }
}

__global__ void advance_cursor_kernel(int32_t* cursor, const int32_t* sched, int n, int32_t* t_dev) {
  pdl_trigger();
  pdl_wait();
  const int c = *cursor + 1;
  *cursor = c;
  *t_dev = sched[c < n ? c : n - 1];
}

__global__ void __launch_bounds__(256) philox_fill_kernel(float* out, int64_t n4, int64_t e4_per_clip, uint64_t seed,
                                                          int64_t clip0, int t) {
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t b = i / e4_per_clip;
    reinterpret_cast<float4*>(out)[i] =
        philox_normal4(seed, static_cast<uint32_t>(clip0 + b), static_cast<uint32_t>(t), static_cast<uint64_t>(i - b * e4_per_clip));
  }
}

inline int grid_for(int64_t n4) {
  const int64_t want = ceil_div64(n4, 256);
  const int64_t cap = static_cast<int64_t>(fdm_sm_count()) * 8;  // 8 resident 256-thread CTAs per SM
  return static_cast<int>(want < cap ? (want > 0 ? want : 1) : cap);
}

}  // namespace

extern "C" int fdm_ddpm_step(const fdm_ddpm_args* args, void* stream) {
  FDM_CHECK_ARG(args != nullptr, "fdm_ddpm_step: null args");
  const fdm_ddpm_args& a = *args;
  FDM_CHECK_ARG(a.x0_cond && a.x_t && a.out && a.c1 && a.c2 && a.sigma, "fdm_ddpm_step: null operand");
  FDM_CHECK_ARG(a.t_per_clip || a.t_dev, "fdm_ddpm_step: need t_per_clip or t_dev");
  FDM_CHECK_ARG(a.B > 0 && a.elems_per_clip > 0 && a.elems_per_clip % 4 == 0, "fdm_ddpm_step: elems_per_clip must be a positive multiple of 4");
  const uintptr_t al = reinterpret_cast<uintptr_t>(a.x0_cond) | reinterpret_cast<uintptr_t>(a.x0_uncond) |
                       reinterpret_cast<uintptr_t>(a.x_t) | reinterpret_cast<uintptr_t>(a.noise) |
                       reinterpret_cast<uintptr_t>(a.out);
  FDM_CHECK_ARG(al % 16 == 0 && reinterpret_cast<uintptr_t>(a.out_bf16) % 8 == 0, "fdm_ddpm_step: operands must be 16-byte aligned");
  FDM_CHECK_ARG(a.B <= 65535, "fdm_ddpm_step: at most 65535 clips per call");
  const int64_t e4 = a.elems_per_clip / 4;
  // ~8 resident 256-thread CTAs per SM over the whole batch, two float4 per thread and iteration
  int64_t gx = ceil_div64(static_cast<int64_t>(fdm_sm_count()) * 8, a.B);
  const int64_t gx_max = ceil_div64(e4, 512);
  if (gx > gx_max) gx = gx_max;
  if (gx < 1) gx = 1;
  FDM_CHECK_CUDA(fdm_launch_pdl(ddpm_step_kernel, dim3(static_cast<unsigned>(gx), static_cast<unsigned>(a.B)), dim3(256), 0,
                                reinterpret_cast<cudaStream_t>(stream), 1, a, e4));
  return 0;
}

extern "C" int fdm_ddim_step(const fdm_ddim_args* args, void* stream) {
  FDM_CHECK_ARG(args != nullptr, "fdm_ddim_step: null args");
  const fdm_ddim_args& a = *args;
  FDM_CHECK_ARG(a.x0_cond && a.x_t && a.out && a.a_recip && a.a_recipm1 && a.sqrt_an && a.c && a.index_dev, "fdm_ddim_step: null operand");
  FDM_CHECK_ARG(a.n > 0 && a.n % 4 == 0, "fdm_ddim_step: n must be a positive multiple of 4");
  const uintptr_t al = reinterpret_cast<uintptr_t>(a.x0_cond) | reinterpret_cast<uintptr_t>(a.x0_uncond) |
                       reinterpret_cast<uintptr_t>(a.x_t) | reinterpret_cast<uintptr_t>(a.out);
  FDM_CHECK_ARG(al % 16 == 0 && reinterpret_cast<uintptr_t>(a.out_bf16) % 8 == 0, "fdm_ddim_step: operands must be 16-byte aligned");
  FDM_CHECK_CUDA(fdm_launch_pdl(ddim_step_kernel, dim3(grid_for(a.n / 4)), dim3(256), 0, reinterpret_cast<cudaStream_t>(stream), 1, a,
                                a.n / 4));
  return 0;
}

extern "C" int fdm_known_frames(const fdm_known_args* args, void* stream) {
  FDM_CHECK_ARG(args != nullptr, "fdm_known_frames: null args");
  const fdm_known_args& a = *args;
  FDM_CHECK_ARG(a.x && a.known && a.mask && a.ka && a.kb && a.index_dev, "fdm_known_frames: null operand");
  FDM_CHECK_ARG(a.noise || (a.seed_dev && a.t_dev), "fdm_known_frames: need noise or seed_dev and t_dev");
  FDM_CHECK_ARG(a.B > 0 && a.T > 0 && a.d > 0 && a.d % 4 == 0, "fdm_known_frames: need B, T > 0 and d a positive multiple of 4");
  FDM_CHECK_ARG(a.B * a.T <= 0x7fffffff, "fdm_known_frames: at most 2^31 - 1 rows per call");
  const uintptr_t al = reinterpret_cast<uintptr_t>(a.x) | reinterpret_cast<uintptr_t>(a.known) | reinterpret_cast<uintptr_t>(a.noise);
  FDM_CHECK_ARG(al % 16 == 0 && reinterpret_cast<uintptr_t>(a.x_bf16) % 8 == 0, "fdm_known_frames: operands must be 16-byte aligned");
  FDM_CHECK_CUDA(fdm_launch_pdl(known_frames_kernel, dim3(static_cast<unsigned>(a.B * a.T)), dim3(128), 0,
                                reinterpret_cast<cudaStream_t>(stream), 1, a, a.d / 4));
  return 0;
}

extern "C" int fdm_advance_cursor(int32_t* cursor_dev, const int32_t* t_sched, int32_t n_sched, int32_t* t_dev, void* stream) {
  FDM_CHECK_ARG(cursor_dev && t_sched && t_dev && n_sched > 0, "fdm_advance_cursor: bad arguments");
  FDM_CHECK_CUDA(fdm_launch_pdl(advance_cursor_kernel, dim3(1), dim3(1), 0, reinterpret_cast<cudaStream_t>(stream), 1, cursor_dev, t_sched,
                                static_cast<int>(n_sched), t_dev));
  return 0;
}

extern "C" int fdm_philox_normal(float* out, int64_t B, int64_t elems_per_clip, uint64_t seed, int64_t clip_index0, int32_t t,
                                 void* stream) {
  FDM_CHECK_ARG(out && B > 0 && elems_per_clip > 0 && elems_per_clip % 4 == 0 && reinterpret_cast<uintptr_t>(out) % 16 == 0,
                "fdm_philox_normal: bad arguments");
  const int64_t n4 = B * elems_per_clip / 4;
  philox_fill_kernel<<<grid_for(n4), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(out, n4, elems_per_clip / 4, seed, clip_index0, t);
  FDM_CHECK_LAUNCH();
  return 0;
}
