// Shared helpers for libfdm_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>
#include "../../include/fdm_b200.h"

void fdm_set_error(const char* fmt, ...);

#define FDM_CHECK_ARG(cond, ...)            \
  do {                                      \
    if (!(cond)) {                          \
      fdm_set_error(__VA_ARGS__);           \
      return 1;                             \
    }                                       \
  } while (0)

#define FDM_CHECK_CUDA(expr)                                                            \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess) {                                                            \
      fdm_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return 2;                                                                         \
    }                                                                                   \
  } while (0)

#define FDM_CHECK_LAUNCH() FDM_CHECK_CUDA(cudaGetLastError())

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

const void* fdm_gemm_identity();  // 64 x 64 bf16 identity of the current device (gemm_tc.cu), or nullptr before fdm_gemm_init_device()
int fdm_gemm_init_device();
int fdm_sm_count();  // cached multiprocessor count of the current device
bool fdm_pdl_enabled();  // programmatic dependent launch for the hot-loop kernels (on by default; env FDM_B200_PDL=0 turns it off)

// One tile of a VQ kernel with per-row codebook slices (fdm_vq_quantize_runs): rows [l0, l0 + nrows) of clip b, codebook
// slice offset `off`. vq.cu cuts the run table into these per call (no tile crosses a run); the kernels read one per tile.
struct alignas(16) VqTile { int b, l0, nrows, off; };

// ---- programmatic dependent launch (PDL) -------------------------------------------------------
// Hot-loop kernels are launched with programmaticStreamSerialization: kernel N+1 may be scheduled while kernel N
// drains, runs its prologue (barrier init, TMEM alloc, descriptor prefetch, index math) and then blocks in
// pdl_wait() until kernel N has completed and its memory is visible. Every kernel launched this way calls
// pdl_wait() before its first dependent global access; pdl_trigger() lets the next kernel's launch proceed.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t fdm_launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, int cluster_x,
                                  Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int n = 0;
  if (fdm_pdl_enabled()) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  if (cluster_x > 1) {  // thread-block cluster (CTA pair for tcgen05 cta_group::2)
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = cluster_x;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- dtype-generic loads / stores (fp32 math everywhere) --------------------------------------
__device__ __forceinline__ float ld_as_float(const void* p, int32_t dtype, int64_t i) {
  return dtype == FDM_BF16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[i])
                           : reinterpret_cast<const float*>(p)[i];
}
__device__ __forceinline__ void st_from_float(void* p, int32_t dtype, int64_t i, float v) {
  if (dtype == FDM_BF16) reinterpret_cast<__nv_bfloat16*>(p)[i] = __float2bfloat16_rn(v);
  else reinterpret_cast<float*>(p)[i] = v;
}

// ---- activations (match the PyTorch definitions used by the reference) -------------------------
__device__ __forceinline__ float act_mish(float x) {
  // x * tanh(softplus(x)) with tanh(log(1+e^x)) = n / (n + 2), n = e^x (e^x + 2); softplus threshold 20 as in ATen
  if (x > 20.f) return x;
  const float e = expf(x);
  const float n = e * (e + 2.f);
  return x * (n / (n + 2.f));
}
__device__ __forceinline__ float act_gelu_erf(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752440f)); }
// erf-GELU for outputs that are rounded to bf16 (bf16 GEMM epilogues, the bf16 path of the HuBERT conv0 kernel; fp32 outputs keep erff):
// no MUFU at all. erf(x / sqrt 2) = w P(w^2) with w = clamp(x / (2 R sqrt 2), -1/2, 1/2), R = 2.85, P of degree 7 fitted on
// Chebyshev nodes with P(1/4) / 2 = 1 pinned, so beyond |x| = 4.03 the result is exactly x or 0. |GELU error| < 1.3e-4
// (at |x| ~ 4, where a bf16 ulp is 1.6e-2); 13 FMA-pipe instructions per element against ~22 + 2 MUFU.
__device__ __forceinline__ float act_gelu_erf_poly(float x) {
  const float w = __saturatef(fmaf(x, 0.12405407f, 0.5f)) - 0.5f;  // 1 / (2 * 2.85 * sqrt 2)
  const float s = w * w;
  float p = fmaf(-108514.76f, s, 133392.03f);
  p = fmaf(p, s, -71527.083f);
  p = fmaf(p, s, 22276.801f);
  p = fmaf(p, s, -4549.4910f);
  p = fmaf(p, s, 653.65449f);
  p = fmaf(p, s, -69.234234f);
  p = fmaf(p, s, 6.4296663f);
  return x * fmaf(0.5f, w * p, 0.5f);
}
__device__ __forceinline__ float act_gelu_tanh(float x) {
  // models/utils/base_model_util.py:81-94
  float inner = 0.7978845608028654f * (x + 0.044715f * x * x * x);
  return x * (0.5f * (1.f + tanhf(inner)));
}
__device__ __forceinline__ float apply_act(float x, int act) {
  switch (act) {
    case FDM_ACT_RELU: return x > 0.f ? x : 0.f;
    case FDM_ACT_MISH: return act_mish(x);
    case FDM_ACT_GELU_ERF: return act_gelu_erf(x);
    case FDM_ACT_GELU_TANH: return act_gelu_tanh(x);
    case FDM_ACT_LEAKY02: return x > 0.f ? x : 0.2f * x;
    default: return x;
  }
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
