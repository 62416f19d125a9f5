// Small data-movement kernels around the GEMMs: casts, the (B,C,L)->(B,L,C) transpose of VQAutoEncoder.decode,
// per-clip time padding for the implicit convolutions, and HuBERT's first conv layer (1 input channel).
#include "common.cuh"
#include <stdlib.h>

namespace {

__global__ void __launch_bounds__(256) cast_kernel(const void* src, int sd, void* dst, int dd, int64_t n) {
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x)
    st_from_float(dst, dd, i, ld_as_float(src, sd, i));
}

// x = hi + lo + r, |r| <= 2^-17 |x|: operand pair of the split-bf16 GEMM. 4 elements per thread (16-byte load, two 8-byte stores).
__global__ void __launch_bounds__(256) split_bf16x2_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ hi,
                                                           __nv_bfloat16* __restrict__ lo, int64_t n) {
  const int64_t n4 = n >> 2;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(src)[i];
    const __nv_bfloat162 h0 = __floats2bfloat162_rn(v.x, v.y), h1 = __floats2bfloat162_rn(v.z, v.w);
    const float2 f0 = __bfloat1622float2(h0), f1 = __bfloat1622float2(h1);
    const __nv_bfloat162 l0 = __floats2bfloat162_rn(v.x - f0.x, v.y - f0.y), l1 = __floats2bfloat162_rn(v.z - f1.x, v.w - f1.y);
    uint2 uh, ul;
    uh.x = *reinterpret_cast<const uint32_t*>(&h0); uh.y = *reinterpret_cast<const uint32_t*>(&h1);
    ul.x = *reinterpret_cast<const uint32_t*>(&l0); ul.y = *reinterpret_cast<const uint32_t*>(&l1);
    reinterpret_cast<uint2*>(hi)[i] = uh;
    reinterpret_cast<uint2*>(lo)[i] = ul;
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {  // tail
    const int64_t i = (n4 << 2) + threadIdx.x;
    const __nv_bfloat16 h = __float2bfloat16_rn(src[i]);
    hi[i] = h;
    lo[i] = __float2bfloat16_rn(src[i] - __bfloat162float(h));
  }
}

__global__ void __launch_bounds__(256) transpose_kernel(const float* src, void* dst, int dd, int C, int L) {
  __shared__ float tile[32][33];
  const int64_t b = blockIdx.z;
  const int c0 = blockIdx.y * 32, l0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int i = ty; i < 32; i += 8) {
    const int c = c0 + i, l = l0 + tx;
    tile[i][tx] = (c < C && l < L) ? src[(b * C + c) * L + l] : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int l = l0 + i, c = c0 + tx;
    if (l < L && c < C) st_from_float(dst, dd, (b * L + l) * C + c, tile[tx][i]);
  }
}

__global__ void __launch_bounds__(256) pad_time_kernel(const void* src, int64_t src_t_stride, void* dst, int dtype, int T, int C,
                                                       int pad_l, int pad_r, int mode) {
  const int64_t b = blockIdx.y;
  const int P = pad_l + T + pad_r;
  const int64_t n = static_cast<int64_t>(P) * C;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int p = static_cast<int>(i / C), c = static_cast<int>(i - static_cast<int64_t>(p) * C);
    int t = p - pad_l;
    float v = 0.f;
    if (mode == 1) t = t < 0 ? 0 : (t >= T ? T - 1 : t);
    if (t >= 0 && t < T) v = ld_as_float(src, dtype, (b * src_t_stride + t) * C + c);
    st_from_float(dst, dtype, b * n + i, v);
  }
}

// same, 16 bytes per thread and iteration (row bytes a multiple of 16, aligned pointers): the scalar kernel's per-element 64-bit
// division made the replicate padding of the EVQ-VAE expander (64 clips x 498 frames x 1024) a 196 us copy of 65 MB
__global__ void __launch_bounds__(256) pad_time_vec_kernel(const uint4* __restrict__ src, int64_t src_t_stride, uint4* __restrict__ dst,
                                                           int T, int C16, int pad_l, int pad_r, int mode) {
  const int64_t b = blockIdx.y;
  const int P = pad_l + T + pad_r;
  const int n = P * C16;  // 16-byte chunks per clip (< 2^31: checked by the caller)
  const uint4* sb = src + b * src_t_stride * C16;
  uint4* db = dst + b * static_cast<int64_t>(n);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int p = i / C16, c = i - p * C16;
    int t = p - pad_l;
    if (mode == 1) t = t < 0 ? 0 : (t >= T ? T - 1 : t);
    db[i] = (t >= 0 && t < T) ? sb[static_cast<int64_t>(t) * C16 + c] : make_uint4(0u, 0u, 0u, 0u);
  }
}

// one warp per output frame; C <= 1024 channels, C % 32 == 0
template <int CPL>  // channels per lane
__global__ void __launch_bounds__(256) hubert_conv0_kernel(const float* __restrict__ audio, int64_t L, const float* __restrict__ w,
                                                           const float* __restrict__ bias, const float* __restrict__ g,
                                                           const float* __restrict__ beta, void* out, int od, int Lout,
                                                           int64_t out_t_stride) {
  constexpr int C = CPL * 32;
  __shared__ float ws[C * 10];
  for (int i = threadIdx.x; i < C * 10; i += blockDim.x) ws[i] = w[i];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t b = blockIdx.y;
  const int64_t t = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= out_t_stride) return;
  const int64_t orow = (b * out_t_stride + t) * C;
  if (t >= Lout) {
#pragma unroll
    for (int j = 0; j < CPL; ++j) st_from_float(out, od, orow + lane + 32 * j, 0.f);
    return;
  }
  float x[10];
#pragma unroll
  for (int k = 0; k < 10; ++k) x[k] = audio[b * L + t * 5 + k];
  float v[CPL];
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < CPL; ++j) {
    const int c = lane + 32 * j;
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < 10; ++k) acc = fmaf(ws[c * 10 + k], x[k], acc);
    v[j] = acc + (bias ? bias[c] : 0.f);
    s += v[j];
  }
  if (g == nullptr) {  // raw conv output: normalised over time by a later kernel (wav2vec2 "group" variant)
#pragma unroll
    for (int j = 0; j < CPL; ++j) st_from_float(out, od, orow + lane + 32 * j, v[j]);
    return;
  }
  const float mean = warp_sum(s) / C;
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < CPL; ++j) q += (v[j] - mean) * (v[j] - mean);
  const float rstd = 1.f / sqrtf(warp_sum(q) / C + 1e-5f);
#pragma unroll
  for (int j = 0; j < CPL; ++j) {
    const int c = lane + 32 * j;
    st_from_float(out, od, orow + c, act_gelu_erf((v[j] - mean) * rstd * g[c] + beta[c]));
  }
}

// C = 512 (hubert-large / wav2vec2-base first layer). The kernel above reads every weight from shared memory once per
// frame (160 two-way-conflicting LDS.32 against 160 FMAs per lane: 1.08 ms for 64 clips x 4 s, 14 % of the FFMA rate).
// Here a warp computes FOUR consecutive frames per pass from k-major float4 weights (one conflict-free LDS.128 feeds 16
// FMAs), a lane owns channels 128 j + 4 lane .. + 3 (8- / 16-byte output stores, 256 / 512 contiguous bytes per warp), the
// four frames' LayerNorm reductions are interleaved, and bf16 outputs take the polynomial erf-GELU.
constexpr int C0_FRAMES = 4;       // frames per warp pass
constexpr int C0_PASSES = 4;       // passes per warp: a CTA of 8 warps covers 128 frames per weight load
__global__ void __launch_bounds__(256) hubert_conv0_c512_kernel(const float* __restrict__ audio, int64_t L, const float* __restrict__ w,
                                                                const float* __restrict__ bias, const float* __restrict__ g,
                                                                const float* __restrict__ beta, void* out, int od, int Lout,
                                                                int64_t out_t_stride) {
  constexpr int C = 512;
  __shared__ float4 ws4[10 * 4 * 32];  // [k][j][lane] = w[128 j + 4 lane + 0..3][k]
  __shared__ float4 pb4[3 * 4 * 32];   // bias, gamma, beta in the same channel order
  for (int i = threadIdx.x; i < 10 * 4 * 32; i += blockDim.x) {
    const int k = i / 128, c = 4 * (i % 128);  // (j, lane) -> channel 128 j + 4 lane = 4 (i % 128)
    ws4[i] = make_float4(w[(c + 0) * 10 + k], w[(c + 1) * 10 + k], w[(c + 2) * 10 + k], w[(c + 3) * 10 + k]);
  }
  for (int i = threadIdx.x; i < 3 * 128; i += blockDim.x) {
    const int which = i / 128, c = 4 * (i % 128);
    const float* src = which == 0 ? bias : (which == 1 ? g : beta);
    pb4[i] = src ? make_float4(src[c], src[c + 1], src[c + 2], src[c + 3]) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t b = blockIdx.y;
  const float* a = audio + b * L;
  const bool bf = od == FDM_BF16;
#pragma unroll 1
  for (int pass = 0; pass < C0_PASSES; ++pass) {
    const int64_t t0 = (static_cast<int64_t>(blockIdx.x) * C0_PASSES + pass) * (8 * C0_FRAMES) + warp * C0_FRAMES;
    if (t0 >= out_t_stride) return;
    float x[5 * (C0_FRAMES - 1) + 10];
#pragma unroll
    for (int i = 0; i < 5 * (C0_FRAMES - 1) + 10; ++i) {
      const int64_t si = t0 * 5 + i;
      x[i] = __ldg(a + (si < L ? si : L - 1));  // (frames >= Lout are masked below)
    }
    float acc[C0_FRAMES][16];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 b4 = pb4[j * 32 + lane];
#pragma unroll
      for (int f = 0; f < C0_FRAMES; ++f) { acc[f][4 * j] = b4.x; acc[f][4 * j + 1] = b4.y; acc[f][4 * j + 2] = b4.z; acc[f][4 * j + 3] = b4.w; }
    }
#pragma unroll
    for (int k = 0; k < 10; ++k) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 w4 = ws4[(k * 4 + j) * 32 + lane];
#pragma unroll
        for (int f = 0; f < C0_FRAMES; ++f) {
          const float xv = x[5 * f + k];
          acc[f][4 * j] = fmaf(w4.x, xv, acc[f][4 * j]);
          acc[f][4 * j + 1] = fmaf(w4.y, xv, acc[f][4 * j + 1]);
          acc[f][4 * j + 2] = fmaf(w4.z, xv, acc[f][4 * j + 2]);
          acc[f][4 * j + 3] = fmaf(w4.w, xv, acc[f][4 * j + 3]);
        }
      }
    }
    float mean[C0_FRAMES], rstd[C0_FRAMES];
    if (g != nullptr) {  // LayerNorm over the 512 channels of each frame: the four frames' butterflies interleaved
      float s[C0_FRAMES], q[C0_FRAMES];
#pragma unroll
      for (int f = 0; f < C0_FRAMES; ++f) {
        s[f] = 0.f;
#pragma unroll
        for (int i = 0; i < 16; ++i) s[f] += acc[f][i];
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int f = 0; f < C0_FRAMES; ++f) s[f] += __shfl_xor_sync(0xffffffffu, s[f], o);
      }
#pragma unroll
      for (int f = 0; f < C0_FRAMES; ++f) {
        mean[f] = s[f] * (1.f / C);
        q[f] = 0.f;
#pragma unroll
        for (int i = 0; i < 16; ++i) q[f] = fmaf(acc[f][i] - mean[f], acc[f][i] - mean[f], q[f]);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int f = 0; f < C0_FRAMES; ++f) q[f] += __shfl_xor_sync(0xffffffffu, q[f], o);
      }
#pragma unroll
      for (int f = 0; f < C0_FRAMES; ++f) rstd[f] = 1.f / sqrtf(q[f] * (1.f / C) + 1e-5f);
    }
#pragma unroll
    for (int f = 0; f < C0_FRAMES; ++f) {
      const int64_t t = t0 + f;
      if (t >= out_t_stride) break;
      const bool live = t < Lout;  // padding frames of the per-clip stride stay zero
      const int64_t orow = (b * out_t_stride + t) * C;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float o[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) o[i] = acc[f][4 * j + i];
        if (g != nullptr) {
          const float4 g4 = pb4[(4 + j) * 32 + lane], e4 = pb4[(8 + j) * 32 + lane];
          const float gg[4] = {g4.x, g4.y, g4.z, g4.w}, ee[4] = {e4.x, e4.y, e4.z, e4.w};
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float y = fmaf((o[i] - mean[f]) * rstd[f], gg[i], ee[i]);
            o[i] = bf ? act_gelu_erf_poly(y) : act_gelu_erf(y);
          }
        }
        if (!live) { o[0] = o[1] = o[2] = o[3] = 0.f; }
        const int64_t oi = orow + 128 * j + 4 * lane;
        if (bf) {
          const __nv_bfloat162 p0 = __floats2bfloat162_rn(o[0], o[1]), p1 = __floats2bfloat162_rn(o[2], o[3]);
          uint2 v;
          v.x = *reinterpret_cast<const uint32_t*>(&p0);
          v.y = *reinterpret_cast<const uint32_t*>(&p1);
          *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(out) + oi) = v;
        } else {
          *reinterpret_cast<float4*>(reinterpret_cast<float*>(out) + oi) = make_float4(o[0], o[1], o[2], o[3]);
        }
      }
    }
  }
}

// dst[r, 0:ld_dst] = cast(src[r, 0:cols]) followed by zeros: pads K to a 16-byte row pitch for the TMA-fed GEMMs
__global__ void __launch_bounds__(256) cast_rows_kernel(const float* __restrict__ src, int64_t ld_src, void* dst, int dd,
                                                        int64_t ld_dst, int64_t rows, int64_t cols) {
  const int64_t n = rows * ld_dst;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t r = i / ld_dst, c = i - r * ld_dst;
    st_from_float(dst, dd, i, c < cols ? src[r * ld_src + c] : 0.f);
  }
}

__device__ __forceinline__ float block_sum_1024(float v, float* red) {
  v = warp_sum(v);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float t = lane < (blockDim.x >> 5) ? red[lane] : 0.f;
  t = warp_sum(t);
  return t;  // every thread holds the total
}

// One CTA per clip: zero-mean / unit-variance normalisation of Wav2Vec2Processor (do_normalize=True:
// (x - mean) / sqrt(var + 1e-7), population variance) followed by `Lout - L` zero samples (the demos append 1 s).
__global__ void __launch_bounds__(1024) audio_normalize_pad_kernel(const float* __restrict__ in, int64_t L, float* __restrict__ out,
                                                                   int64_t Lout, float eps) {
  __shared__ float red[32];
  const float* x = in + static_cast<int64_t>(blockIdx.x) * L;
  float* y = out + static_cast<int64_t>(blockIdx.x) * Lout;
  float s = 0.f;
  for (int64_t i = threadIdx.x; i < L; i += blockDim.x) s += x[i];
  const float mean = block_sum_1024(s, red) / static_cast<float>(L);
  float q = 0.f;
  for (int64_t i = threadIdx.x; i < L; i += blockDim.x) { const float d = x[i] - mean; q = fmaf(d, d, q); }
  const float var = block_sum_1024(q, red) / static_cast<float>(L);
  const float rstd = 1.f / sqrtf(var + eps);
  for (int64_t i = threadIdx.x; i < Lout; i += blockDim.x) y[i] = i < L ? (x[i] - mean) * rstd : 0.f;
}

// Polyphase FIR resampler (scipy.signal.resample_poly / upfirdn semantics): out[m] = sum_k taps[k] * xup[(m + pre) * down - k]
// with xup the input zero-stuffed by `up`. One thread per output sample; only the taps that meet a non-zero sample are visited
// (k = k0 + up * q), ~ n_taps / up multiply-adds per output. The demo path's librosa.load(sr=16000) resampling
// (demo/demo_3d_mead.py:83) on the GPU; the filter itself is designed on the host (fdm_b200/frontend.py).
__global__ void __launch_bounds__(256) resample_poly_kernel(const float* __restrict__ in, int64_t L_in, float* __restrict__ out,
                                                            int64_t L_out, const float* __restrict__ taps, int n_taps, int up, int down,
                                                            int64_t pre) {
  const int64_t m = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (m >= L_out) return;
  const float* x = in + static_cast<int64_t>(blockIdx.y) * L_in;
  const int64_t p = (m + pre) * down;
  const int k0 = static_cast<int>(p % up);
  int64_t i = p / up;  // input sample that meets taps[k0]
  float acc = 0.f;
  for (int k = k0; k < n_taps; k += up, --i) {
    if (i < 0) break;
    if (i < L_in) acc = fmaf(taps[k], x[i], acc);
  }
  out[static_cast<int64_t>(blockIdx.y) * L_out + m] = acc;
}

// By-products of VectorQuantizer.forward that the sampling scripts discard but the API returns (models/lib/quantizer.py:52-61):
// sum over all elements of (z_q - z)^2 (the commitment / codebook loss is (1 + beta) * mean) and the code histogram behind
// the perplexity. One pass over z and the indices (the winning code rows come from the L2-resident codebook) instead of
// torch's three passes over (rows, D) temporaries. One warp per row; per-block partial sums in a fixed order (the host adds
// the `gridDim.x` partials), integer atomics for the histogram: deterministic.
// Codebook offset of a row: per clip (code_offset), from the run table (runs.clip_run != NULL: the last run of the row's clip that
// starts at or before it, by bisection), or 0.
__device__ __forceinline__ int64_t row_slice(const int64_t* __restrict__ code_offset, const fdm_vq_runs& runs, int64_t row,
                                             int64_t L) {
  const int64_t b = row / L;
  if (runs.clip_run) {
    const int64_t l = row - b * L;
    int64_t lo = runs.clip_run[b], hi = runs.clip_run[b + 1] - 1;
    while (lo < hi) {
      const int64_t mid = (lo + hi + 1) >> 1;
      if (runs.run_l0[mid] <= l) lo = mid; else hi = mid - 1;
    }
    return runs.run_offset[lo];
  }
  return code_offset ? code_offset[b] : 0;
}

__global__ void __launch_bounds__(256) vq_stats_kernel(const float* __restrict__ z, const float* __restrict__ codebook,
                                                       const int64_t* __restrict__ code_offset, const int64_t* __restrict__ indices,
                                                       int64_t rows, int64_t L, int D, int n_codes, float* __restrict__ partials,
                                                       unsigned long long* __restrict__ hist, const fdm_vq_runs runs) {
  extern __shared__ unsigned int sh_hist[];  // n_codes counters, then 8 floats
  float* red = reinterpret_cast<float*>(sh_hist + n_codes);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < n_codes; i += blockDim.x) sh_hist[i] = 0u;
  __syncthreads();
  float acc = 0.f;
  // eight rows per warp and iteration: the index loads and the (index-independent) latent loads go out first, then the code
  // rows they select (L2-resident); D = 64: float2 per lane
  constexpr int RW = 8;
  for (int64_t row0 = (static_cast<int64_t>(blockIdx.x) * 8 + warp) * RW; row0 < rows; row0 += static_cast<int64_t>(gridDim.x) * 8 * RW) {
    if (D == 64) {
      int64_t idx[RW];
      float2 a[RW];
#pragma unroll
      for (int q = 0; q < RW; ++q) {
        const bool ok = row0 + q < rows;
        idx[q] = ok ? indices[row0 + q] : -1;
        a[q] = ok ? reinterpret_cast<const float2*>(z + (row0 + q) * 64)[lane] : make_float2(0.f, 0.f);
      }
#pragma unroll
      for (int q = 0; q < RW; ++q) {
        if (idx[q] < 0) continue;
        const int64_t off = row_slice(code_offset, runs, row0 + q, L);
        const float2 e = __ldg(reinterpret_cast<const float2*>(codebook + (off + idx[q]) * 64) + lane);
        const float d0 = e.x - a[q].x, d1 = e.y - a[q].y;
        acc = fmaf(d0, d0, acc);
        acc = fmaf(d1, d1, acc);
        if (lane == 0 && idx[q] < n_codes) atomicAdd(&sh_hist[idx[q]], 1u);
      }
    } else {
      for (int q = 0; q < RW && row0 + q < rows; ++q) {
        const int64_t row = row0 + q, id = indices[row];
        const int64_t off = row_slice(code_offset, runs, row, L);
        const float* zr = z + row * D;
        const float* er = codebook + (off + id) * D;
        for (int k = lane; k < D; k += 32) {
          const float d = __ldg(er + k) - zr[k];
          acc = fmaf(d, d, acc);
        }
        if (lane == 0 && id >= 0 && id < n_codes) atomicAdd(&sh_hist[id], 1u);
      }
    }
  }
  acc = warp_sum(acc);
  if (lane == 0) red[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < 8; ++w) s += red[w];
    partials[blockIdx.x] = s;
  }
  for (int i = threadIdx.x; i < n_codes; i += blockDim.x)
    if (sh_hist[i]) atomicAdd(hist + i, static_cast<unsigned long long>(sh_hist[i]));
}

// One CTA per frame: reduce over a vertex subset the squared L2 distance between prediction and ground truth
// (metric/metric.py:115-138: per-frame max for LVE / FVE / all-vertex error, per-frame mean for EME).
__global__ void __launch_bounds__(256) vertex_error_kernel(const float* __restrict__ pred, const float* __restrict__ gt, int64_t V,
                                                           const int64_t* __restrict__ idx, int64_t n, int mode,
                                                           float* __restrict__ out) {
  __shared__ float red[8];
  const int64_t f = blockIdx.x;
  const float* p = pred + f * V * 3;
  const float* g = gt ? gt + f * V * 3 : nullptr;
  const int64_t cnt = idx ? n : V;
  float acc = mode == 0 ? 0.f : 0.f;  // distances are >= 0: 0 is the identity of both reductions
  for (int64_t i = threadIdx.x; i < cnt; i += blockDim.x) {
    const int64_t v = idx ? idx[i] : i;
    float d2 = 0.f;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float d = (g ? g[v * 3 + k] : 0.f) - p[v * 3 + k];
      d2 += d * d;  // same order as np.sum(np.square(.), axis=2)
    }
    acc = mode == 0 ? fmaxf(acc, d2) : acc + d2;
  }
  acc = mode == 0 ? warp_max(acc) : warp_sum(acc);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) red[warp] = acc;
  __syncthreads();
  if (warp == 0) {
    float t = lane < 8 ? red[lane] : 0.f;
    t = mode == 0 ? warp_max(t) : warp_sum(t);
    if (lane == 0) out[f] = mode == 0 ? t : t / static_cast<float>(cnt);
  }
}

inline int grid1d(int64_t n) {
  const int64_t want = ceil_div64(n, 256), cap = static_cast<int64_t>(fdm_sm_count()) * 8;
  return static_cast<int>(want < cap ? (want > 0 ? want : 1) : cap);
}

}  // namespace

extern "C" int fdm_cast(const void* src, int32_t src_dtype, void* dst, int32_t dst_dtype, int64_t n, void* stream) {
  FDM_CHECK_ARG(src && dst && n >= 0, "fdm_cast: bad arguments");
  if (n == 0) return 0;
  cast_kernel<<<grid1d(n), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(src, src_dtype, dst, dst_dtype, n);
  FDM_CHECK_LAUNCH();
  return 0;
}

extern "C" int fdm_split_bf16x2(const float* src, void* hi, void* lo, int64_t n, void* stream) {
  FDM_CHECK_ARG(src && hi && lo && n >= 0, "fdm_split_bf16x2: bad arguments");
  FDM_CHECK_ARG(reinterpret_cast<uintptr_t>(src) % 16 == 0 && reinterpret_cast<uintptr_t>(hi) % 8 == 0 &&
                    reinterpret_cast<uintptr_t>(lo) % 8 == 0,
                "fdm_split_bf16x2: src must be 16-byte, hi / lo 8-byte aligned");
  if (n == 0) return 0;
  split_bf16x2_kernel<<<grid1d((n + 3) / 4), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      src, reinterpret_cast<__nv_bfloat16*>(hi), reinterpret_cast<__nv_bfloat16*>(lo), n);
  FDM_CHECK_LAUNCH();
  return 0;
}

extern "C" int fdm_transpose_bcl_to_blc(const float* src, void* dst, int32_t dst_dtype, int64_t B, int64_t C, int64_t L, void* stream) {
  FDM_CHECK_ARG(src && dst && B > 0 && C > 0 && L > 0 && B <= 65535 && C <= 65535 * 32, "fdm_transpose_bcl_to_blc: bad arguments");
  dim3 grid(static_cast<unsigned>(ceil_div64(L, 32)), static_cast<unsigned>(ceil_div64(C, 32)), static_cast<unsigned>(B));
  transpose_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(src, dst, dst_dtype, static_cast<int>(C), static_cast<int>(L));
  FDM_CHECK_LAUNCH();
  return 0;
}

extern "C" int fdm_pad_time(const void* src, int64_t src_t_stride, void* dst, int32_t dtype, int64_t B, int64_t T, int64_t C,
                            int64_t pad_l, int64_t pad_r, int32_t mode, void* stream) {
  FDM_CHECK_ARG(src && dst && B > 0 && T > 0 && C > 0 && pad_l >= 0 && pad_r >= 0 && B <= 65535 && src_t_stride >= T,
                "fdm_pad_time: bad arguments");
  const int64_t esz = dtype == FDM_BF16 ? 2 : 4;
  if ((C * esz) % 16 == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15u) == 0 &&
      (pad_l + T + pad_r) * (C * esz / 16) < (1ll << 31)) {
    const int64_t c16 = C * esz / 16, n = (pad_l + T + pad_r) * c16;
    dim3 gridv(static_cast<unsigned>(ceil_div64(n, 256 * 4) < 1 ? 1 : ceil_div64(n, 256 * 4)), static_cast<unsigned>(B));
    pad_time_vec_kernel<<<gridv, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const uint4*>(src), src_t_stride, reinterpret_cast<uint4*>(dst), static_cast<int>(T), static_cast<int>(c16),
        static_cast<int>(pad_l), static_cast<int>(pad_r), mode);
    FDM_CHECK_LAUNCH();
    return 0;
  }
  dim3 grid(static_cast<unsigned>(grid1d((pad_l + T + pad_r) * C)), static_cast<unsigned>(B));
  pad_time_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(src, src_t_stride, dst, dtype, static_cast<int>(T),
                                                                            static_cast<int>(C), static_cast<int>(pad_l),
                                                                            static_cast<int>(pad_r), mode);
  FDM_CHECK_LAUNCH();
  return 0;
}

extern "C" int fdm_hubert_conv0(const float* audio, int64_t B, int64_t L, const float* w, const float* bias, const float* ln_g,
                                const float* ln_b, void* out, int32_t out_dtype, int64_t Lout, int64_t out_t_stride, int64_t C,
                                void* stream) {
  FDM_CHECK_ARG(audio && w && out && ((ln_g == nullptr) == (ln_b == nullptr)), "fdm_hubert_conv0: null operand");
  FDM_CHECK_ARG(B > 0 && B <= 65535 && Lout > 0 && out_t_stride >= Lout && (Lout - 1) * 5 + 10 <= L, "fdm_hubert_conv0: bad sizes");
  dim3 grid(static_cast<unsigned>(ceil_div64(out_t_stride, 8)), static_cast<unsigned>(B));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  static const bool c512_fast = [] { const char* e = getenv("FDM_B200_CONV0_FAST"); return !(e && e[0] == '0'); }();
  const int64_t esz = out_dtype == FDM_BF16 ? 2 : 4;
  if (C == 512 && c512_fast && reinterpret_cast<uintptr_t>(out) % 16 == 0 && (out_t_stride * C * esz) % 16 == 0) {
    dim3 grid4(static_cast<unsigned>(ceil_div64(out_t_stride, 8 * C0_FRAMES * C0_PASSES)), static_cast<unsigned>(B));
    hubert_conv0_c512_kernel<<<grid4, 256, 0, s>>>(audio, L, w, bias, ln_g, ln_b, out, out_dtype, static_cast<int>(Lout), out_t_stride);
  } else if (C == 512) hubert_conv0_kernel<16><<<grid, 256, 0, s>>>(audio, L, w, bias, ln_g, ln_b, out, out_dtype, static_cast<int>(Lout), out_t_stride);
  else if (C == 32) hubert_conv0_kernel<1><<<grid, 256, 0, s>>>(audio, L, w, bias, ln_g, ln_b, out, out_dtype, static_cast<int>(Lout), out_t_stride);
  else if (C == 64) hubert_conv0_kernel<2><<<grid, 256, 0, s>>>(audio, L, w, bias, ln_g, ln_b, out, out_dtype, static_cast<int>(Lout), out_t_stride);
  else FDM_CHECK_ARG(false, "fdm_hubert_conv0: C=%lld not in {32,64,512}", (long long)C);
  FDM_CHECK_LAUNCH();
  return 0;
}

extern "C" int fdm_cast_rows(const float* src, int64_t ld_src, void* dst, int32_t dst_dtype, int64_t ld_dst, int64_t rows,
                             int64_t cols, void* stream) {
  FDM_CHECK_ARG(src && dst && rows > 0 && cols > 0 && ld_src >= cols && ld_dst >= cols, "fdm_cast_rows: bad arguments");
  cast_rows_kernel<<<grid1d(rows * ld_dst), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(src, ld_src, dst, dst_dtype, ld_dst,
                                                                                                rows, cols);
  FDM_CHECK_LAUNCH();
  return 0;
}

extern "C" int fdm_audio_normalize_pad(const float* audio, int64_t B, int64_t L, float* out, int64_t Lout, float eps, void* stream) {
  FDM_CHECK_ARG(audio && out && B > 0 && L > 0 && Lout >= L, "fdm_audio_normalize_pad: bad arguments");
  audio_normalize_pad_kernel<<<static_cast<unsigned>(B), 1024, 0, reinterpret_cast<cudaStream_t>(stream)>>>(audio, L, out, Lout, eps);
  FDM_CHECK_LAUNCH();
  return 0;
}

extern "C" int fdm_resample_poly(const float* audio, int64_t B, int64_t L_in, float* out, int64_t L_out, const float* taps,
                                 int64_t n_taps, int64_t up, int64_t down, int64_t pre, void* stream) {
  FDM_CHECK_ARG(audio && out && taps && B > 0 && B <= 65535 && L_in > 0 && L_out > 0 && n_taps > 0 && n_taps < (1ll << 30) && up > 0 &&
                    down > 0 && up < (1 << 20) && down < (1 << 20) && pre >= 0,
                "fdm_resample_poly: bad arguments");
  dim3 grid(static_cast<unsigned>(ceil_div64(L_out, 256)), static_cast<unsigned>(B));
  resample_poly_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(audio, L_in, out, L_out, taps, static_cast<int>(n_taps),
                                                                                static_cast<int>(up), static_cast<int>(down), pre);
  FDM_CHECK_LAUNCH();
  return 0;
}

extern "C" int fdm_vq_stats(const float* z, const float* codebook, const int64_t* code_offset, const int64_t* indices, int64_t B,
                            int64_t L, int64_t D, int64_t n_codes, float* sqerr_partials, int64_t n_partials, int64_t* hist,
                            void* stream) {
  FDM_CHECK_ARG(z && codebook && indices && sqerr_partials && hist && B > 0 && L > 0 && D > 0 && D <= 1024 && n_codes > 0 &&
                    n_codes <= 8192 && n_partials > 0 && n_partials <= 65535,
                "fdm_vq_stats: bad arguments");
  const size_t smem = static_cast<size_t>(n_codes) * 4 + 32;
  vq_stats_kernel<<<static_cast<unsigned>(n_partials), 256, smem, reinterpret_cast<cudaStream_t>(stream)>>>(
      z, codebook, code_offset, indices, B * L, L, static_cast<int>(D), static_cast<int>(n_codes), sqerr_partials,
      reinterpret_cast<unsigned long long*>(hist), fdm_vq_runs{nullptr, nullptr, nullptr, 0});
  FDM_CHECK_LAUNCH();
  return 0;
}

extern "C" int fdm_vq_stats_runs(const float* z, const float* codebook, const fdm_vq_runs* runs, const int64_t* indices,
                                 int64_t B, int64_t L, int64_t D, int64_t n_codes, float* sqerr_partials, int64_t n_partials,
                                 int64_t* hist, void* stream) {
  FDM_CHECK_ARG(z && codebook && indices && sqerr_partials && hist && B > 0 && L > 0 && D > 0 && D <= 1024 && n_codes > 0 &&
                    n_codes <= 8192 && n_partials > 0 && n_partials <= 65535,
                "fdm_vq_stats_runs: bad arguments");
  FDM_CHECK_ARG(runs && runs->clip_run && runs->run_l0 && runs->run_offset && runs->n_runs >= B,
                "fdm_vq_stats_runs: the run table needs clip_run, run_l0, run_offset and at least one run per clip");
  const size_t smem = static_cast<size_t>(n_codes) * 4 + 32;
  vq_stats_kernel<<<static_cast<unsigned>(n_partials), 256, smem, reinterpret_cast<cudaStream_t>(stream)>>>(
      z, codebook, nullptr, indices, B * L, L, static_cast<int>(D), static_cast<int>(n_codes), sqerr_partials,
      reinterpret_cast<unsigned long long*>(hist), *runs);
  FDM_CHECK_LAUNCH();
  return 0;
}

extern "C" int fdm_vertex_error(const float* pred, const float* gt, int64_t frames, int64_t V, const int64_t* vertex_idx,
                                int64_t n_idx, int32_t mode, float* out_per_frame, void* stream) {
  FDM_CHECK_ARG(pred && out_per_frame && frames > 0 && V > 0 && (mode == 0 || mode == 1) && (!vertex_idx || n_idx > 0),
                "fdm_vertex_error: bad arguments");
  vertex_error_kernel<<<static_cast<unsigned>(frames), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(pred, gt, V, vertex_idx, n_idx,
                                                                                                        mode, out_per_frame);
  FDM_CHECK_LAUNCH();
  return 0;
}
