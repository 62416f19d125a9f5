// fdm_vq_quantize: EVQ-VAE nearest-code search with a DEFINED fp32 expression so that indices are bit-exact
// against the CPU oracle (oracle/vq_ref.c):
//     d_j = (zz + ee_j) - 2 * dot_j,   zz = sum_k z_k^2, ee_j = sum_k e_jk^2, dot_j = sum_k z_k e_jk,
// every sum a sequential fmaf chain over k = 0..D-1 starting at +0.0f; argmin with the lowest index on ties.
// Persistent CTAs keep the (per-clip) codebook slice resident in shared memory; each CTA tile is 64 latent
// rows x all codes, register-tiled 8 rows x 8 codes per thread, then a warp-shuffle (d, index) min-reduction.
// The gather of the winning code and the (B, L, D) -> (B, D, L) permute of the reference are fused into the
// store phase.
#include "common.cuh"

namespace {

constexpr int ROWS = 64;      // latent rows per tile
constexpr int THREADS = 256;  // 8 warps; warp w owns rows 8w..8w+7, lane owns codes lane + 32*j
constexpr int MAXJ = 8;       // up to 256 codes

// TL (per-row slices, fdm_vq_quantize_runs): tile t is tiles[t], *tile_count of them, instead of 64-row tiles of whole clips
template <int D, bool TL>
__global__ void __launch_bounds__(THREADS) vq_kernel(const float* __restrict__ z, const float* __restrict__ codebook,
                                                     const int64_t* __restrict__ code_offset, int64_t B, int64_t L, int n_codes,
                                                     int64_t* __restrict__ indices, float* __restrict__ zq_bdl,
                                                     float* __restrict__ zq_rows, const VqTile* __restrict__ tiles,
                                                     const int* __restrict__ tile_count) {
  constexpr int DP = D + 4;  // padded row: conflict-free float4 reads across lanes
  extern __shared__ float sm[];
  float* cb = sm;                   // [n_codes][DP]
  float* zt = cb + 256 * DP;        // [ROWS][DP]
  float* ee = zt + ROWS * DP;       // [256]
  float* zz = ee + 256;             // [ROWS]
  int* widx = reinterpret_cast<int*>(zz + ROWS);  // [ROWS]

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ncj = n_codes / 32;
  const int64_t tiles_per_clip = (L + ROWS - 1) / ROWS;
  const int64_t num_tiles = TL ? *tile_count : B * tiles_per_clip;
  int64_t loaded_off = -1;

  for (int64_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
    int64_t b, l0, off;
    int nrows;
    if constexpr (TL) {
      const VqTile t = tiles[tile];
      b = t.b, l0 = t.l0, nrows = t.nrows, off = t.off;
    } else {
      b = tile / tiles_per_clip;
      l0 = (tile - b * tiles_per_clip) * ROWS;
      nrows = static_cast<int>(min(static_cast<int64_t>(ROWS), L - l0));
      off = code_offset ? code_offset[b] : 0;
    }
    __syncthreads();  // previous tile's store phase is done with cb / widx
    if (off != loaded_off) {
      for (int i = tid; i < n_codes * (D / 4); i += THREADS) {
        const int c = i / (D / 4), k4 = i - c * (D / 4);
        *reinterpret_cast<float4*>(cb + c * DP + k4 * 4) =
            *reinterpret_cast<const float4*>(codebook + (off + c) * D + k4 * 4);
      }
      loaded_off = off;
      __syncthreads();
      for (int c = tid; c < n_codes; c += THREADS) {
        float s = 0.f;
        for (int k = 0; k < D; ++k) s = fmaf(cb[c * DP + k], cb[c * DP + k], s);
        ee[c] = s;
      }
    }
    const float* zsrc = z + (b * L + l0) * D;
    for (int i = tid; i < ROWS * (D / 4); i += THREADS) {
      const int r = i / (D / 4), k4 = i - r * (D / 4);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < nrows) v = *reinterpret_cast<const float4*>(zsrc + static_cast<int64_t>(r) * D + k4 * 4);
      *reinterpret_cast<float4*>(zt + r * DP + k4 * 4) = v;
    }
    __syncthreads();
    if (tid < ROWS) {
      float s = 0.f;
      for (int k = 0; k < D; ++k) s = fmaf(zt[tid * DP + k], zt[tid * DP + k], s);
      zz[tid] = s;
    }

    float dot[8][MAXJ];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < MAXJ; ++j) dot[i][j] = 0.f;
#pragma unroll 2
    for (int k4 = 0; k4 < D / 4; ++k4) {
      float4 zv[8], ev[MAXJ];
#pragma unroll
      for (int i = 0; i < 8; ++i) zv[i] = *reinterpret_cast<const float4*>(zt + (warp * 8 + i) * DP + k4 * 4);
#pragma unroll
      for (int j = 0; j < MAXJ; ++j)
        ev[j] = j < ncj ? *reinterpret_cast<const float4*>(cb + (lane + 32 * j) * DP + k4 * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < MAXJ; ++j) {
          float a = dot[i][j];
          a = fmaf(zv[i].x, ev[j].x, a);
          a = fmaf(zv[i].y, ev[j].y, a);
          a = fmaf(zv[i].z, ev[j].z, a);
          a = fmaf(zv[i].w, ev[j].w, a);
          dot[i][j] = a;
        }
    }
    __syncthreads();  // zz ready (and every warp done reading zt)
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = warp * 8 + i;
      const float zzr = zz[r];
      float best = INFINITY;
      int bidx = 0x7fffffff;
#pragma unroll
      for (int j = 0; j < MAXJ; ++j)
        if (j < ncj) {
          const int c = lane + 32 * j;
          const float dist = __fsub_rn(__fadd_rn(zzr, ee[c]), __fmul_rn(2.f, dot[i][j]));
          if (dist < best || (dist == best && c < bidx)) { best = dist; bidx = c; }
        }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float od = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bidx, o);
        if (od < best || (od == best && oi < bidx)) { best = od; bidx = oi; }
      }
      // NaN / Inf row: no distance compares below +inf (the oracle's strict '<' from +inf keeps index 0; vq_tc.cu agrees)
      if (bidx == 0x7fffffff || !(best < INFINITY)) bidx = 0;
      if (lane == 0) {
        widx[r] = bidx;
        if (r < nrows && indices) indices[b * L + l0 + r] = bidx;
      }
    }
    __syncthreads();
    if (zq_bdl) {  // [b, k, l0 + r]: r fastest -> coalesced 256-byte runs
      for (int i = tid; i < D * ROWS; i += THREADS) {
        const int k = i / ROWS, r = i - k * ROWS;
        if (r < nrows) zq_bdl[(b * D + k) * L + l0 + r] = cb[widx[r] * DP + k];
      }
    }
    if (zq_rows) {
      for (int i = tid; i < ROWS * D; i += THREADS) {
        const int r = i / D, k = i - r * D;
        if (r < nrows) zq_rows[(b * L + l0 + r) * D + k] = cb[widx[r] * DP + k];
      }
    }
  }
}

template <int D>
int launch_vq(const float* z, const float* codebook, const int64_t* code_offset, int64_t B, int64_t L, int n_codes,
              int64_t* indices, float* zq_bdl, float* zq_rows, const VqTile* tiles, const int* tile_count, int64_t max_tiles,
              cudaStream_t stream) {
  constexpr int DP = D + 4;
  const size_t smem = sizeof(float) * (256 * DP + ROWS * DP + 256 + ROWS) + sizeof(int) * ROWS;
  static bool attr = false;
  if (!attr) {
    FDM_CHECK_CUDA(cudaFuncSetAttribute(vq_kernel<D, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    FDM_CHECK_CUDA(cudaFuncSetAttribute(vq_kernel<D, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    attr = true;
  }
  const int64_t tiles_n = tiles ? max_tiles : B * ceil_div64(L, ROWS);
  const int per_sm = smem * 2 <= 220 * 1024 ? 2 : 1;
  const int64_t cap = static_cast<int64_t>(fdm_sm_count()) * per_sm;
  const int grid = static_cast<int>(tiles_n < cap ? tiles_n : cap);
  if (tiles)
    vq_kernel<D, true><<<grid, THREADS, smem, stream>>>(z, codebook, code_offset, B, L, n_codes, indices, zq_bdl, zq_rows, tiles,
                                                      tile_count);
  else
    vq_kernel<D, false><<<grid, THREADS, smem, stream>>>(z, codebook, code_offset, B, L, n_codes, indices, zq_bdl, zq_rows,
                                                       nullptr, nullptr);
  FDM_CHECK_LAUNCH();
  return 0;
}

// The tile table of a run table (fdm_vq_runs), one CTA: thread t takes runs [n t / 1024, n (t + 1) / 1024), counts their
// tiles of `tile_rows` rows, a block scan gives each thread its first slot, and the threads write their tiles in run order.
// Header: the tile count (int) in the first 16 bytes, then the VqTile entries.
constexpr int BUILD_THREADS = 1024;
__global__ void __launch_bounds__(BUILD_THREADS) vq_build_tiles_kernel(fdm_vq_runs runs, int B, int L, int tile_rows,
                                                                       int* __restrict__ count, VqTile* __restrict__ tiles) {
  __shared__ int part[BUILD_THREADS];
  const int t = threadIdx.x;
  const int64_t n = runs.n_runs;
  const int64_t r0 = n * t / BUILD_THREADS, r1 = n * (t + 1) / BUILD_THREADS;
  int b = 0;
  if (r0 < r1) {  // the clip of run r0: the last b with clip_run[b] <= r0
    int lo = 0, hi = B - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (runs.clip_run[mid] <= r0) lo = mid; else hi = mid - 1;
    }
    b = lo;
  }
  const int b0 = b;
  int s = 0;
  for (int64_t r = r0; r < r1; ++r) {
    while (runs.clip_run[b + 1] <= r) ++b;
    const int64_t l1 = r + 1 < runs.clip_run[b + 1] ? runs.run_l0[r + 1] : L;
    s += static_cast<int>((l1 - runs.run_l0[r] + tile_rows - 1) / tile_rows);
  }
  part[t] = s;
  __syncthreads();
  for (int o = 1; o < BUILD_THREADS; o <<= 1) {  // inclusive scan
    const int v = t >= o ? part[t - o] : 0;
    __syncthreads();
    part[t] += v;
    __syncthreads();
  }
  if (t == BUILD_THREADS - 1) *count = part[t];
  int pos = part[t] - s;
  b = b0;
  for (int64_t r = r0; r < r1; ++r) {
    while (runs.clip_run[b + 1] <= r) ++b;
    const int64_t l1 = r + 1 < runs.clip_run[b + 1] ? runs.run_l0[r + 1] : L;
    const int off = static_cast<int>(runs.run_offset[r]);
    for (int64_t l = runs.run_l0[r]; l < l1; l += tile_rows)
      tiles[pos++] = VqTile{b, static_cast<int>(l), static_cast<int>(min(static_cast<int64_t>(tile_rows), l1 - l)), off};
  }
}

}  // namespace

// tensor-core filter + exact recheck (vq_tc.cu), D = 64 / 128
int fdm_vq_tc_launch(const float* z, const float* codebook, const int64_t* code_offset, int64_t B, int64_t L, int64_t D,
                     int n_codes, int64_t* indices, float* zq_bdl, float* zq_rows, unsigned long long* recheck_rows,
                     float* dbg_acc, const VqTile* tiles, const int* tile_count, int64_t max_tiles, cudaStream_t stream);

extern "C" int fdm_vq_quantize_ex(const float* z, const float* codebook, const int64_t* code_offset, int64_t B, int64_t L,
                                  int64_t D, int64_t n_codes, int64_t* indices, float* zq_bdl, float* zq_rows, int32_t algo,
                                  uint64_t* recheck_rows, float* dbg_acc, void* stream) {
  FDM_CHECK_ARG(z && codebook && B > 0 && L > 0, "fdm_vq_quantize: bad arguments");
  FDM_CHECK_ARG(n_codes > 0 && n_codes <= 256 && n_codes % 32 == 0, "fdm_vq_quantize: n_codes must be a multiple of 32, <= 256");
  FDM_CHECK_ARG(reinterpret_cast<uintptr_t>(z) % 16 == 0 && reinterpret_cast<uintptr_t>(codebook) % 16 == 0,
                "fdm_vq_quantize: z and codebook must be 16-byte aligned");
  FDM_CHECK_ARG(algo >= FDM_VQ_AUTO && algo <= FDM_VQ_TENSOR, "fdm_vq_quantize: unknown algo %d", algo);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (algo == FDM_VQ_AUTO) algo = (D == 64 || D == 128) ? FDM_VQ_TENSOR : FDM_VQ_FFMA;
  if (algo == FDM_VQ_TENSOR) {
    FDM_CHECK_ARG(D == 64 || D == 128, "fdm_vq_quantize: the tensor-core path needs D = 64 or 128 (got %lld)", (long long)D);
    return fdm_vq_tc_launch(z, codebook, code_offset, B, L, D, static_cast<int>(n_codes), indices, zq_bdl, zq_rows,
                            reinterpret_cast<unsigned long long*>(recheck_rows), dbg_acc, nullptr, nullptr, 0, s);
  }
  FDM_CHECK_ARG(!dbg_acc, "fdm_vq_quantize: dbg_acc is a tensor-core path output");
  switch (D) {
    case 32: return launch_vq<32>(z, codebook, code_offset, B, L, static_cast<int>(n_codes), indices, zq_bdl, zq_rows, nullptr, nullptr, 0, s);
    case 64: return launch_vq<64>(z, codebook, code_offset, B, L, static_cast<int>(n_codes), indices, zq_bdl, zq_rows, nullptr, nullptr, 0, s);
    case 128: return launch_vq<128>(z, codebook, code_offset, B, L, static_cast<int>(n_codes), indices, zq_bdl, zq_rows, nullptr, nullptr, 0, s);
    default: FDM_CHECK_ARG(false, "fdm_vq_quantize: D=%lld not in {32,64,128}", (long long)D);
  }
  return 0;
}

extern "C" int fdm_vq_quantize(const float* z, const float* codebook, const int64_t* code_offset, int64_t B, int64_t L,
                               int64_t D, int64_t n_codes, int64_t* indices, float* zq_bdl, float* zq_rows, void* stream) {
  return fdm_vq_quantize_ex(z, codebook, code_offset, B, L, D, n_codes, indices, zq_bdl, zq_rows, FDM_VQ_AUTO, nullptr, nullptr,
                            stream);
}

// Tiles of a run table at the smallest tile height (64 rows, the FFMA kernel): sum over runs of ceil(len / 64) is at most
// rows / 64 + n_runs.
static int64_t max_run_tiles(int64_t B, int64_t L, int64_t n_runs) { return ceil_div64(B * L, 64) + n_runs; }

extern "C" int64_t fdm_vq_runs_workspace_bytes(int64_t B, int64_t L, int64_t n_runs) {
  return 16 + static_cast<int64_t>(sizeof(VqTile)) * max_run_tiles(B, L, n_runs);
}

extern "C" int fdm_vq_quantize_runs(const float* z, const float* codebook, const fdm_vq_runs* runs, int64_t B, int64_t L,
                                    int64_t D, int64_t n_codes, int64_t* indices, float* zq_bdl, float* zq_rows, int32_t algo,
                                    uint64_t* recheck_rows, void* workspace, int64_t workspace_bytes, void* stream) {
  FDM_CHECK_ARG(z && codebook && B > 0 && L > 0, "fdm_vq_quantize_runs: bad arguments");
  FDM_CHECK_ARG(runs && runs->clip_run && runs->run_l0 && runs->run_offset && runs->n_runs >= B,
                "fdm_vq_quantize_runs: the run table needs clip_run, run_l0, run_offset and at least one run per clip");
  FDM_CHECK_ARG(B * L < (1ll << 31), "fdm_vq_quantize_runs: too many rows for one launch");
  FDM_CHECK_ARG(n_codes > 0 && n_codes <= 256 && n_codes % 32 == 0, "fdm_vq_quantize_runs: n_codes must be a multiple of 32, <= 256");
  FDM_CHECK_ARG(reinterpret_cast<uintptr_t>(z) % 16 == 0 && reinterpret_cast<uintptr_t>(codebook) % 16 == 0,
                "fdm_vq_quantize_runs: z and codebook must be 16-byte aligned");
  FDM_CHECK_ARG(workspace && reinterpret_cast<uintptr_t>(workspace) % 16 == 0 &&
                    workspace_bytes >= fdm_vq_runs_workspace_bytes(B, L, runs->n_runs),
                "fdm_vq_quantize_runs: the workspace must be 16-byte aligned and hold fdm_vq_runs_workspace_bytes");
  FDM_CHECK_ARG(algo >= FDM_VQ_AUTO && algo <= FDM_VQ_TENSOR, "fdm_vq_quantize_runs: unknown algo %d", algo);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (algo == FDM_VQ_AUTO) algo = (D == 64 || D == 128) ? FDM_VQ_TENSOR : FDM_VQ_FFMA;
  FDM_CHECK_ARG(algo == FDM_VQ_FFMA || D == 64 || D == 128,
                "fdm_vq_quantize_runs: the tensor-core path needs D = 64 or 128 (got %lld)", (long long)D);
  FDM_CHECK_ARG(D == 32 || D == 64 || D == 128, "fdm_vq_quantize_runs: D=%lld not in {32,64,128}", (long long)D);
  const int tile_rows = algo == FDM_VQ_TENSOR ? 128 : ROWS;
  int* count = reinterpret_cast<int*>(workspace);
  VqTile* tiles = reinterpret_cast<VqTile*>(static_cast<char*>(workspace) + 16);
  vq_build_tiles_kernel<<<1, BUILD_THREADS, 0, s>>>(*runs, static_cast<int>(B), static_cast<int>(L), tile_rows, count, tiles);
  FDM_CHECK_LAUNCH();
  const int64_t max_tiles = max_run_tiles(B, L, runs->n_runs);
  if (algo == FDM_VQ_TENSOR)
    return fdm_vq_tc_launch(z, codebook, nullptr, B, L, D, static_cast<int>(n_codes), indices, zq_bdl, zq_rows,
                            reinterpret_cast<unsigned long long*>(recheck_rows), nullptr, tiles, count, max_tiles, s);
  switch (D) {
    case 32: return launch_vq<32>(z, codebook, nullptr, B, L, static_cast<int>(n_codes), indices, zq_bdl, zq_rows, tiles, count, max_tiles, s);
    case 64: return launch_vq<64>(z, codebook, nullptr, B, L, static_cast<int>(n_codes), indices, zq_bdl, zq_rows, tiles, count, max_tiles, s);
    default: return launch_vq<128>(z, codebook, nullptr, B, L, static_cast<int>(n_codes), indices, zq_bdl, zq_rows, tiles, count, max_tiles, s);
  }
}
