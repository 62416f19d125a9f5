// fdm_vq_quantize, tensor-core path (D = 64 / 128): EVQ-VAE nearest-code search as a distance GEMM on tcgen05 with an exact
// recheck, so that the indices stay BIT-EXACT against the defined fp32 expression of the oracle (oracle/vq_ref.c,
// restating models/lib/quantizer.py:35-64 and models/vq_vae_emotion.py:221-252):
//     d_j = fl(fl(zz + ee_j) - fl(2 * dot_j)),  zz / ee_j / dot_j sequential fmaf chains over k = 0..63 from +0.0f,
//     index = argmin_j d_j, lowest j on ties.
// The FFMA kernel (vq.cu) evaluates all 256 chains per row: 32.8 kFLOP per 520 bytes of traffic, compute-bound at 5 % of
// the HBM roofline. Here the tensor cores only FILTER:
//   * z and the codebook are split into bf16 pairs (x = hi + lo + r, |r| <= 2^-18 |x|); one tcgen05.mma chain per
//     128-row tile against the smem-resident codebook (N = 256 codes) accumulates, in fp32 in TMEM,
//         a_j = z_hi.e_hi + z_lo.e_hi + z_hi.e_lo - ee_j / 2       ~  (zz - d_j) / 2
//     (bf16 products are exact in fp32; -ee_j/2 enters through a 13th k-step: a constant A column of ones against
//     three bf16 terms of -ee_j/2). The best code MAXIMISES a_j.
//   * error budget, in units of a:  eta = DOT + RND with
//         DOT  = 2^-15 |z| |e|_max   >= |acc - dot_ref|. Worst case 2^-15.8: 3 * 2^-18 for the dropped split terms
//                (z_lo.e_lo and the two residuals), 64 * 2^-24 = 2^-18 for the reference's own fmaf chain, 13 fp32
//                accumulation steps in the tensor core (< 2^-19.3 even if each truncates by 2 ulp); Cauchy-Schwarz turns
//                sum |z_k e_k| into |z| |e|. Measured on the device: 2^-17.8 over millions of pairs (tests assert < 2^-16),
//         RND  = 2^-23 zz + 2^-21 ee_max >= half of the three fp32 roundings in d_j (1.5 * 2^-24 (zz + ee_j)) plus the
//                bf16x3 image of ee_j / 2 and the rounding when it meets the dot product (measured < 2^-22 ee_j).
//     A code with a_j < max_j a_j - 2 eta cannot be the arg-min of d. A row with exactly one code inside that window is
//     decided; otherwise (ties, near-ties, NaNs: a fraction of a percent of the rows) the warp evaluates the exact fmaf
//     chains of the candidate codes only and takes the lexicographic (d, j) minimum like the oracle's ascending strict '<'.
//   * the per-row scan reads the accumulator ONCE (TMEM reads run at 64 B/clk/SM, ~2k cycles per 128 KB sweep: a second
//     sweep costs as much as the MMAs) and is split over the two arithmetic pipes: per 32-code chunk the running maximum
//     comes from 3-input FMNMX (half-rate ALU pipe, 0.5 instruction per code), then FFMA.SAT / FADD / FFMA (full-rate FMA
//     pipe, 3 per code) count the codes inside the window of the running maximum and accumulate their index:
//     ind_j = sat((a_j - thr) 2^60) in {0, 1}, S = sum ind_j, J = sum ind_j j; S == 1 means "decided, index J".
//     (Tracking (max, second max, index) with min/max/select was ALU-pipe-bound; two sweeps were TMEM-bound.)
// Rows containing +-Inf / NaN (|z|^2 not finite) always take the exact pass and come out as code 0, like the oracle.
// Pipeline of one persistent CTA (448 threads, 1 CTA / SM, contiguous range of 128-row tiles):
//   warps 10-13 fp32 rows from global memory (L2 hits: cp.async.bulk.prefetch.L2 two tiles ahead; the next tile's 16-byte units
//               are loaded into the registers as the current ones are consumed) -> (hi, lo) bf16 in the 128B-swizzled K-major
//               A-operand layout, |z|^2 estimate per row
//   warp 8      idle (it fed a shared-memory staging ring with 1-D TMA copies in the first version: -DVQ_RING64=1)
//   warp 9      13 x tcgen05.mma (128 x 256 x 16) per tile into one of two 256-column TMEM accumulators
//   warps 0-7   two epilogue groups (one per accumulator): tcgen05.ld, pass A / pass B over the scores, recheck,
//               int64 index, gather of the winning code row into z_q (B, D, L) and / or (B, L, D)
// Per-clip codebook slices (MEAD emotions) are handled as segments: the CTA drains, reloads the slice, continues. Per-row
// slices (fdm_vq_quantize_runs) come as a table of tiles that never cross a run, so a segment is a stretch of tiles of runs with
// one slice; a run's last tile may be partial and is handled like a clip's ragged last tile.
// This file is the kernel body; vq_tc.cu includes it once per latent width (VQ_D = 64, 128; VQ_NS = its namespace).
// D = 128 (BIWI, models/utils/config.py:44-60 / models/vq_vae.py:219-248): a 128-row tile is processed as KH = 2
// K-HALVES of 64 dimensions. Each half is one A-operand stage (hi, lo; the same 32 KB the D = 64 kernel uses per tile)
// and its 12 MMAs accumulate into the tile's TMEM accumulator; the codebook operands take 4 x 32 KB (two halves x hi, lo),
// which leaves no room for the fp32 staging ring: the converter warps read their 8-float units straight from global
// memory (L2 hits: the tiles are prefetched into L2 two tiles ahead), 16 x 16 bytes in flight per thread, issued BEFORE
// the wait for the free A stage so that the load latency hides behind the previous half's MMAs.
namespace VQ_NS {

constexpr int D = VQ_D;
constexpr int KH = D / 64;                    // 64-dimension K-halves per row (one A stage each)
// The first D = 64 kernel staged the fp32 rows through a 9-deep shared-memory ring fed by 1-D TMA copies (warp 8) and converted
// them from there; reading global memory directly with the register prefetch below is faster (8.16 M rows: indices 1.03 -> 0.90 ms,
// with z_q 1.26 -> 1.24 ms, A/B on one box) because the converter warps, not the loads, set the pace and the ring added a barrier
// wait and a shared-memory round trip per 32 rows. -DVQ_RING64=1 builds the ring variant (D = 64 only) for comparison.
#ifndef VQ_RING64
#define VQ_RING64 0
#endif
constexpr bool RING = (D == 64) && VQ_RING64;
constexpr int TILE_ROWS = 128;
constexpr int STG_ROWS = 32;
constexpr int STG_STAGES = RING ? 9 : 1;       // (D = 128: no ring; one dummy barrier pair)
constexpr int STG_BYTES = STG_ROWS * 64 * 4;  // 8 KB of fp32 rows
constexpr int A_STAGES = 2;
constexpr int A_OP_BYTES = TILE_ROWS * 128;   // 128 rows x 64 bf16
constexpr int A_STAGE_BYTES = 2 * A_OP_BYTES; // hi, lo
constexpr int B_OP_BYTES = 256 * 128;         // 256 codes x 64 bf16 (one K-half)
constexpr int AUG_A_BYTES = TILE_ROWS * 32;   // 128 rows x 16 bf16, no swizzle (8 x 16 B core matrices)
constexpr int AUG_B_BYTES = 256 * 32;
constexpr int AUG_LBO = 128, AUG_SBO = 256;   // k-chunk stride, 8-row group stride
constexpr int ZZ_SLOTS = 4;
constexpr int L2_AHEAD = 2;  // tiles prefetched into L2 ahead of the shared-memory ring (8 tiles = 38 MB chip-wide were partly evicted before
                             // use: ncu DRAM reads 2.51 GB for 2.09 GB of latents; 2 tiles: 2.09 GB, same speed)
#ifndef VQ_CONV_WARPS
#define VQ_CONV_WARPS 4
#endif
constexpr int CONV_THREADS = VQ_CONV_WARPS * 32;  // 4 (448 threads, 128 registers) or 8 converter warps (576 threads, 96 registers)
constexpr int CONV_RPP = CONV_THREADS / 8;           // rows per pass of the converter group (8 threads per row)
constexpr int CONV_UNITS = TILE_ROWS / CONV_RPP;     // 8-float units per thread and K-half
static_assert(!RING || VQ_CONV_WARPS == 4, "the ring variant is written for four converter warps");
constexpr int NUM_THREADS = 320 + CONV_THREADS;
// Warp roles. The SMSP arbiter prefers the HIGHEST warp id among eligible warps, so the converters - the head of the
// pipeline, one warp per scheduler - get the top ids; with ids 0-3 they only issued when both epilogue warps of their
// scheduler were stalled and took ~4k cycles per tile.
constexpr int EPI_WARP0 = 0;    // warps 0-7: epilogue (group = warp >> 2, TMEM lane quadrant = warp & 3)
constexpr int LOAD_WARP = 8;
constexpr int MMA_WARP = 9;
constexpr int CONV_WARP0 = 10;  // warps 10-13

constexpr int OFF_B = 0;                                   // per K-half: e_hi, e_lo
constexpr int OFF_A = OFF_B + KH * 2 * B_OP_BYTES;         // 2 stages x (z_hi, z_lo)
constexpr int OFF_STG = OFF_A + A_STAGES * A_STAGE_BYTES;  // fp32 staging ring
constexpr int OFF_AUG_A = OFF_STG + (RING ? STG_STAGES * STG_BYTES : 0);
constexpr int OFF_AUG_B = OFF_AUG_A + AUG_A_BYTES;
constexpr int OFF_EE = OFF_AUG_B + AUG_B_BYTES;            // ee[256]
constexpr int OFF_ZZ = OFF_EE + 256 * 4;                   // zz estimate [ZZ_SLOTS][128]
constexpr int OFF_BAR = OFF_ZZ + ZZ_SLOTS * TILE_ROWS * 4;
constexpr int NUM_BARS = 2 * STG_STAGES + 2 * A_STAGES + 2 * 2;
constexpr int OFF_MISC = OFF_BAR + NUM_BARS * 8;           // tmem slot, ee_max bits
constexpr int OFF_ZROW = OFF_MISC + 16;                    // one fp32 latent row per epilogue warp (exact pass)
// Deferred exact pass: rows whose tensor-core scores leave more than one candidate are queued here (row, candidate
// masks) and decided after the segment's last tile, one row per thread, instead of stalling their epilogue group for a
// 3-4k-cycle dependent fmaf chain in the middle of the tile pipeline (0.2 % of the rows, but 6 % of the warps and 22 % of
// the tiles had one: the inline pass cost 20 % of the kernel). A full queue falls back to the inline pass.
constexpr int DEFER_CAP = 192;
constexpr int DEFER_ENTRY_BYTES = 40;                                    // int64 row + 8 candidate-mask words
constexpr int OFF_DEFER = OFF_ZROW + 8 * (D + 16) * 4;                    // uint32 count (16 bytes), then the entries
constexpr int SMEM_BYTES = OFF_DEFER + 16 + DEFER_CAP * DEFER_ENTRY_BYTES + 1024;  // + manual 1024-byte alignment
static_assert(SMEM_BYTES <= 232448, "shared memory budget");

// D = 128: the reference chain's own error doubles (128 * 2^-24 = 2^-17) and the tensor core takes 25 accumulation steps
// (< 2^-18.3): worst case 2^-15.5, budget 1.5 * 2^-15
constexpr float C_DOT = (D == 64 ? 1.0f : 1.5f) / 32768.0f;     // 2^-15
constexpr float C_RND_ZZ = 1.0f / 8388608.0f;  // 2^-23
constexpr float C_RND_EE = 1.0f / 2097152.0f;  // 2^-21

// tcgen05 / TMEM / mbarrier PTX wrappers: tc_common.cuh (namespace tc), shared with the GEMM and attention kernels. This kernel keeps
// its own mbar_wait - same try_wait loop and watchdog trap, no printf in the time-out path: the kernel runs at its register limit
// and the printf call costs a stack frame in every role - and the 1-D bulk-copy / L2-prefetch forms only it uses.
using namespace tc;
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0, spins = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if (done) break;
    if (++spins > (1u << 26)) __trap();  // watchdog: a protocol bug must trap, never hang the GPU
  }
}
__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void bulk_prefetch_l2(const void* src, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(reinterpret_cast<uint64_t>(src)), "r"(bytes) : "memory");
}
// K-major SWIZZLE_128B operand descriptor (8-row x 128-byte atoms, SBO = 1024 B) and the bf16 x bf16 -> f32 instruction descriptor
__device__ __forceinline__ uint64_t make_kmajor_sw128_desc(uint32_t smem_addr) { return make_desc_sw128(smem_addr, 16, 1024); }
__device__ __forceinline__ uint32_t make_idesc_bf16_f32(int m, int n) { return make_idesc_bf16(m, n, 0); }
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// x[0..7] -> bf16 hi (round to nearest) and bf16 lo = rn(x - hi); element k sits at byte 2k of the 16-byte chunk
__device__ __forceinline__ void split8(const float4& a, const float4& b, uint4& hi, uint4& lo) {
  const float x[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  uint32_t h[4], l[4];
#pragma unroll
  for (int p = 0; p < 4; ++p) {
    const __nv_bfloat162 hh = __floats2bfloat162_rn(x[2 * p], x[2 * p + 1]);
    const float2 hf = __bfloat1622float2(hh);
    const __nv_bfloat162 ll = __floats2bfloat162_rn(x[2 * p] - hf.x, x[2 * p + 1] - hf.y);
    h[p] = *reinterpret_cast<const uint32_t*>(&hh);
    l[p] = *reinterpret_cast<const uint32_t*>(&ll);
  }
  hi = make_uint4(h[0], h[1], h[2], h[3]);
  lo = make_uint4(l[0], l[1], l[2], l[3]);
}

// K-major, no swizzle: 8-row x 16-byte core matrices, LBO = next k chunk, SBO = next 8-row group
__device__ __forceinline__ uint64_t make_kmajor_noswz_desc(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  return d;
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
__device__ __forceinline__ float sqrt_approx(float x) {
  float y;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint16_t bf16_bits(float x) {
  const __nv_bfloat16 h = __float2bfloat16_rn(x);
  return *reinterpret_cast<const uint16_t*>(&h);
}

// -DVQ_TRACE: CTA 0 records clock64() stamps per tile and role into dbg_acc (as long long) for timeline analysis
#ifdef VQ_TRACE
#define TRACE(slot) do { if (p.dbg_acc && blockIdx.x == 0 && lane == 0 && it < 96) reinterpret_cast<long long*>(p.dbg_acc)[it * 16 + (slot)] = clock64(); } while (0)
#else
#define TRACE(slot) do {} while (0)
#endif

struct Params {
  const float* z;
  const float* codebook;
  const int64_t* code_offset;
  int64_t B, L;
  int n_codes;
  int64_t* indices;
  float* zq_bdl;
  float* zq_rows;
  unsigned long long* recheck_rows;  // optional counter of rows that took the exact path
  float* dbg_acc;                    // optional [rows, n_codes] dump of a_j = dot_j - ee_j / 2 from the tensor cores (tests)
  int tiles_per_clip, num_tiles;  // 32-bit on purpose: tile -> (clip, row) divisions stay inline
  const VqTile* tiles;            // per-row slices (fdm_vq_quantize_runs): tile t is tiles[t], *tile_count of them; else NULL
  const int* tile_count;
  float window_scale;  // 1.0; profiling knob FDM_B200_VQ_WINDOW (0 = never take the exact pass: NOT bit-exact)
  int l2_ahead;        // tiles prefetched into L2 ahead of the shared-memory ring (FDM_B200_VQ_L2_AHEAD, default L2_AHEAD)
};

// Clip, first row and row count of tile tl: 128-row tiles of whole clips, or (TL: fdm_vq_quantize_runs) the caller's tile table,
// one 16-byte load per tile. The kernel is instantiated for both, so the per-clip path compiles exactly as without tables.
struct TileRef { int b; int64_t l0; int nrows; };
template <bool TL>
__device__ __forceinline__ TileRef tile_ref(const VqTile* tiles, int tpc, int64_t L, int tl) {
  if constexpr (TL) {
    const int4 t = __ldg(reinterpret_cast<const int4*>(tiles) + tl);
    return TileRef{t.x, t.y, t.z};
  }
  const int b = tl / tpc;
  const int64_t l0 = static_cast<int64_t>(tl - b * tpc) * TILE_ROWS;
  return TileRef{b, l0, static_cast<int>(min(static_cast<int64_t>(TILE_ROWS), L - l0))};
}

// Exact pass for ONE flagged row (rare, latency-bound; out of line and lean on registers: with 226 KB of the SM's
// 256 KB carved out as shared memory every local-memory spill is an L2 round trip, and an earlier version that kept 16
// float4 of a code row live spent ~16k cycles per flagged warp in spill traffic). scratch = the row's 64 floats followed
// by its 8 candidate-mask words, in shared memory. Lane i evaluates the oracle's chains for the candidate codes
// j = 32 c + i in ascending c; the warp then takes the lexicographic (d, j) minimum (= ascending j with strict '<').
__device__ __noinline__ int exact_one(const float* __restrict__ cbg, const float* ee, const float* scratch, int lane) {
  const float4* z4 = reinterpret_cast<const float4*>(scratch);
  const uint32_t* mk = reinterpret_cast<const uint32_t*>(scratch + D);
  float zz = 0.f;
#pragma unroll
  for (int k = 0; k < D / 4; ++k) {
    const float4 a = z4[k];
    zz = fmaf(a.x, a.x, zz); zz = fmaf(a.y, a.y, zz); zz = fmaf(a.z, a.z, zz); zz = fmaf(a.w, a.w, zz);
  }
  float best = INFINITY;
  int bi = 0x7fffffff;
#pragma unroll 1
  for (int c = 0; c < 8; ++c) {
    if ((mk[c] >> lane) & 1u) {
      const int j = c * 32 + lane;
      const float4* e4 = reinterpret_cast<const float4*>(cbg + j * D);
      float dot = 0.f;
#pragma unroll
      for (int h = 0; h < D / 32; ++h) {
        float4 ev[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) ev[k] = __ldg(e4 + h * 8 + k);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float4 a = z4[h * 8 + k], e = ev[k];
          dot = fmaf(a.x, e.x, dot); dot = fmaf(a.y, e.y, dot); dot = fmaf(a.z, e.z, dot); dot = fmaf(a.w, e.w, dot);
        }
      }
      const float dist = __fsub_rn(__fadd_rn(zz, ee[j]), __fmul_rn(2.f, dot));
      if (dist < best) { best = dist; bi = j; }  // NaN / +Inf never win (oracle: strict '<' from +Inf)
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float od = __shfl_xor_sync(0xffffffffu, best, o);
    const int oj = __shfl_xor_sync(0xffffffffu, bi, o);
    if (od < best || (od == best && oj < bi)) { best = od; bi = oj; }
  }
  return bi == 0x7fffffff ? 0 : bi;
}

// ---- barriers (shared-memory addresses relative to the 1024-aligned base) -------------------------------------------
__device__ __forceinline__ uint32_t bar_stg_full(uint32_t base, int s) { return base + OFF_BAR + 8u * s; }
__device__ __forceinline__ uint32_t bar_stg_empty(uint32_t base, int s) { return base + OFF_BAR + 8u * (STG_STAGES + s); }
__device__ __forceinline__ uint32_t bar_a_full(uint32_t base, int s) { return base + OFF_BAR + 8u * (2 * STG_STAGES + s); }
__device__ __forceinline__ uint32_t bar_a_empty(uint32_t base, int s) { return base + OFF_BAR + 8u * (2 * STG_STAGES + A_STAGES + s); }
__device__ __forceinline__ uint32_t bar_t_full(uint32_t base, int s) { return base + OFF_BAR + 8u * (2 * STG_STAGES + 2 * A_STAGES + s); }
__device__ __forceinline__ uint32_t bar_t_empty(uint32_t base, int s) { return base + OFF_BAR + 8u * (2 * STG_STAGES + 2 * A_STAGES + 2 + s); }

// What every role needs. Each role is its own __noinline__ function so that it gets its own register allocation: inlined
// into one kernel body the loop counters of the light roles were spilled to local memory (L1 is almost entirely carved
// out as shared memory here, so every reload was an L2 round trip on the converters' critical path).
struct Ctx {
  uint32_t base;      // shared-memory address of the 1024-aligned carve-up
  uint8_t* smem;      // generic pointer to the same place
  uint32_t tmem_base;
  int t_begin, t_end; // this CTA's tiles
};

// A segment is a maximal run of this CTA's tiles that share one codebook slice. All threads call this at the start
// of every segment: they drain (barrier), convert the slice into the B operands, compute ee, and return its end.
template <bool TL>
__device__ __noinline__ int segment_begin(const Params& p, const Ctx& cx, int tile, int64_t* off_out) {
  const int tid = threadIdx.x;
  const int n_codes = p.n_codes, tpc = p.tiles_per_clip;
  const uint32_t base = cx.base;
  float* ee = reinterpret_cast<float*>(cx.smem + OFF_EE);
  uint32_t* ee_max_bits = reinterpret_cast<uint32_t*>(cx.smem + OFF_MISC + 4);
  int64_t off = 0;
  int seg_end = cx.t_end;
  if constexpr (TL) {  // (a run's tiles are consecutive, so a slice change between tiles is a run boundary)
    off = p.tiles[tile].off;
    for (int t = tile + 1; t < cx.t_end; ++t)
      if (p.tiles[t].off != off) { seg_end = t; break; }
  } else if (p.code_offset) {
    const int b0 = tile / tpc;
    off = p.code_offset[b0];
    for (int bb = b0 + 1; bb * tpc < cx.t_end; ++bb)
      if (p.code_offset[bb] != off) { seg_end = bb * tpc; break; }
  }
  const float* cbg = p.codebook + off * D;
  __syncthreads();  // every role is done with the previous slice (epilogue waits imply its MMAs have retired)
  if (tid == 0) {
    *ee_max_bits = 0u;
    *reinterpret_cast<uint32_t*>(cx.smem + OFF_DEFER) = 0u;  // deferred-row queue of this segment
  }
  for (int i = tid; i < n_codes * (D / 8); i += NUM_THREADS) {
    const int c = i / (D / 8), cc = i % (D / 8), h = cc >> 3, c8 = cc & 7;
    const float4* src = reinterpret_cast<const float4*>(cbg + c * D + cc * 8);
    uint4 hi, lo;
    split8(__ldg(src), __ldg(src + 1), hi, lo);
    const uint32_t o = static_cast<uint32_t>(h * 2 * B_OP_BYTES + c * 128 + ((c8 ^ (c & 7)) << 4));
    st_shared_v4(base + OFF_B + o, hi);
    st_shared_v4(base + OFF_B + B_OP_BYTES + o, lo);
  }
  __syncthreads();
  for (int c = tid; c < n_codes; c += NUM_THREADS) {
    float s = 0.f;
    for (int k = 0; k < D; ++k) { const float e = __ldg(cbg + c * D + k); s = fmaf(e, e, s); }
    ee[c] = s;
    if (s == s) atomicMax(ee_max_bits, __float_as_uint(fabsf(s)));  // non-negative floats order like their bit patterns
    // B row of the 13th k-step: -ee/2 as three bf16 terms
    const float g = -0.5f * s;
    const uint16_t g0 = bf16_bits(g);
    const float r1 = g - __uint_as_float(static_cast<uint32_t>(g0) << 16);
    const uint16_t g1 = bf16_bits(r1);
    const float r2 = r1 - __uint_as_float(static_cast<uint32_t>(g1) << 16);
    const uint16_t g2 = bf16_bits(r2);
    const uint32_t o = static_cast<uint32_t>((c & 7) * 16 + (c >> 3) * AUG_SBO);
    st_shared_v4(base + OFF_AUG_B + o, make_uint4(static_cast<uint32_t>(g0) | (static_cast<uint32_t>(g1) << 16), g2, 0u, 0u));
    st_shared_v4(base + OFF_AUG_B + o + AUG_LBO, make_uint4(0u, 0u, 0u, 0u));
  }
  fence_async_smem();
  __syncthreads();
  *off_out = off;
  return seg_end;
}

// ===== converters (warps 10-13): staged fp32 rows -> bf16 (hi, lo) A operand + |z|^2 estimate =====
template <bool TL>
__device__ __noinline__ void role_convert(const Params& p, const Ctx& cx) {
  const int tid = threadIdx.x - CONV_WARP0 * 32, lane = tid & 31;
  const int64_t L = p.L;
  const int tpc = p.tiles_per_clip;
  const VqTile* const tiles = p.tiles;
  const uint32_t base = cx.base;
  // (Params / Ctx live in memory behind references: everything the loops need is copied into registers first)
  uint8_t* const smem = cx.smem;
  const int t_end = cx.t_end;
  float* zzs = reinterpret_cast<float*>(smem + OFF_ZZ);
  uint32_t it = 0, hc = 0;
  const int row_q = tid >> 3, c8 = tid & 7;  // this thread's (row, 8-float column block) inside a 16-row slab
  // (D = 128) address of this thread's unit 0 (row row_q, columns 64 h + 8 c8 ..) of sub-tile (tile, K-half), rows in the tile
  auto unit0_of = [&](int tl2, int h2, int& nrows2) -> const float* {
    const TileRef t2 = tile_ref<TL>(tiles, tpc, L, tl2);
    nrows2 = t2.nrows;
    return p.z + (static_cast<int64_t>(t2.b) * L + t2.l0 + row_q) * D + h2 * 64 + c8 * 8;
  };
  float4 x0[CONV_UNITS], x1[CONV_UNITS];
  if (!RING && cx.t_begin < t_end) {  // the first sub-tile's loads
    int nr0;
    const float* s0 = unit0_of(cx.t_begin, 0, nr0);
#pragma unroll
    for (int u = 0; u < CONV_UNITS; ++u) {
      if (row_q + CONV_RPP * u < nr0) {
        const float4* src = reinterpret_cast<const float4*>(s0 + static_cast<int64_t>(CONV_RPP * u) * D);
        x0[u] = __ldg(src);
        x1[u] = __ldg(src + 1);
      } else {
        x0[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        x1[u] = x0[u];
      }
    }
  }
  for (int tile = cx.t_begin; tile < t_end;) {
    int64_t off;
    const int seg_end = segment_begin<TL>(p, cx, tile, &off);
    for (int tl = tile; tl < seg_end; ++tl, ++it) {
      const int nrows = RING ? tile_ref<TL>(tiles, tpc, L, tl).nrows : 0;  // (the no-ring path takes row counts from unit0_of)
      float* zz = zzs + (it & (ZZ_SLOTS - 1)) * TILE_ROWS;
      if (RING) {
        const int as = it & 1;
        TRACE(0);
        mbar_wait(bar_a_empty(base, as), ((it >> 1) & 1u) ^ 1u);
        TRACE(1);
        const uint32_t a_hi = base + OFF_A + as * A_STAGE_BYTES, a_lo = a_hi + A_OP_BYTES;
        // All staged quarters of the tile are converted in one unrolled sweep (8 independent 8-float units per thread):
        // with one quarter at a time the four converter warps were latency-bound at ~950 cycles per quarter.
        const int nparts = (nrows + STG_ROWS - 1) / STG_ROWS;
        float sqv[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int part = 0; part < TILE_ROWS / STG_ROWS; ++part) {
          if (part < nparts) {
            const int s = (hc + part) % STG_STAGES;
            mbar_wait(bar_stg_full(base, s), ((hc + part) / STG_STAGES) & 1u);
            const uint8_t* stg = smem + OFF_STG + s * STG_BYTES;
            float4 x0[2], x1[2];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              const float4* src = reinterpret_cast<const float4*>(stg + (row_q + 16 * q) * (64 * 4) + c8 * 32);
              x0[q] = src[0];
              x1[q] = src[1];
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_stg_empty(base, s));  // this warp has read its rows of the staging slot
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              const int row = row_q + 16 * q;
              uint4 hi, lo;
              split8(x0[q], x1[q], hi, lo);
              const int arow = part * STG_ROWS + row;
              const uint32_t o = static_cast<uint32_t>(arow * 128 + ((c8 ^ (row & 7)) << 4));
              st_shared_v4(a_hi + o, hi);
              st_shared_v4(a_lo + o, lo);
              float sq = x0[q].x * x0[q].x;
              sq = fmaf(x0[q].y, x0[q].y, sq); sq = fmaf(x0[q].z, x0[q].z, sq); sq = fmaf(x0[q].w, x0[q].w, sq);
              sq = fmaf(x1[q].x, x1[q].x, sq); sq = fmaf(x1[q].y, x1[q].y, sq); sq = fmaf(x1[q].z, x1[q].z, sq); sq = fmaf(x1[q].w, x1[q].w, sq);
              sqv[part * 2 + q] = sq;
            }
          }
        }
        // the eight row sums' butterfly rounds back to back: within a round the shuffles are independent, so the warp does not
        // sit out a shuffle latency per unit (D = 128 converter: 0.38 -> 0.31 ms for 1.22 M rows with the same change)
#pragma unroll
        for (int o = 1; o <= 4; o <<= 1) {
#pragma unroll
          for (int u = 0; u < 8; ++u) sqv[u] += __shfl_xor_sync(0xffffffffu, sqv[u], o);
        }
        if (c8 == 0) {
#pragma unroll
          for (int u = 0; u < 8; ++u)
            if ((u >> 1) < nparts) zz[(u >> 1) * STG_ROWS + row_q + 16 * (u & 1)] = sqv[u];
        }
        hc += nparts;
        fence_async_smem();  // generic-proxy stores -> visible to tcgen05.mma (async proxy)
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_a_full(base, as));
        TRACE(2);
      } else {
        // ---- no staging ring (D = 128): global -> registers -> (hi, lo) A stage, one K-half at a time. The registers hold
        //      the sub-tile being converted; as soon as a unit has been consumed its registers receive the same unit of the
        //      NEXT sub-tile, so 16 x 16 bytes per thread stay in flight through the whole conversion. (The converters are the
        //      bottleneck of this variant: ~3k cycles per K-half, a 600-instruction dependent sequence on one warp per
        //      scheduler - ncu: 19 % issue slots, the rest fixed-latency and shuffle waits. Two converter groups - 576
        //      threads, 96 registers - were tried on alternate K-halves and on alternate tiles: 0.35-0.37 ms against 0.38 ms
        //      for 1.22 M rows, not worth the second producer protocol.) ----
        if (tid == 0) {  // pull the tiles ahead into L2 (the loads then hit L2)
          const int ahead = p.l2_ahead;
          const int first = (tl == cx.t_begin) ? tl + 1 : tl + ahead;
          for (int ta = first; ta <= tl + ahead && ta < t_end; ++ta) {
            const TileRef a = tile_ref<TL>(tiles, tpc, L, ta);
            bulk_prefetch_l2(p.z + (static_cast<int64_t>(a.b) * L + a.l0) * D, static_cast<uint32_t>(a.nrows) * D * 4);
          }
        }
#pragma unroll 1
        for (int h = 0; h < KH; ++h) {
          const uint32_t sit = it * KH + h;
          const int as = sit & 1;
          // the sub-tile after this one: the other K-half, or the first K-half of the next tile
          const int ntl = (h + 1 < KH) ? tl : tl + 1, nh = (h + 1 < KH) ? h + 1 : 0;
          int nnr = 0;
          const float* nsrc = nullptr;
          if (ntl < t_end) nsrc = unit0_of(ntl, nh, nnr);
          TRACE(h == KH - 1 ? 0 : 13);
          mbar_wait(bar_a_empty(base, as), ((sit >> 1) & 1u) ^ 1u);
          TRACE(h == KH - 1 ? 1 : 14);
          const uint32_t a_hi = base + OFF_A + as * A_STAGE_BYTES, a_lo = a_hi + A_OP_BYTES;
          float sq[CONV_UNITS];
#pragma unroll
          for (int u = 0; u < CONV_UNITS; ++u) {
            const int row = row_q + CONV_RPP * u;
            uint4 hi, lo;
            split8(x0[u], x1[u], hi, lo);
            const uint32_t o = static_cast<uint32_t>(row * 128 + ((c8 ^ (row & 7)) << 4));
            st_shared_v4(a_hi + o, hi);
            st_shared_v4(a_lo + o, lo);
            float q = x0[u].x * x0[u].x;
            q = fmaf(x0[u].y, x0[u].y, q); q = fmaf(x0[u].z, x0[u].z, q); q = fmaf(x0[u].w, x0[u].w, q);
            q = fmaf(x1[u].x, x1[u].x, q); q = fmaf(x1[u].y, x1[u].y, q); q = fmaf(x1[u].z, x1[u].z, q); q = fmaf(x1[u].w, x1[u].w, q);
            sq[u] = q;
            if (row < nnr) {  // (nnr = 0 when there is no next sub-tile)
              const float4* src = reinterpret_cast<const float4*>(nsrc + static_cast<int64_t>(CONV_RPP * u) * D);
              x0[u] = __ldg(src);
              x1[u] = __ldg(src + 1);
            } else {
              x0[u] = make_float4(0.f, 0.f, 0.f, 0.f);
              x1[u] = x0[u];
            }
          }
          // the eight row sums' butterfly rounds back to back (each round's shuffles are independent of one another)
#pragma unroll
          for (int o = 1; o <= 4; o <<= 1) {
#pragma unroll
            for (int u = 0; u < CONV_UNITS; ++u) sq[u] += __shfl_xor_sync(0xffffffffu, sq[u], o);
          }
          if (c8 == 0) {  // the same thread owns (row, c8 = 0) in both K-halves
#pragma unroll
            for (int u = 0; u < CONV_UNITS; ++u) zz[row_q + CONV_RPP * u] = (h == 0) ? sq[u] : zz[row_q + CONV_RPP * u] + sq[u];
          }
          fence_async_smem();  // generic-proxy stores -> visible to tcgen05.mma (async proxy)
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_a_full(base, as));
          TRACE(h == KH - 1 ? 2 : 15);
        }
      }
    }
    tile = seg_end;
  }
}

// ===== MMA issuer (warp 9) =====
template <bool TL>
__device__ __noinline__ void role_mma(const Params& p, const Ctx& cx) {
  const int lane = threadIdx.x & 31;
  const uint32_t base = cx.base;
  const uint32_t idesc = make_idesc_bf16_f32(TILE_ROWS, p.n_codes);
  const uint64_t b_hi0 = make_kmajor_sw128_desc(base + OFF_B);  // K-half h: + h * 2 * B_OP_BYTES; lo: + B_OP_BYTES
  const uint64_t aug_a = make_kmajor_noswz_desc(base + OFF_AUG_A, AUG_LBO, AUG_SBO);
  const uint64_t aug_b = make_kmajor_noswz_desc(base + OFF_AUG_B, AUG_LBO, AUG_SBO);
  const uint32_t tmem_base = cx.tmem_base;
  const int t_end = cx.t_end;
  uint32_t it = 0;
  for (int tile = cx.t_begin; tile < t_end;) {
    int64_t off;
    const int seg_end = segment_begin<TL>(p, cx, tile, &off);
    for (int tl = tile; tl < seg_end; ++tl, ++it) {
      if (lane == 0) {
        const int acc = it & 1;
        TRACE(3);
        mbar_wait(bar_t_empty(base, acc), ((it >> 1) & 1u) ^ 1u);  // the epilogue group has drained this accumulator
        TRACE(4);
        const uint32_t tmem_d = tmem_base + acc * 256;
#pragma unroll 1
        for (int h = 0; h < KH; ++h) {
          const uint32_t sit = it * KH + h;  // A stages cycle per K-half
          const int as = sit & 1;
          mbar_wait(bar_a_full(base, as), (sit >> 1) & 1u);
          TRACE(5);
          tcgen05_fence_after();
          const uint64_t a_hi = make_kmajor_sw128_desc(base + OFF_A + as * A_STAGE_BYTES);
          const uint64_t a_lo = make_kmajor_sw128_desc(base + OFF_A + as * A_STAGE_BYTES + A_OP_BYTES);
          const uint64_t b_hi = b_hi0 + static_cast<uint64_t>((h * 2 * B_OP_BYTES) >> 4);
          const uint64_t b_lo = b_hi + static_cast<uint64_t>(B_OP_BYTES >> 4);
          // small cross terms first, the large -ee_j / 2 last: it meets the finished dot product in a single rounding
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16(tmem_d, a_lo + 2u * k, b_hi + 2u * k, idesc, (h != 0 || k != 0) ? 1u : 0u);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16(tmem_d, a_hi + 2u * k, b_lo + 2u * k, idesc, 1u);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16(tmem_d, a_hi + 2u * k, b_hi + 2u * k, idesc, 1u);
          if (h == KH - 1) umma_bf16(tmem_d, aug_a, aug_b, idesc, 1u);
          umma_commit(bar_a_empty(base, as));
        }
        umma_commit(bar_t_full(base, acc));
        TRACE(6);
      }
      __syncwarp();
    }
    tile = seg_end;
  }
}

// ===== loader (warp 8): 1-D bulk copies of contiguous fp32 rows =====
template <bool TL>
__device__ __noinline__ void role_load(const Params& p, const Ctx& cx) {
  const int lane = threadIdx.x & 31;
  const int64_t L = p.L;
  const int tpc = p.tiles_per_clip;
  const uint32_t base = cx.base;
  const float* const zsrc = p.z;
  const VqTile* const tiles = p.tiles;
  const int t_end = cx.t_end;
  uint32_t it = 0, hc = 0;
  for (int tile = cx.t_begin; tile < t_end;) {
    int64_t off;
    const int seg_end = segment_begin<TL>(p, cx, tile, &off);
    for (int tl = tile; RING && tl < seg_end; ++tl, ++it) {  // (D = 128: the converters load; this warp only takes part in the segment barriers)
      const TileRef t0 = tile_ref<TL>(tiles, tpc, L, tl);
      const int b = t0.b;
      const int64_t l0 = t0.l0;
      const int nrows = t0.nrows;
      // The ring holds 2.25 tiles = 72 KB, which at ~1.8 us of loaded HBM latency is ~40 GB/s per SM: latency-bound at
      // a third of the HBM rate. Tiles further ahead are pulled into L2 so that the ring's copies are L2 hits.
      if (lane == 0) {
        const int ahead = p.l2_ahead;
        const int first = (tl == cx.t_begin) ? tl + 1 : tl + ahead;
        for (int ta = first; ta <= tl + ahead && ta < t_end; ++ta) {
          const TileRef a = tile_ref<TL>(tiles, tpc, L, ta);
          bulk_prefetch_l2(zsrc + (static_cast<int64_t>(a.b) * L + a.l0) * D, static_cast<uint32_t>(a.nrows) * D * 4);
        }
      }
      for (int part = 0; part < TILE_ROWS / STG_ROWS; ++part) {
        const int hr = min(STG_ROWS, nrows - part * STG_ROWS);
        if (hr <= 0) break;
        if (lane == 0) {
          const int s = hc % STG_STAGES;
          mbar_wait(bar_stg_empty(base, s), ((hc / STG_STAGES) & 1u) ^ 1u);
          mbar_expect_tx(bar_stg_full(base, s), static_cast<uint32_t>(hr) * D * 4);
          bulk_load_1d(base + (RING ? OFF_STG + s * STG_BYTES : 0), zsrc + (static_cast<int64_t>(b) * L + l0 + part * STG_ROWS) * D,
                       static_cast<uint32_t>(hr) * D * 4, bar_stg_full(base, s));
        }
        ++hc;
      }
      TRACE(12);
      __syncwarp();
    }
    tile = seg_end;
  }
}

// Decide the queued rows of this segment: one row per epilogue thread, the oracle's chains for its candidate codes in
// ascending order (strict '<': lowest index on ties), then every output of that row.
__device__ __noinline__ void drain_deferred(const Params& p, const Ctx& cx, const float* __restrict__ cbg) {
  const int t = threadIdx.x - EPI_WARP0 * 32;  // 0 .. 255
  const uint32_t n = min(*reinterpret_cast<const uint32_t*>(cx.smem + OFF_DEFER), static_cast<uint32_t>(DEFER_CAP));
  const float* ee = reinterpret_cast<const float*>(cx.smem + OFF_EE);
  for (uint32_t e = t; e < n; e += 256) {
    const uint8_t* ent = cx.smem + OFF_DEFER + 16 + e * DEFER_ENTRY_BYTES;
    const int64_t grow = *reinterpret_cast<const int64_t*>(ent);
    const uint32_t* mk = reinterpret_cast<const uint32_t*>(ent + 8);
    const float4* z4 = reinterpret_cast<const float4*>(p.z + grow * D);
    float zz = 0.f;
#pragma unroll 4
    for (int k = 0; k < D / 4; ++k) {
      const float4 a = __ldg(z4 + k);
      zz = fmaf(a.x, a.x, zz); zz = fmaf(a.y, a.y, zz); zz = fmaf(a.z, a.z, zz); zz = fmaf(a.w, a.w, zz);
    }
    float best = INFINITY;
    int bi = 0;
#pragma unroll 1
    for (int c = 0; c < 8; ++c) {
      uint32_t m = mk[c];
      while (m) {
        const int j = c * 32 + __ffs(m) - 1;
        m &= m - 1u;
        const float4* e4 = reinterpret_cast<const float4*>(cbg + j * D);
        float dot = 0.f;
#pragma unroll 4
        for (int k = 0; k < D / 4; ++k) {
          const float4 a = __ldg(z4 + k), ev = __ldg(e4 + k);
          dot = fmaf(a.x, ev.x, dot); dot = fmaf(a.y, ev.y, dot); dot = fmaf(a.z, ev.z, dot); dot = fmaf(a.w, ev.w, dot);
        }
        const float dist = __fsub_rn(__fadd_rn(zz, ee[j]), __fmul_rn(2.f, dot));
        if (dist < best) { best = dist; bi = j; }  // ascending j, strict '<'; NaN / +Inf never win -> index 0
      }
    }
    if (p.indices) p.indices[grow] = bi;
    const int64_t b = grow / p.L, l = grow - b * p.L;
    const float* src = cbg + bi * D;
    if (p.zq_bdl) {
      float* dst = p.zq_bdl + (b * D) * p.L + l;
      for (int k = 0; k < D; ++k) dst[k * p.L] = __ldg(src + k);
    }
    if (p.zq_rows) {
      float4* dst = reinterpret_cast<float4*>(p.zq_rows + grow * D);
      for (int k = 0; k < D / 4; ++k) dst[k] = __ldg(reinterpret_cast<const float4*>(src) + k);
    }
  }
}

// ===== epilogue (warps 0-7): group g owns accumulator g =====
template <bool TL>
__device__ __noinline__ void role_epilogue(const Params& p, const Ctx& cx) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_codes = p.n_codes, nchunks = n_codes >> 5;
  const int64_t L = p.L;
  const int tpc = p.tiles_per_clip;
  const uint32_t base = cx.base;
  uint8_t* smem = cx.smem;
  const float* ee = reinterpret_cast<const float*>(smem + OFF_EE);
  const float* zzs = reinterpret_cast<const float*>(smem + OFF_ZZ);
  const int grp = (warp - EPI_WARP0) >> 2;
  const int quad = warp & 3;
  const int row = quad * 32 + lane;
  const uint32_t tmem_base = cx.tmem_base;
  const int t_end = cx.t_end;
  const float window_scale = p.window_scale;
  const float* const zsrc = p.z;
  const float* const codebook = p.codebook;
  int64_t* const out_idx = p.indices;
  float* const out_bdl = p.zq_bdl;
  float* const out_rows = p.zq_rows;
  unsigned long long* const out_recheck = p.recheck_rows;
  float* const out_dbg = p.dbg_acc;
  uint32_t it = 0;
  for (int tile = cx.t_begin; tile < t_end;) {
    int64_t off;
    const int seg_end = segment_begin<TL>(p, cx, tile, &off);
    const float* cbg = codebook + off * D;
    const float ee_max = __uint_as_float(*reinterpret_cast<const uint32_t*>(smem + OFF_MISC + 4));
    const float se_max = sqrtf(ee_max) * 1.001f;
    for (int tl = tile; tl < seg_end; ++tl, ++it) {
      if ((it & 1) != static_cast<uint32_t>(grp)) continue;
      const TileRef t0 = tile_ref<TL>(p.tiles, tpc, L, tl);
      const int64_t b = t0.b;
      const int64_t l0 = t0.l0;
      const int nrows = t0.nrows;
      const bool row_ok = row < nrows;
      const int64_t grow = b * L + l0 + row;
      if (quad == 0) TRACE(7);
      mbar_wait(bar_t_full(base, grp), (it >> 1) & 1u);
      tcgen05_fence_after();
      if (quad == 0) TRACE(8);
      const uint32_t tacc = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + grp * 256;
      const float zzr = zzs[(it & (ZZ_SLOTS - 1)) * TILE_ROWS + row];

#ifndef VQ_TRACE
      if (out_dbg) {  // tests only
#pragma unroll 1
        for (int c = 0; c < nchunks; ++c) {
          uint32_t r[32];
          tmem_ld_32x32b_x32(tacc + c * 32, r);
          tmem_ld_wait();
          if (row_ok) {
#pragma unroll
            for (int j = 0; j < 32; ++j) out_dbg[grow * n_codes + c * 32 + j] = __uint_as_float(r[j]);
          }
        }
      }
#endif

      // ---- single pass over the scores ----
      // per 32-code chunk: chunk max with 3-input FMNMX (ALU pipe, 0.5 / code), running max M, then on the FMA pipe
      // (3 / code) ind_j = [a_j >= M - w] as sat((a_j - thr) 2^60) in {0, 1}, S += ind_j, J += ind_j j. When M grows by
      // more than w the earlier counts are void and are reset; when it grows by less they are kept (conservative: the
      // row then shows S >= 2 and takes the exact pass). At the end S == 1 <=> exactly one code inside the window of
      // the final maximum, and J is its index. (A fractional ind needs 0 < a_j - thr < 2^-60: S is then not 1, or the
      // sliver lies inside the 1e-4 margin of w.)
      const float eta = (C_DOT * sqrt_approx(zzr * 1.001f) * se_max + C_RND_ZZ * zzr + C_RND_EE * ee_max) * 1.001f + 1e-37f;
      const float window = 2.f * eta * window_scale;
      const float w = window * 1.0001f;  // codes with a_j < max - w cannot be the arg-min of d
      const float big = 1.152921504606846976e18f;  // 2^60
      float M1 = -INFINITY;
      // Count and index of the codes inside the window ride in ONE accumulator per chunk: T = sum ind_j (j + 1024) over the
      // chunk's 32 codes (ind_j in {0, 1}: T = 1024 n + sum of the n candidates' local indices, exact in fp32, sum j <= 496),
      // so the per-code work is FFMA.SAT + FFMA (+ half an FMNMX) instead of FFMA.SAT + FADD + FFMA, and n = floor(T / 1024)
      // is taken once per chunk. A fractional ind (a_j within 2^-60 of the threshold) leaves T, hence J, fractional: such rows
      // are flagged like the rows with S != 1.
      float S = 0.f, J = 0.f;
      uint32_t cmask = 0u;
      auto scan_chunk = [&](const uint32_t (&r)[32], int c) {
        float cm[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) cm[t] = fmaxf(__uint_as_float(r[t]), __uint_as_float(r[t + 4]));
#pragma unroll
        for (int q = 1; q < 4; ++q)
#pragma unroll
          for (int t = 0; t < 4; ++t) cm[t] = fmax3(cm[t], __uint_as_float(r[8 * q + t]), __uint_as_float(r[8 * q + 4 + t]));
        const float Mn = fmaxf(M1, fmax3(fmaxf(cm[0], cm[1]), cm[2], cm[3]));
        if (Mn - M1 > w) {
          S = 0.f;
          J = 0.f;
          cmask = 0u;
        }
        M1 = Mn;
        const float cc = -(M1 - w) * big;
        float tc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float ind = __saturatef(fmaf(__uint_as_float(r[j]), big, cc));
          tc[j & 3] = fmaf(ind, static_cast<float>(j + 1024), tc[j & 3]);
        }
        const float tl = (tc[0] + tc[1]) + (tc[2] + tc[3]);
        const float cnt = floorf(tl * 0.0009765625f);  // codes of this chunk inside the window
        S += cnt;
        J += fmaf(cnt, static_cast<float>(c * 32 - 1024), tl);  // + sum of their global indices
        if (tl > 0.f) cmask |= 1u << c;  // chunks that hold codes inside the window
      };
      if (VQ_CONV_WARPS == 4) {
#pragma unroll 1
        for (int c = 0; c < nchunks; c += 2) {  // two chunks per TMEM round trip (the round trip, not the bandwidth, costs)
          uint32_t ra[32], rb[32];
          tmem_ld_32x32b_x32(tacc + c * 32, ra);
          if (c + 1 < nchunks) tmem_ld_32x32b_x32(tacc + (c + 1) * 32, rb);
          tmem_ld_wait();
          scan_chunk(ra, c);
          if (c + 1 < nchunks) scan_chunk(rb, c + 1);
        }
      } else {
#pragma unroll 1
        for (int c = 0; c < nchunks; ++c) {  // (96 registers per thread: one chunk in flight)
          uint32_t ra[32];
          tmem_ld_32x32b_x32(tacc + c * 32, ra);
          tmem_ld_wait();
          scan_chunk(ra, c);
        }
      }
      const float thr = M1 - w;
      if (quad == 0) TRACE(9);
      // exactly one whole candidate: S == 1 and J an integer (a second code with a fractional ind would show up in J)
      const float Ssum = (J == rintf(J)) ? S : 2.f;
      int idx = static_cast<int>(J + 0.5f);
      // a row whose |z|^2 is +Inf / NaN has no finite distance: the oracle's strict '<' from +Inf keeps index 0. Its scores
      // are Inf / NaN mixtures that could fake S == 1, so such rows always take the exact pass (empty candidate masks -> 0).
      const bool nonfinite = !(zzr < INFINITY);
      const bool flagged = row_ok && (!(Ssum == 1.0f) || nonfinite) && window_scale > 0.f;  // (<= 0: profiling, no exact pass)
      if (!(Ssum == 1.0f) || nonfinite) idx = 0;
      uint32_t fl = __ballot_sync(0xffffffffu, flagged);
      uint32_t deferred = 0u;  // lanes whose row went to the deferred queue: their outputs are written by drain_deferred
      if (fl) {
        // ---- second look at the accumulator, only at the chunks that hold candidates of a flagged row: per-row candidate
        //      masks (a_j >= final max - w; the counts above were taken against the smaller running max: a superset) ----
        uint32_t want = flagged ? cmask : 0u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) want |= __shfl_xor_sync(0xffffffffu, want, o);
        uint32_t mask[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          mask[c] = 0u;
          if ((want >> c) & 1u) {
            uint32_t r[32];
            tmem_ld_32x32b_x32(tacc + c * 32, r);
            tmem_ld_wait();
            uint32_t m = 0u;
#pragma unroll
            for (int j = 0; j < 32; ++j) m |= (__uint_as_float(r[j]) >= thr ? 1u : 0u) << j;
            mask[c] = flagged ? m : 0u;
          }
        }
        // the accumulator is no longer needed: release it before the (latency-bound) exact chains
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_t_empty(base, grp));
        // queue the flagged rows for the end of the segment; only a full queue keeps them here
        {
          const int nfl = __popc(fl);
          uint32_t* qcount = reinterpret_cast<uint32_t*>(smem + OFF_DEFER);
          uint32_t pos = 0xffffffffu;
          if (lane == 0) {
            uint32_t old = *reinterpret_cast<volatile uint32_t*>(qcount);
            while (old + nfl <= DEFER_CAP) {
              const uint32_t seen = atomicCAS(qcount, old, old + nfl);
              if (seen == old) { pos = old; break; }
              old = seen;
            }
          }
          pos = __shfl_sync(0xffffffffu, pos, 0);
          if (pos != 0xffffffffu) {
            if (flagged) {
              uint8_t* ent = smem + OFF_DEFER + 16 + (pos + __popc(fl & ((1u << lane) - 1u))) * DEFER_ENTRY_BYTES;
              *reinterpret_cast<int64_t*>(ent) = grow;
#pragma unroll
              for (int c = 0; c < 8; ++c) reinterpret_cast<uint32_t*>(ent + 8)[c] = mask[c];
            }
            deferred = fl;
            if (flagged && out_recheck) atomicAdd(out_recheck, 1ull);
            fl = 0u;
          }
        }
        float* scratch = reinterpret_cast<float*>(smem + OFF_ZROW) + (warp - EPI_WARP0) * (D + 16);
        while (fl) {
          const int f = __ffs(fl) - 1;
          fl &= fl - 1u;
          const int64_t grow_f = __shfl_sync(0xffffffffu, grow, f);
          __syncwarp();
          if (D == 64) reinterpret_cast<float2*>(scratch)[lane] = reinterpret_cast<const float2*>(zsrc + grow_f * D)[lane];
          else reinterpret_cast<float4*>(scratch)[lane] = reinterpret_cast<const float4*>(zsrc + grow_f * D)[lane];
          if (lane == f) {
#pragma unroll
            for (int c = 0; c < 8; ++c) reinterpret_cast<uint32_t*>(scratch + D)[c] = mask[c];
          }
          __syncwarp();
          const int bi = exact_one(cbg, ee, scratch, lane);
          if (lane == f) idx = bi;
        }
        if (!deferred && flagged && out_recheck) atomicAdd(out_recheck, 1ull);
      } else {
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_t_empty(base, grp));  // accumulator free: the MMAs of tile it + 2 may start
      }
      if (quad == 0) TRACE(10);

      // ---- outputs: index, gathered code rows ----
      const bool mine = row_ok && !((deferred >> lane) & 1u);
      if (mine && out_idx) out_idx[grow] = idx;
      if (out_bdl && mine) {  // (B, D, L): for each k the warp writes 32 consecutive floats
        const float4* src = reinterpret_cast<const float4*>(cbg + idx * D);
        float* dst = out_bdl + (b * D) * L + l0 + row;
#pragma unroll
        for (int h = 0; h < D / 32; ++h) {
          float4 v[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = __ldg(src + h * 8 + i);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int k = h * 32 + i * 4;
            dst[(k + 0) * L] = v[i].x;
            dst[(k + 1) * L] = v[i].y;
            dst[(k + 2) * L] = v[i].z;
            dst[(k + 3) * L] = v[i].w;
          }
        }
      }
      if (out_rows) {  // (B, L, D): the warp copies 512 bytes of code rows per iteration (D / 4 lanes x float4 per row)
        constexpr int LPR = D / 4, RPI = 32 / LPR;  // lanes per row, rows per iteration
        const int wrows = min(32, nrows - quad * 32);
        const int sub = lane / LPR, lr = lane % LPR;
        for (int rr = 0; rr < wrows; rr += RPI) {
          const int r2 = rr + sub;
          const int ci = __shfl_sync(0xffffffffu, idx, r2 & 31);
          if (r2 < wrows && !((deferred >> r2) & 1u)) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(cbg + ci * D) + lr);
            reinterpret_cast<float4*>(out_rows + (b * L + l0 + quad * 32 + r2) * D)[lr] = v;
          }
        }
      }
      if (quad == 0) TRACE(11);
    }
    // both epilogue groups have pushed the last rows of this segment: decide the queued ones (the next segment_begin's
    // barrier orders this before the codebook slice and ee[] change)
    asm volatile("bar.sync 1, 256;" ::: "memory");
    drain_deferred(p, cx, cbg);
    tile = seg_end;
  }
}

template <bool TL>
__global__ void __launch_bounds__(NUM_THREADS, 1) vq_tc_kernel(const __grid_constant__ Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  Ctx cx;
  cx.base = (raw_addr + 1023u) & ~1023u;
  cx.smem = smem_raw + (cx.base - raw_addr);
  const uint32_t base = cx.base;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(cx.smem + OFF_MISC);
  const int tid = threadIdx.x, warp = tid >> 5;

  if (tid == 0) {
    for (int s = 0; s < STG_STAGES; ++s) { mbar_init(bar_stg_full(base, s), 1); mbar_init(bar_stg_empty(base, s), CONV_THREADS / 32); }
    for (int s = 0; s < A_STAGES; ++s) { mbar_init(bar_a_full(base, s), CONV_THREADS / 32); mbar_init(bar_a_empty(base, s), 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(bar_t_full(base, s), 1); mbar_init(bar_t_empty(base, s), 4); }
    fence_barrier_init();
  } else if (warp == MMA_WARP) {
    tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), 512);
  }
  // constant A column block of the 13th k-step: k = 0, 1, 2 -> 1.0 (one per bf16 term of -ee_j / 2), k = 3..15 -> 0
  for (int i = tid; i < TILE_ROWS * 2; i += NUM_THREADS) {
    const int row = i >> 1, kc = i & 1;
    const uint32_t o = static_cast<uint32_t>((row & 7) * 16 + (row >> 3) * AUG_SBO + kc * AUG_LBO);
    st_shared_v4(base + OFF_AUG_A + o, kc == 0 ? make_uint4(0x3F803F80u, 0x00003F80u, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u));
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  cx.tmem_base = *tmem_slot;
  const uint32_t num_tiles = static_cast<uint32_t>(TL ? *p.tile_count : p.num_tiles);
  cx.t_begin = static_cast<int>(static_cast<uint64_t>(blockIdx.x) * num_tiles / gridDim.x);
  cx.t_end = static_cast<int>(static_cast<uint64_t>(blockIdx.x + 1) * num_tiles / gridDim.x);

  if (warp >= CONV_WARP0) role_convert<TL>(p, cx);
  else if (warp == MMA_WARP) role_mma<TL>(p, cx);
  else if (warp == LOAD_WARP) role_load<TL>(p, cx);
  else role_epilogue<TL>(p, cx);

  tcgen05_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) tmem_dealloc(cx.tmem_base, 512);
}

// tiles != NULL: the caller's tile table (device count *tile_count, at most max_tiles) replaces the per-clip tiles
int launch(const float* z, const float* codebook, const int64_t* code_offset, int64_t B, int64_t L, int n_codes,
           int64_t* indices, float* zq_bdl, float* zq_rows, unsigned long long* recheck_rows, float* dbg_acc,
           const VqTile* tiles, const int* tile_count, int64_t max_tiles, cudaStream_t stream) {
  static bool attr = false;
  if (!attr) {
    FDM_CHECK_CUDA(cudaFuncSetAttribute(vq_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    FDM_CHECK_CUDA(cudaFuncSetAttribute(vq_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    attr = true;
  }
  Params p;
  p.z = z; p.codebook = codebook; p.code_offset = code_offset; p.B = B; p.L = L; p.n_codes = n_codes;
  p.indices = indices; p.zq_bdl = zq_bdl; p.zq_rows = zq_rows; p.recheck_rows = recheck_rows; p.dbg_acc = dbg_acc;
  FDM_CHECK_ARG(B * ceil_div64(L, TILE_ROWS) < (1ll << 31), "fdm_vq_quantize: too many rows for one launch");
  p.tiles_per_clip = static_cast<int>(ceil_div64(L, TILE_ROWS));
  p.num_tiles = static_cast<int>(B * p.tiles_per_clip);
  p.tiles = tiles;
  p.tile_count = tile_count;
  static float wscale = -1.f;
  static bool wscale_set = false;
  if (!wscale_set) {
    wscale_set = true;
    const char* e = getenv("FDM_B200_VQ_WINDOW");
    wscale = e ? static_cast<float>(atof(e)) : 1.f;
    if (wscale < 0.f) wscale = 0.f;
  }
  p.window_scale = wscale;
  static const int l2_ahead = [] { const char* e = getenv("FDM_B200_VQ_L2_AHEAD"); return e ? atoi(e) : L2_AHEAD; }();
  p.l2_ahead = l2_ahead;
  const int64_t sms = fdm_sm_count();
  const int64_t n_t = tiles ? max_tiles : p.num_tiles;
  const int grid = static_cast<int>(n_t < sms ? n_t : sms);
  if (tiles) vq_tc_kernel<true><<<grid, NUM_THREADS, SMEM_BYTES, stream>>>(p);
  else vq_tc_kernel<false><<<grid, NUM_THREADS, SMEM_BYTES, stream>>>(p);
  FDM_CHECK_LAUNCH();
  return 0;
}

}  // namespace VQ_NS
