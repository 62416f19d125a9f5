// fdm_vq_quantize, tensor-core path: the kernel body (vq_tc_impl.cuh) instantiated for the two latent widths of the
// reference's EVQ-VAEs - D = 64 (VOCASET, MEAD: models/utils/config.py:5-42) and D = 128 (BIWI: config.py:44-60).
#include "tc_common.cuh"
#include <stdlib.h>

// Converter warps: four at D = 64 (the accumulator-slot cycle MMA -> scan sets the pace there: eight change nothing), eight at
// D = 128 (twice the conversion work per tile: 1.22 M rows 0.31 -> 0.27 ms indices-only, 0.49 -> 0.46 ms with z_q).
#define VQ_D 64
#define VQ_NS vq_tc64
#define VQ_CONV_WARPS 4
#include "vq_tc_impl.cuh"
#undef VQ_D
#undef VQ_NS
#undef VQ_CONV_WARPS
#undef TRACE

#define VQ_D 128
#define VQ_NS vq_tc128
#define VQ_CONV_WARPS 8
#include "vq_tc_impl.cuh"
#undef VQ_D
#undef VQ_NS
#undef VQ_CONV_WARPS
#undef TRACE

int fdm_vq_tc_launch(const float* z, const float* codebook, const int64_t* code_offset, int64_t B, int64_t L, int64_t D,
                     int n_codes, int64_t* indices, float* zq_bdl, float* zq_rows, unsigned long long* recheck_rows,
                     float* dbg_acc, const VqTile* tiles, const int* tile_count, int64_t max_tiles, cudaStream_t stream) {
  if (D == 64)
    return vq_tc64::launch(z, codebook, code_offset, B, L, n_codes, indices, zq_bdl, zq_rows, recheck_rows, dbg_acc, tiles,
                           tile_count, max_tiles, stream);
  if (D == 128)
    return vq_tc128::launch(z, codebook, code_offset, B, L, n_codes, indices, zq_bdl, zq_rows, recheck_rows, dbg_acc, tiles,
                            tile_count, max_tiles, stream);
  FDM_CHECK_ARG(false, "fdm_vq_quantize: the tensor-core path needs D = 64 or 128 (got %lld)", (long long)D);
  return 0;
}
