// Tensor-map (TMA descriptor) helpers: host-side encoding through the driver entry point (the library links
// only the CUDA runtime) and the device-side cp.async.bulk.tensor wrappers (SASS: UTMALDG / UTMASTG).  sm_100a only.
#pragma once
#include <cuda.h>
#include <cudaTypedefs.h>
#include "bulk.cuh"

namespace dgod {

// cuTensorMapEncodeTiled, looked up once per process; nullptr when the driver does not offer it.
PFN_cuTensorMapEncodeTiled tensor_map_encoder();

// rank-2 map over 32-bit words: `rows` rows of `row_words` words (row pitch = row_words * 4 bytes, a multiple of 16),
// box = box_rows x row_words.  No swizzle, no interleave; out-of-range rows read as zero.
int encode_words_2d(CUtensorMap* map, const void* base, unsigned long long rows, unsigned row_words, unsigned box_rows);
// rank-2 fp32 map: `rows` rows of `cols` floats (cols * 4 a multiple of 16), box = box_rows x 32 floats (one 128-byte
// row per box row), 128-byte swizzle: the layout tcgen05.mma's K-major SWIZZLE_128B operand descriptors read.
// Out-of-range rows and columns read as zero.
int encode_f32_2d_sw128(CUtensorMap* map, const void* base, unsigned long long rows, unsigned long long cols, unsigned box_rows);

__device__ __forceinline__ void tmap_prefetch(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];\n" ::"l"(reinterpret_cast<unsigned long long>(map)) : "memory");
}
// global -> shared tile load, completion counted in bytes on an mbarrier
__device__ __forceinline__ void tmap_load_2d(void* smem_dst, const CUtensorMap* map, int c0, int c1, unsigned long long* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<unsigned long long>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
      : "memory");
}

}  // namespace dgod
