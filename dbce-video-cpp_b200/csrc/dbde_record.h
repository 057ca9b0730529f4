// The frame record's layout, for the kernels and the host code alike.  The reference's record (dbde_util.cpp:141-191)
// with a minimum plane of mb bytes per tile -- 1: the reference's 8-bit records, 2: DBDE16:
//   I32 2 | U64 index | F64 0.0 | I32 wh | U8 depth[wh] | I32 mb*wh | min[wh] (mb bytes, little-endian) | I32 n64 | U64 words[n64]
// Byte offsets from the record's start for a frame of wh tiles.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

namespace dbde {

constexpr size_t kRecIndex = 4;            // U64 index
constexpr size_t kRecDepthCount = 20;      // I32 wh
constexpr size_t kRecDepth = 24;           // U8 depth[wh]
__host__ __device__ constexpr size_t rec_min_count(size_t wh) { return 24 + wh; }                   // I32 mb*wh
__host__ __device__ constexpr size_t rec_min(size_t wh) { return 28 + wh; }                         // min[wh]
__host__ __device__ constexpr size_t rec_n64(size_t wh, size_t mb) { return 28 + (1 + mb) * wh; }  // I32 n64
__host__ __device__ constexpr size_t rec_fixed(size_t wh, size_t mb) { return 32 + (1 + mb) * wh; } // U64 words[n64]
// the largest record: every tile at the full depth of 8 * mb bits, i.e. 8 * mb U64 words
__host__ __device__ constexpr size_t rec_bound(size_t wh, size_t mb) { return rec_fixed(wh, mb) + 64 * mb * wh; }

}  // namespace dbde
