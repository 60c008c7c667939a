// Host-side construction of TMA tensor maps (cuTensorMapEncodeTiled fetched through the runtime's driver
// entry point, so the library does not link libcuda).
#pragma once
#include <cuda.h>
#include <stdint.h>

namespace fk {

// Generic bf16 tiled map.  dims/box are innermost-first; strides_bytes has rank-1 entries (dims 1..rank-1).
int make_tmap_bf16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                   const uint32_t* box, CUtensorMapSwizzle swizzle);

// bf16 row-major [rows, cols] matrix, box = 64 columns x box_rows rows, 128-byte swizzle.
int make_tmap_bf16_sw128(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows);

// bf16 row-major [rows, cols] with leading dimension ld (elements): box = 64 columns x box_rows rows, 128-byte swizzle;
// out-of-range rows / columns are filled with zeros.
int make_tmap_bf16_2d(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows);

// Same with 32-column boxes (64-byte rows) and the 64-byte swizzle.
int make_tmap_bf16_2d_sw64(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows);

// The same matrix as an MN-major operand source: dims (64 columns of a chunk, rows, chunk index), box = 64 x 64 rows x 4
// chunks -> shared memory [chunk][row][64 elements] (8 KB per chunk), 128-byte swizzle.  cols % 64 == 0.
int make_tmap_bf16_chunks(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows);

// bf16 [B][S][H][32] with token / batch strides (elements): box = one head's 32 columns x box_rows tokens,
// 64-byte swizzle.  Coordinates: (0, head, token, batch).
int make_tmap_aug_sw32(CUtensorMap* map, const void* base, int B, int S, int H, uint32_t box_rows);
int make_tmap_heads_sw64(CUtensorMap* map, const void* base, int B, int S, int H, long long batch_stride,
                         long long token_stride, uint32_t box_rows);
// Same for bf16 [B][S][H][64]: box = one head's 64 columns (128-byte rows) x box_rows tokens, 128-byte swizzle.
int make_tmap_heads_sw128(CUtensorMap* map, const void* base, int B, int S, int H, long long batch_stride,
                          long long token_stride, uint32_t box_rows);
// Same for bf16 [B][S][H][16]: box = one head's 16 columns (32-byte rows) x box_rows tokens, 32-byte swizzle.
int make_tmap_heads_sw32(CUtensorMap* map, const void* base, int B, int S, int H, long long batch_stride,
                         long long token_stride, uint32_t box_rows);

}  // namespace fk
