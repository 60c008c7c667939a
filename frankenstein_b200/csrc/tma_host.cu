#include "tma_host.cuh"

#include "common.cuh"

namespace fk {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* ptr = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(ptr);
  return fn;
}

int make_tmap_bf16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                   const uint32_t* box, CUtensorMapSwizzle swizzle) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return FK_ERR_DRIVER;
  cuuint64_t gdim[5], gstride[4];
  cuuint32_t bx[5], estr[5];
  for (int i = 0; i < rank; ++i) { gdim[i] = dims[i]; bx[i] = box[i]; estr[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) gstride[i] = strides_bytes[i];
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, static_cast<cuuint32_t>(rank), const_cast<void*>(base), gdim,
                   gstride, bx, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? FK_OK : FK_ERR_DRIVER;
}

int make_tmap_bf16_sw128(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  const uint64_t dims[2] = {cols, rows};
  const uint64_t strides[1] = {cols * 2};
  const uint32_t box[2] = {64, box_rows};
  return make_tmap_bf16(map, base, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

int make_tmap_bf16_2d(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
  const uint64_t dims[2] = {cols, rows};
  const uint64_t strides[1] = {ld * 2};
  const uint32_t box[2] = {64, box_rows};
  return make_tmap_bf16(map, base, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

int make_tmap_bf16_2d_sw64(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
  const uint64_t dims[2] = {cols, rows};
  const uint64_t strides[1] = {ld * 2};
  const uint32_t box[2] = {32, box_rows};
  return make_tmap_bf16(map, base, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B);
}

int make_tmap_bf16_chunks(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
  const uint64_t dims[3] = {64, rows, cols / 64};
  const uint64_t strides[2] = {ld * 2, 128};
  const uint32_t box[3] = {64, box_rows, 4};
  return make_tmap_bf16(map, base, 3, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

int make_tmap_heads_sw64(CUtensorMap* map, const void* base, int B, int S, int H, long long batch_stride,
                         long long token_stride, uint32_t box_rows) {
  const uint64_t dims[4] = {32, static_cast<uint64_t>(H), static_cast<uint64_t>(S), static_cast<uint64_t>(B)};
  const uint64_t strides[3] = {64, static_cast<uint64_t>(token_stride) * 2, static_cast<uint64_t>(batch_stride) * 2};
  const uint32_t box[4] = {32, 1, box_rows, 1};
  return make_tmap_bf16(map, base, 4, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B);
}

// bf16 [B][S][H][16] (strided tokens / trials): box = one head's 16 columns (32-byte rows) x box_rows tokens, 32-byte
// swizzle.  Coordinates: (0, head, token, batch).
int make_tmap_heads_sw32(CUtensorMap* map, const void* base, int B, int S, int H, long long batch_stride,
                         long long token_stride, uint32_t box_rows) {
  const uint64_t dims[4] = {16, static_cast<uint64_t>(H), static_cast<uint64_t>(S), static_cast<uint64_t>(B)};
  const uint64_t strides[3] = {32, static_cast<uint64_t>(token_stride) * 2, static_cast<uint64_t>(batch_stride) * 2};
  const uint32_t box[4] = {16, 1, box_rows, 1};
  return make_tmap_bf16(map, base, 4, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_32B);
}

// bf16 [B][S][H][64] (strided tokens / trials): box = one head's 64 columns (128-byte rows) x box_rows tokens, 128-byte
// swizzle.  Coordinates: (0, head, token, batch).
int make_tmap_heads_sw128(CUtensorMap* map, const void* base, int B, int S, int H, long long batch_stride,
                          long long token_stride, uint32_t box_rows) {
  const uint64_t dims[4] = {64, static_cast<uint64_t>(H), static_cast<uint64_t>(S), static_cast<uint64_t>(B)};
  const uint64_t strides[3] = {128, static_cast<uint64_t>(token_stride) * 2, static_cast<uint64_t>(batch_stride) * 2};
  const uint32_t box[4] = {64, 1, box_rows, 1};
  return make_tmap_bf16(map, base, 4, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

// [B][H][S][16] bf16 rows of 32 bytes (the statistics operand of the attention backward): box = box_rows x 16 elements of
// one (trial, head), 32-byte swizzle
int make_tmap_aug_sw32(CUtensorMap* map, const void* base, int B, int S, int H, uint32_t box_rows) {
  const uint64_t dims[4] = {16, static_cast<uint64_t>(S), static_cast<uint64_t>(H), static_cast<uint64_t>(B)};
  const uint64_t strides[3] = {32, static_cast<uint64_t>(S) * 32, static_cast<uint64_t>(S) * H * 32};
  const uint32_t box[4] = {16, box_rows, 1, 1};
  return make_tmap_bf16(map, base, 4, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_32B);
}

}  // namespace fk
