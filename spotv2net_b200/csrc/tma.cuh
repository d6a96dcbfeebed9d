// TMA (cp.async.bulk.tensor) helpers shared by the GEMM and attention kernels: tensor-map encoding through
// the driver entry point (no libcuda link dependency) and the device-side load wrapper.
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace spotv2 {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* sym = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(sym);
  return fn;
}

inline bool tma_available() { return encode_fn() != nullptr; }

// 2-D tensor [rows, cols] (cols contiguous, row pitch ld elements), box = box_cols x box_rows, given
// shared-memory swizzle, out-of-bounds elements read as zero.
inline int make_tmap_typed(CUtensorMap* tm, const void* base, CUtensorMapDataType dtype, size_t elem_bytes, uint64_t rows,
                           uint64_t cols, uint64_t ld, uint32_t box_cols, uint32_t box_rows, CUtensorMapSwizzle swz,
                           CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_256B) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(SPOTV2_ERR_NO_DEVICE, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * elem_bytes};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(tm, dtype, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                  promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(SPOTV2_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return SPOTV2_OK;
}
inline int make_tmap(CUtensorMap* tm, const float* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_cols,
                     uint32_t box_rows, CUtensorMapSwizzle swz, CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_256B) {
  return make_tmap_typed(tm, base, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, sizeof(float), rows, cols, ld, box_cols, box_rows, swz, promo);
}
// fp32 tensor [planes][rows][ld >= cols] with a (box_cols x box_rows x 1) box: the output side of the split-K GEMM
inline int make_tmap3(CUtensorMap* tm, const float* base, uint64_t planes, uint64_t plane_stride, uint64_t rows, uint64_t cols,
                      uint64_t ld, uint32_t box_cols, uint32_t box_rows, CUtensorMapSwizzle swz) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(SPOTV2_ERR_NO_DEVICE, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[3] = {cols, rows, planes};
  cuuint64_t strides[2] = {ld * sizeof(float), plane_stride * sizeof(float)};
  cuuint32_t box[3] = {box_cols, box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(SPOTV2_ERR_CUDA, "cuTensorMapEncodeTiled (3-D) failed with CUresult %d", (int)r);
  return SPOTV2_OK;
}
// fp16 tensor [planes][rows][ld >= cols] with a (box_cols x box_rows x 1) box: the hi | lo planes of an operand pair
inline int make_tmap3_f16(CUtensorMap* tm, const void* base, uint64_t planes, uint64_t plane_stride, uint64_t rows, uint64_t cols,
                          uint64_t ld, uint32_t box_cols, uint32_t box_rows, CUtensorMapSwizzle swz) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(SPOTV2_ERR_NO_DEVICE, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[3] = {cols, rows, planes};
  cuuint64_t strides[2] = {ld * 2, plane_stride * 2};
  cuuint32_t box[3] = {box_cols, box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(SPOTV2_ERR_CUDA, "cuTensorMapEncodeTiled (3-D fp16) failed with CUresult %d", (int)r);
  return SPOTV2_OK;
}
inline int make_tmap_f16(CUtensorMap* tm, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_cols,
                         uint32_t box_rows, CUtensorMapSwizzle swz, CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_256B) {
  return make_tmap_typed(tm, base, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, rows, cols, ld, box_cols, box_rows, swz, promo);
}

// Groups of `grp` adjacent 32-column tiles of an fp16 operand pair in ONE load: the planes [planes][rows][ld] are viewed as
// the 4-D tensor (column, row, tile, plane) with the tile dimension overlapping the column dimension (stride 32 elements),
// so that a box (32, 32, grp, planes) at (c0, r0, 0, 0) lands in shared memory as [plane][tile][row][64 B] - `grp` tiles of
// the hi plane, each in the 2-D 64B-swizzled layout, then the lo plane's.  The caller guarantees c0 + 32 * grp <= ld
// (the box never leaves the last row's pitch).
inline int make_tmap_tile_groups_f16(CUtensorMap* tm, const void* base, uint64_t plane_stride, uint32_t planes, uint64_t rows, uint64_t cols,
                                     uint64_t ld, uint32_t grp, CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_256B) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(SPOTV2_ERR_NO_DEVICE, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[4] = {cols, rows, grp, planes};
  cuuint64_t strides[3] = {ld * 2, 64, (planes > 1 ? plane_stride : 32) * 2};
  cuuint32_t box[4] = {32, 32, grp, planes};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(SPOTV2_ERR_CUDA, "cuTensorMapEncodeTiled (4-D tile groups) failed with CUresult %d", (int)r);
  return SPOTV2_OK;
}
// fp16 operand pair planes [planes][rows][ld] seen head by head: (column inside the head [cols_per_head: columns past it read
// as zero, so a tile never picks up the next head], row, head [stride head_pitch elements, % 8 == 0], plane); box (32, 32,
// box_heads, planes) lands as [plane][head][row][64 B], every 32 x 32 tile in the 2-D 64B-swizzled layout.
inline int make_tmap_heads_f16(CUtensorMap* tm, const void* base, uint64_t plane_stride, uint32_t planes, uint64_t rows,
                               uint64_t cols_per_head, uint64_t head_pitch, uint64_t heads, uint64_t ld, uint32_t box_heads,
                               CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_NONE, uint32_t box_rows = 32) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(SPOTV2_ERR_NO_DEVICE, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[4] = {cols_per_head, rows, heads, planes};
  cuuint64_t strides[3] = {ld * 2, (heads > 1 ? head_pitch : 8) * 2, (planes > 1 ? plane_stride : 8) * 2};
  cuuint32_t box[4] = {32, box_rows, box_heads, planes};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(SPOTV2_ERR_CUDA, "cuTensorMapEncodeTiled (4-D heads) failed with CUresult %d", (int)r);
  return SPOTV2_OK;
}
// shared -> global tensor store (bulk async group of the issuing thread)
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* tm, uint32_t smem_src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(tm), "r"(smem_src), "r"(c0),
               "r"(c1), "r"(c2), "r"(c3)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* tm, int c0, int c1, int c2, int c3, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_hint(void* smem_dst, const CUtensorMap* tm, int c0, int c1, int c2, int c3, uint64_t* bar,
                                                 uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5, %6}], "
      "[%2], %7;" ::"r"(smem_u32(smem_dst)),
      "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "l"(hint)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tm, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// pair form: the bytes land in this CTA's shared memory and complete on an mbarrier of either CTA of the pair
// (bar_cluster: a shared::cluster address, mapa_shared)
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* tm, int c0, int c1, uint32_t bar_cluster) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(tm), "r"(bar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_hint(void* smem_dst, const CUtensorMap* tm, int c0, int c1, uint64_t* bar,
                                                 uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], "
      "[%2], %5;" ::"r"(smem_u32(smem_dst)),
      "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "l"(hint)
      : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tm) : "memory");
}

}  // namespace spotv2
