// TMA helpers shared by the GEMM and attention kernels: tensor-map encoding through the driver entry point (no libcuda link
// dependency), and the device-side bulk and tensor (cp.async.bulk[.tensor]) stores and loads.
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

// Encodes a tiled tensor map of `rank` dimensions (element strides 1, no interleave, out-of-bounds elements read as zero):
// dims[0] is the contiguous one, byte_strides[i] is the stride of dims[i + 1].  `what` names the layout in the error
// message, e.g. "(4-D heads)" ("" for none).
inline int encode_tiled(CUtensorMap* tm, CUtensorMapDataType dtype, cuuint32_t rank, const void* base, const cuuint64_t* dims,
                        const cuuint64_t* byte_strides, const cuuint32_t* box, CUtensorMapSwizzle swz, CUtensorMapL2promotion promo,
                        const char* what) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(SPOTV2_ERR_NO_DEVICE, "cuTensorMapEncodeTiled is not available from the driver");
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = fn(tm, dtype, rank, const_cast<void*>(base), dims, byte_strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz, promo,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(SPOTV2_ERR_CUDA, "cuTensorMapEncodeTiled%s%s failed with CUresult %d", *what ? " " : "", what, (int)r);
  return SPOTV2_OK;
}

// 2-D tensor [rows, cols] (cols contiguous, row pitch ld elements), box = box_cols x box_rows, given
// shared-memory swizzle, out-of-bounds elements read as zero.
inline int make_tmap_typed(CUtensorMap* tm, const void* base, CUtensorMapDataType dtype, size_t elem_bytes, uint64_t rows,
                           uint64_t cols, uint64_t ld, uint32_t box_cols, uint32_t box_rows, CUtensorMapSwizzle swz,
                           CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_256B) {
  const cuuint64_t dims[2] = {cols, rows};
  const cuuint64_t strides[1] = {ld * elem_bytes};
  const cuuint32_t box[2] = {box_cols, box_rows};
  return encode_tiled(tm, dtype, 2, base, dims, strides, box, swz, promo, "");
}
inline int make_tmap(CUtensorMap* tm, const float* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_cols,
                     uint32_t box_rows, CUtensorMapSwizzle swz, CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_256B) {
  return make_tmap_typed(tm, base, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, sizeof(float), rows, cols, ld, box_cols, box_rows, swz, promo);
}
// fp32 tensor [planes][rows][ld >= cols] with a (box_cols x box_rows x 1) box: the output side of the split-K GEMM
inline int make_tmap3(CUtensorMap* tm, const float* base, uint64_t planes, uint64_t plane_stride, uint64_t rows, uint64_t cols,
                      uint64_t ld, uint32_t box_cols, uint32_t box_rows, CUtensorMapSwizzle swz) {
  const cuuint64_t dims[3] = {cols, rows, planes};
  const cuuint64_t strides[2] = {ld * sizeof(float), plane_stride * sizeof(float)};
  const cuuint32_t box[3] = {box_cols, box_rows, 1};
  return encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, base, dims, strides, box, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, "(3-D)");
}
// fp32 tensor (d0, d1, d2) with strides in elements and a (b0 x b1 x 1) box, no L2 promotion: the attention backward's
// P, dout and dout^T (attn_bwd3.cu)
inline int make_tmap3_f32(CUtensorMap* tm, const float* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_elems,
                          uint64_t stride2_elems, uint32_t b0, uint32_t b1, CUtensorMapSwizzle swz) {
  const cuuint64_t dims[3] = {d0, d1, d2};
  const cuuint64_t strides[2] = {stride1_elems * sizeof(float), stride2_elems * sizeof(float)};
  const cuuint32_t box[3] = {b0, b1, 1};
  return encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, base, dims, strides, box, swz, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                      "(attention backward, 3-D)");
}
// fp16 tensor [planes][rows][ld >= cols] with a (box_cols x box_rows x 1) box: the hi | lo planes of an operand pair
inline int make_tmap3_f16(CUtensorMap* tm, const void* base, uint64_t planes, uint64_t plane_stride, uint64_t rows, uint64_t cols,
                          uint64_t ld, uint32_t box_cols, uint32_t box_rows, CUtensorMapSwizzle swz) {
  const cuuint64_t dims[3] = {cols, rows, planes};
  const cuuint64_t strides[2] = {ld * 2, plane_stride * 2};
  const cuuint32_t box[3] = {box_cols, box_rows, 1};
  return encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, base, dims, strides, box, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      "(3-D fp16)");
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
  const cuuint64_t dims[4] = {cols, rows, grp, planes};
  const cuuint64_t strides[3] = {ld * 2, 64, (planes > 1 ? plane_stride : 32) * 2};
  const cuuint32_t box[4] = {32, 32, grp, planes};
  return encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B, promo,
                      "(4-D tile groups)");
}
// fp16 operand pair planes [planes][rows][ld] seen head by head: (column inside the head [cols_per_head: columns past it read
// as zero, so a tile never picks up the next head], row, head [stride head_pitch elements, % 8 == 0], plane); box (32, 32,
// box_heads, planes) lands as [plane][head][row][64 B], every 32 x 32 tile in the 2-D 64B-swizzled layout.
inline int make_tmap_heads_f16(CUtensorMap* tm, const void* base, uint64_t plane_stride, uint32_t planes, uint64_t rows,
                               uint64_t cols_per_head, uint64_t head_pitch, uint64_t heads, uint64_t ld, uint32_t box_heads,
                               CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_NONE, uint32_t box_rows = 32) {
  const cuuint64_t dims[4] = {cols_per_head, rows, heads, planes};
  const cuuint64_t strides[3] = {ld * 2, (heads > 1 ? head_pitch : 8) * 2, (planes > 1 ? plane_stride : 8) * 2};
  const cuuint32_t box[4] = {32, box_rows, box_heads, planes};
  return encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B, promo,
                      "(4-D heads)");
}

// ---- bulk stores (shared -> global, bulk async group of the issuing thread) ---------------------------------------------
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// waits until at most N of this thread's committed groups are still reading shared memory
template <int N = 0>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
// waits until at most N of this thread's committed groups have not completed (their global writes are done)
template <int N = 0>
__device__ __forceinline__ void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }
// 1-D bulk store of `bytes` (% 16 == 0) from shared memory, committed as a group of its own
__device__ __forceinline__ void bulk_s2g_commit(void* gmem_dst, uint32_t smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_src), "r"(bytes) : "memory");
  bulk_commit();
}
// tensor stores; the caller commits
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* tm, uint32_t smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(tm), "r"(smem_src), "r"(c0),
               "r"(c1), "r"(c2)
               : "memory");
}
// this one commits its store as a group of its own
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* tm, uint32_t smem_src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(tm), "r"(smem_src), "r"(c0),
               "r"(c1), "r"(c2), "r"(c3)
               : "memory");
  bulk_commit();
}

// ---- tensor loads ---------------------------------------------------------------------------------------------------------
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
__device__ __forceinline__ void tma_load_3d_hint(uint32_t smem_dst, const CUtensorMap* tm, int c0, int c1, int c2, uint32_t bar,
                                                 uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], "
      "[%2], %6;" ::"r"(smem_dst),
      "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "l"(hint)
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
