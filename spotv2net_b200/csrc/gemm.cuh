// GEMM back ends of the projection path.
#pragma once
#include "common.cuh"

namespace spotv2 {

// Exact-fp32 CUDA-core GEMM: C[M,N] = sum_k A(m,k) B(n,k).  a_kc / b_kc: the operand is stored
// K-contiguous ([rows, K]) rather than row-contiguous-in-M|N ([K, rows]).
int sgemm_simt(bool a_kc, bool b_kc, int M, int N, int K, const float* A, int lda, const float* B,
               int ldb, float* C, int ldc, int splits, void* ws, size_t ws_bytes, cudaStream_t st);

// Batched exact-fp32 GEMM (same tiles as sgemm_simt) used by the large-universe attention path.
// C_z[M,N] = scale * sum_seg sum_k A_z,seg(m,k) B_z,seg(n,k) + bias; z = zo * inner + zi.
struct BGemm {
  int M, N, K;
  const float* A;
  const float* B;
  float* C;
  int lda, ldb, ldc;
  int inner;                               // batch index z -> (z / inner, z % inner)
  long long a_o, a_i, b_o, b_i, c_o, c_i;  // element offsets per outer / inner batch index
  int segs;                                // contraction segments (heads) summed into one C
  long long a_s, b_s;                      // element offsets per segment
  float scale;
  const float* bias;                       // null or [inner * bias_i + N]
  long long bias_i;
  int vecA, vecB;                          // filled by bgemm_simt
  int tensor_cores;                        // 1: mma.sync TF32 with the 3-product split (fp32-accurate); 0: FFMA2
};
int bgemm_simt(bool a_kc, bool b_kc, BGemm g, int batches, cudaStream_t st);

// CTA pairs of the fp16-pair GEMM kernel resident at once on the current device (sm_count / 2 without one).
int gemm3x_f16_resident_pairs();

// Split-K factor used for the weight-gradient GEMM (contraction over all B*N node rows): keeps
// every fp32 accumulation chain short (<= ~8K terms) and fills the machine.  pair_tiles: the product runs on 256 x 256
// pair tiles over the resident CTA pairs (the 3-product class); false: 128 x 256 tiles over the SMs (half precision).
inline int weight_grad_splits(int rows, int m, int n, bool pair_tiles = true) {
  int base = (rows + 8191) / 8192;
  if (base < 1) base = 1;
  if (base > 32) base = 32;
  if (base == 1) return 1;
  // among base .. 1.25 base, the count whose (tile, split) work items fill the resident slots' last wave best
  // (config A on 74 pairs: 60 pair tiles x 15 splits = 12.16 waves, x 16 = 12.97)
  const int tile_m = pair_tiles ? 256 : 128;
  const int tiles = ((m + tile_m - 1) / tile_m) * ((n + 255) / 256);
  const int pairs = pair_tiles ? gemm3x_f16_resident_pairs() : sm_count();
  int best = base;
  double best_eff = 0.0;
  for (int s = base; s <= base + base / 4 + 1 && s <= 32; ++s) {
    const int items = tiles * s;
    const double eff = (double)items / (double)(((items + pairs - 1) / pairs) * pairs);
    if (eff > best_eff + 1e-9) { best = s; best_eff = eff; }
  }
  return best;
}

// fp32-accurate tensor-core GEMM (tcgen05, 3xTF32, chunked accumulation) on operands pre-split into
// tf32 hi/lo arrays.  bn = 128 | 256 (tile N); kb_per_chunk = k-blocks of 32 per TMEM accumulation chain.
bool tc_gemm_supported(bool a_kc, bool b_kc, int M, int N, int K, const float* A_hi, int lda, const float* B_hi, int ldb);
int split_tf32(const float* src, float* hi, float* lo, size_t n, cudaStream_t st);
int gemm3x_tf32(bool a_kc, bool b_kc, int M, int N, int K, const float* A_hi, const float* A_lo, int lda,
                const float* B_hi, const float* B_lo, int ldb, float* C, int ldc, int splits, int bn,
                int kb_per_chunk, void* ws, size_t ws_bytes, cudaStream_t st);

// ---- fp16-pair ("3xFP16") tensor-core GEMM: gemm_f16.cu ----------------------------------------------
// An operand pre-split into scaled fp16 hi/lo arrays.  inv -> 2 floats on the device: the inverse scales of
// the operand's two groups (M|N index < split_at / >= split_at); null = unscaled.
struct F16Operand {
  const void* hi;
  const void* lo;
  int ld;               // elements, % 8 == 0
  const float* inv;
  int split_at;
};
// Output of gemm3x_f16 as an fp16 operand pair instead of fp32 (p_format 1): C * scale[col >= B.split_at] is split into
// hi (and lo, unless null) planes [M, ld] by the epilogue and leaves through TMA stores; scale -> 2 floats on the device.
struct PairOut {
  void* hi;
  void* lo;             // null: hi plane only (half-precision class)
  int ld;               // elements, % 8 == 0
  const float* scale;
  float* tail32;        // optional: the columns >= B.split_at also leave in fp32, unscaled, as [M, tail_ld] (the attention
  int tail_ld;          // logit terms s | d: their LeakyReLU kinks must not depend on the pair's rounding)
};
constexpr int kScaleBlockFloats = 8;   // [0,1] amax bits, [2,3] inverse scales, [4,5] scales
inline int ld16_of(int cols) { return (cols + 15) / 16 * 16; }   // rows of fp16 operands start on 32-byte sectors
// blk[0] <- bit pattern of max |src| (blk is zeroed first)
int amax_flat(const float* src, size_t n, float* blk, cudaStream_t st);
// src [rows, cols] (pitch ld) -> hi/lo fp16 [rows, ld16]; two scale groups along split_dim (0 rows, 1 cols) at
// split_at; optional exact pre-multiplier pre2[row >= pre_split] (power of two).  Fills blk.
int split_f16(const float* src, int rows, int cols, size_t ld, int split_dim, int split_at, const float* pre2,
              int pre_split, void* hi, void* lo, size_t ld16, float* blk, cudaStream_t st);
int gemm3x_f16(bool a_kc, bool b_kc, int M, int N, int K, const F16Operand& A, const F16Operand& B, float* C, int ldc,
               int splits, int bn, int kb_per_chunk, void* ws, size_t ws_bytes, cudaStream_t st,
               float* amax_out = nullptr, int amax_cols = 0,    // amax_out[0] <- bits of max |C[:, :amax_cols]|
               bool single = false,    // true: one fp16 product (A_hi * B_hi) - the half-precision class of gemm_algo 3
               const PairOut* pair = nullptr);   // non-null: C is ignored, the result leaves as an fp16 pair (splits == 1)
// Scale block of a pair output C = x . W^T from the bound |C| <= max|x| * max_row ||W||_1 (x_blk[0] = bits of max|x|);
// two groups: rows of W below / at-or-above split_at.
int pair_out_scale(const float* W, int rows, int cols, int split_at, const float* x_blk, float* blk, cudaStream_t st);
// W's own operand pair and the pair-output scale block in two launches (statistics, split)
int w_pair_and_out_scale(const float* W, int rows, int cols, int split_at, void* hi, void* lo, size_t ld16, float* wblk,
                         const float* x_blk, float* out_blk, cudaStream_t st);
// blk[0] <- bits of max |src[r, c]| over a [rows, cols] matrix with row pitch ld (blk is zeroed first)
int amax_2d(const float* src, int rows, int cols, size_t ld, float* blk, cudaStream_t st);

}  // namespace spotv2
