// Projection entry points: lin_src forward and its two backward products
// ([PyG] nn/dense/linear.py F.linear inside gat_conv.py; /root/reference/utils/models.py:146).
//
// gemm_algo: 0 | 2 = tensor cores (tcgen05, fp16 operand pairs, gemm_f16.cu), 1 = exact-fp32 CUDA-core GEMM
// (gemm_simt.cu, the parity yardstick).  Both back ends are hand-written kernels of this library.
// Operand preparation for the tensor-core path (power-of-two scaled fp16 hi/lo pairs) happens here unless
// the caller passes pairs it made earlier: x is prepared once per step and feeds both proj_fwd and
// proj_bwd_weight; the attention backward emits dP_aug directly as pairs.
#include "attn_bwd.cuh"
#include "gemm.cuh"

using namespace spotv2;

namespace {

constexpr int kNone = 0x7fffffff;

struct ProjShape {
  int rows, n_aug, HC, F, ldp, ldf16, ldp16;
};

ProjShape shape_of(const spotv2_gat_desc* d) {       // HC: first row / column of the s|d group (head pitch padded in p_format 1)
  const int n_aug = n_aug_of(d);
  return {d->B * d->N, n_aug, d->H * head_pitch_of(d), d->F, d->ldp, ld16_of(d->F), ld16_of(n_aug)};
}

bool use_tc(const spotv2_gat_desc* d) { return d->gemm_algo != 1; }
// gemm_algo 3: half-precision class (BASELINE config C's "bf16" variant): the same tcgen05 kernel issues only the
// A_hi * B_hi product of the scaled fp16 operands (11-bit significands, fp32 accumulate): a third of the tensor work.
bool single_product(const spotv2_gat_desc* d) { return d->gemm_algo == 3; }

// Carves the caller's workspace in 256-byte units.  With a null base it only counts (`used`): the workspace query runs the
// products' own carving code that way.
struct Carver {
  unsigned char* p;
  size_t left;
  size_t used = 0;
  void* take(size_t bytes) {
    bytes = round_up(bytes, 256);
    used += bytes;
    if (!p || bytes > left) return nullptr;
    void* r = p;
    p += bytes;
    left -= bytes;
    return r;
  }
};

// Every tensor-core product carves its two scale blocks first.  The query reserves 1 KB for them, and adds 256 B to the
// attention backward's own size: slack it has always given.
constexpr size_t kBlocksBytes = 2 * kScaleBlockFloats * sizeof(float), kBlocksReserve = 1024, kAttnBwdReserve = 256;

// A GEMM operand as an fp16 pair: the caller's (hi, lo and scale block all given), or two planes [rows, ld16] taken from the
// workspace, which split() fills from the fp32 tensor.
struct OperandPair {
  void* hi;
  void* lo;
  const float* scale;
  bool own;
  bool ok() const { return hi && lo; }
  int split(const float* src, int rows, int cols, size_t ld, int split_dim, int split_at, int ld16, float* blk, cudaStream_t st) {
    if (!own) return SPOTV2_OK;
    scale = blk;
    return split_f16(src, rows, cols, ld, split_dim, split_at, nullptr, 0, hi, lo, ld16, blk, st);
  }
};

OperandPair operand_pair(Carver& c, size_t rows, int ld16, const void* hi = nullptr, const void* lo = nullptr,
                         const float* scale = nullptr) {
  if (hi && lo && scale) return {const_cast<void*>(hi), const_cast<void*>(lo), scale, false};
  void* h = c.take(rows * ld16 * 2);
  void* l = c.take(rows * ld16 * 2);
  return {h, l, nullptr, true};
}

}  // namespace

extern "C" int32_t spotv2_gat_ld16(int32_t cols) { return ld16_of(cols); }
extern "C" int32_t spotv2_diag_weight_grad_splits(int32_t rows, int32_t m, int32_t n) { return weight_grad_splits(rows, m, n); }

extern "C" int spotv2_gat_workspace_bytes(const spotv2_gat_desc* d, size_t* proj_fwd,
                                          size_t* attn_bwd, size_t* proj_bwd) {
  if (int rc = check_desc(d)) return rc;
  const ProjShape s = shape_of(d);
  // The products' pairs, counted (proj_fwd_pair takes less than proj_fwd).  proj_bwd serves both backward products: the dP
  // pair, dW's x pair and split-K partials, and dX's W_aug pair.
  Carver f{nullptr, 0}, b{nullptr, 0};
  if (use_tc(d)) {
    operand_pair(f, s.rows, s.ldf16);
    operand_pair(f, s.n_aug, s.ldf16);
    operand_pair(b, s.rows, s.ldp16);
    operand_pair(b, s.rows, s.ldf16);
    operand_pair(b, s.n_aug, s.ldf16);
  }
  const int splits = weight_grad_splits(s.rows, s.n_aug, s.F, !single_product(d));
  b.take((size_t)splits * s.n_aug * s.F * sizeof(float));
  if (proj_fwd) *proj_fwd = kBlocksReserve + f.used;
  if (attn_bwd) *attn_bwd = attn_bwd_ws_bytes(d) + kAttnBwdReserve;
  if (proj_bwd) *proj_bwd = kBlocksReserve + b.used;
  return SPOTV2_OK;
}

extern "C" int spotv2_gat_attn_fwd_workspace_bytes(const spotv2_gat_desc* d, size_t* attn_fwd) {
  if (int rc = check_desc(d)) return rc;
  SPOTV2_REQUIRE(attn_fwd, "attn_fwd_workspace_bytes: null pointer");
  *attn_fwd = attn_large_fwd_ws_bytes(d);
  return SPOTV2_OK;
}

extern "C" int spotv2_gat_edge_terms_bytes(const spotv2_gat_desc* d, size_t* bytes) {
  if (int rc = check_desc(d)) return rc;
  SPOTV2_REQUIRE(bytes, "edge_terms_bytes: null pointer");
  const size_t per_graph = (size_t)d->H * d->N * (d->N > 32 ? (size_t)d->N : (size_t)kEdgeTermNS);
  *bytes = d->Fe > 0 ? (size_t)d->B * per_graph * sizeof(float) : 0;
  return SPOTV2_OK;
}

extern "C" int spotv2_gat_uses_tensor_cores(const spotv2_gat_desc* d) {
  if (check_desc(d)) return 0;
  return use_tc(d) ? 1 : 0;
}

extern "C" int spotv2_split_f16(const float* src, int32_t rows, int32_t cols, int32_t ld, int32_t split_dim,
                                int32_t split_at, void* hi, void* lo, int32_t ld16, float* scale_block, void* stream) {
  SPOTV2_REQUIRE(src && hi && lo && scale_block && rows > 0 && cols > 0, "split_f16: null pointer or empty");
  SPOTV2_REQUIRE(ld >= cols && ld16 >= cols && ld16 % 8 == 0, "split_f16: ld >= cols, ld16 >= cols and ld16 %% 8 == 0");
  SPOTV2_REQUIRE(split_dim == 0 || split_dim == 1, "split_f16: split_dim is 0 (rows) or 1 (cols)");
  return split_f16(src, rows, cols, (size_t)ld, split_dim, split_at <= 0 ? kNone : split_at, nullptr, 0, hi, lo,
                   (size_t)ld16, scale_block, as_stream(stream));
}

extern "C" int spotv2_proj_fwd(const spotv2_gat_desc* d, const float* x, const void* x_hi, const void* x_lo,
                               const float* x_scale, const float* W_aug, float* P_aug, float* p_amax_or_null, void* ws,
                               size_t ws_bytes, void* stream) {
  if (int rc = check_desc(d)) return rc;
  SPOTV2_REQUIRE(x && W_aug && P_aug, "proj_fwd: null pointer");
  const ProjShape s = shape_of(d);
  cudaStream_t st = as_stream(stream);
  if (!use_tc(d)) {
    if (int rc = sgemm_simt(true, true, s.rows, s.n_aug, s.F, x, s.F, W_aug, s.F, P_aug, s.ldp, 1, ws, ws_bytes, st)) return rc;
    return p_amax_or_null ? amax_2d(P_aug, s.rows, s.HC, (size_t)s.ldp, p_amax_or_null, st) : SPOTV2_OK;
  }
  Carver c{static_cast<unsigned char*>(ws), ws ? ws_bytes : 0};
  float* blk = static_cast<float*>(c.take(kBlocksBytes));
  OperandPair xp = operand_pair(c, s.rows, s.ldf16, x_hi, x_lo, x_scale), wp = operand_pair(c, s.n_aug, s.ldf16);
  if (!blk || !xp.ok() || !wp.ok()) return fail(SPOTV2_ERR_WORKSPACE, "proj_fwd: workspace too small (%zu B)", ws_bytes);
  if (int rc = xp.split(x, s.rows, s.F, s.F, 0, kNone, s.ldf16, blk, st)) return rc;
  // W_aug = [W ; u_src ; u_dst]: the folded attention rows carry their own magnitude -> second scale group
  if (int rc = wp.split(W_aug, s.n_aug, s.F, s.F, 0, s.HC, s.ldf16, blk + kScaleBlockFloats, st)) return rc;
  F16Operand A{xp.hi, xp.lo, s.ldf16, xp.scale + 2, kNone}, B{wp.hi, wp.lo, s.ldf16, wp.scale + 2, s.HC};
  return gemm3x_f16(true, true, s.rows, s.n_aug, s.F, A, B, P_aug, s.ldp, 1, 256, 0, nullptr, 0, st, p_amax_or_null, s.HC,
                    single_product(d));
}

extern "C" int spotv2_proj_fwd_pair(const spotv2_gat_desc* d, const void* x_hi, const void* x_lo, const float* x_scale,
                                    const float* W_aug, void* P_hi, void* P_lo_or_null, float* p_scale, float* sd, void* ws,
                                    size_t ws_bytes, void* stream) {
  if (int rc = check_desc(d)) return rc;
  SPOTV2_REQUIRE(d->p_format == 1, "proj_fwd_pair: the descriptor must say p_format 1");
  SPOTV2_REQUIRE(x_hi && x_lo && x_scale && W_aug && P_hi && p_scale && sd, "proj_fwd_pair: null pointer");
  SPOTV2_REQUIRE(P_lo_or_null || single_product(d), "proj_fwd_pair: the lo plane may be omitted with gemm_algo 3 only");
  const ProjShape s = shape_of(d);
  cudaStream_t st = as_stream(stream);
  Carver c{static_cast<unsigned char*>(ws), ws ? ws_bytes : 0};
  float* wblk = static_cast<float*>(c.take(kBlocksBytes));
  const OperandPair wp = operand_pair(c, s.n_aug, s.ldf16);
  if (!wblk || !wp.ok()) return fail(SPOTV2_ERR_WORKSPACE, "proj_fwd_pair: workspace too small (%zu B)", ws_bytes);
  if (int rc = w_pair_and_out_scale(W_aug, s.n_aug, s.F, s.HC, wp.hi, wp.lo, s.ldf16, wblk, x_scale, p_scale, st)) return rc;
  F16Operand A{x_hi, x_lo, s.ldf16, x_scale + 2, kNone}, B{wp.hi, wp.lo, s.ldf16, wblk + 2, s.HC};
  PairOut out{P_hi, single_product(d) ? nullptr : P_lo_or_null, s.ldp16, p_scale + 4, sd, 2 * d->H};
  return gemm3x_f16(true, true, s.rows, s.n_aug, s.F, A, B, nullptr, 0, 1, 256 + 16, 0, nullptr, 0, st, nullptr, 0, single_product(d),
                    &out);
}

extern "C" int spotv2_proj_bwd_weight(const spotv2_gat_desc* d, const float* x, const void* x_hi, const void* x_lo,
                                      const float* x_scale, const float* dP_aug, const void* dP_hi, const void* dP_lo,
                                      const float* dp_scale, float* dW_aug, void* ws, size_t ws_bytes, void* stream) {
  if (int rc = check_desc(d)) return rc;
  SPOTV2_REQUIRE((x || x_hi) && dW_aug && (dP_aug || dP_hi), "proj_bwd_weight: null pointer");
  if (d->p_format == 1 && single_product(d) && dP_hi && !dP_lo) dP_lo = dP_hi;      // hi planes only: lo is never loaded
  SPOTV2_REQUIRE(d->p_format == 0 || (dP_hi && dP_lo && dp_scale && x_hi && x_lo && x_scale),
                 "proj_bwd_weight: p_format 1 takes x and dP as pairs");
  const ProjShape s = shape_of(d);
  cudaStream_t st = as_stream(stream);
  const int splits = weight_grad_splits(s.rows, s.n_aug, s.F, !single_product(d));
  if (!use_tc(d)) {
    SPOTV2_REQUIRE(dP_aug, "proj_bwd_weight: the CUDA-core path takes the fp32 dP_aug");
    return sgemm_simt(false, false, s.n_aug, s.F, s.rows, dP_aug, s.ldp, x, s.F, dW_aug, s.F, splits, ws, ws_bytes, st);
  }
  Carver c{static_cast<unsigned char*>(ws), ws ? ws_bytes : 0};
  float* blk = static_cast<float*>(c.take(kBlocksBytes));
  OperandPair pp = operand_pair(c, s.rows, s.ldp16, dP_hi, dP_lo, dp_scale);
  OperandPair xp = operand_pair(c, s.rows, s.ldf16, x_hi, x_lo, x_scale);
  if (!blk || !pp.ok() || !xp.ok()) return fail(SPOTV2_ERR_WORKSPACE, "proj_bwd_weight: workspace too small (%zu B)", ws_bytes);
  SPOTV2_REQUIRE(!pp.own || dP_aug, "proj_bwd_weight: dP_aug or the complete pair (dP_hi, dP_lo, dp_scale)");
  if (int rc = pp.split(dP_aug, s.rows, s.n_aug, s.ldp, 1, s.HC, s.ldp16, blk, st)) return rc;
  if (int rc = xp.split(x, s.rows, s.F, s.F, 0, kNone, s.ldf16, blk + kScaleBlockFloats, st)) return rc;
  // contraction over the B*N node rows: both operands are MN-major ([K, rows]) for this product
  F16Operand A{pp.hi, pp.lo, s.ldp16, pp.scale + 2, s.HC}, B{xp.hi, xp.lo, s.ldf16, xp.scale + 2, kNone};
  return gemm3x_f16(false, false, s.n_aug, s.F, s.rows, A, B, dW_aug, s.F, splits, 256 + 16, 0, c.p, c.left, st, nullptr, 0,
                    single_product(d));
}

extern "C" int spotv2_proj_bwd_input(const spotv2_gat_desc* d, const float* dP_aug, const void* dP_hi, const void* dP_lo,
                                     const float* dp_scale, const float* W_aug, float* dX, void* ws, size_t ws_bytes,
                                     void* stream) {
  if (int rc = check_desc(d)) return rc;
  SPOTV2_REQUIRE(W_aug && dX && (dP_aug || dP_hi), "proj_bwd_input: null pointer");
  if (d->p_format == 1 && single_product(d) && dP_hi && !dP_lo) dP_lo = dP_hi;      // hi planes only: lo is never loaded
  SPOTV2_REQUIRE(d->p_format == 0 || (dP_hi && dP_lo && dp_scale), "proj_bwd_input: p_format 1 takes dP as a pair");
  const ProjShape s = shape_of(d);
  cudaStream_t st = as_stream(stream);
  if (!use_tc(d)) {
    SPOTV2_REQUIRE(dP_aug, "proj_bwd_input: the CUDA-core path takes the fp32 dP_aug");
    return sgemm_simt(true, false, s.rows, s.F, s.n_aug, dP_aug, s.ldp, W_aug, s.F, dX, s.F, 1, ws, ws_bytes, st);
  }
  Carver c{static_cast<unsigned char*>(ws), ws ? ws_bytes : 0};
  float* blk = static_cast<float*>(c.take(kBlocksBytes));
  OperandPair pp = operand_pair(c, s.rows, s.ldp16, dP_hi, dP_lo, dp_scale), wp = operand_pair(c, s.n_aug, s.ldf16);
  if (!blk || !pp.ok() || !wp.ok()) return fail(SPOTV2_ERR_WORKSPACE, "proj_bwd_input: workspace too small (%zu B)", ws_bytes);
  SPOTV2_REQUIRE(!pp.own || dP_aug, "proj_bwd_input: dP_aug or the complete pair (dP_hi, dP_lo, dp_scale)");
  if (int rc = pp.split(dP_aug, s.rows, s.n_aug, s.ldp, 1, s.HC, s.ldp16, blk, st)) return rc;
  // dX[rows, F] = dP_aug[rows, n_aug] . W_aug[n_aug, F] contracts over the dimension that carries dP's two
  // scale groups, so the groups' inverse scales (powers of two) are folded into the rows of W_aug before
  // W_aug is split with one scale of its own: (dP s_g) . (W / s_g * t) / t.
  float* wblk = blk + kScaleBlockFloats;
  if (int rc = split_f16(W_aug, s.n_aug, s.F, s.F, 0, kNone, pp.scale + 2, s.HC, wp.hi, wp.lo, s.ldf16, wblk, st)) return rc;
  F16Operand A{pp.hi, pp.lo, s.ldp16, nullptr, kNone}, B{wp.hi, wp.lo, s.ldf16, wblk + 2, kNone};
  return gemm3x_f16(true, false, s.rows, s.F, s.n_aug, A, B, dX, s.F, 1, 256 + 16, 0, nullptr, 0, st, nullptr, 0,
                    single_product(d));
}
