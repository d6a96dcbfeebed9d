// Argument block shared by the two attention-backward kernels (attn_bwd.cu: phase-serial, two CTAs per SM,
// any shape; attn_bwd2.cu: warp-specialised and pipelined across graphs, the default whenever its
// shared-memory plan fits).
#pragma once
#include <cuda_fp16.h>
#include <initializer_list>

#include "attn_common.cuh"
#include "gemm.cuh"

namespace spotv2 {

struct AttnFwdArgs {
  AttnParams p;
  const float* bias;
  float* out;
  float* alpha_out;
};
// Edge inputs of one attention entry point as the caller passed them (the forward has no d_edge_terms)
struct AttnEdgeArgs { const float* rows; const int32_t* table; const float* v; const float* terms; float* dterms; bool backward; };
// An entry point's own argument check: fails with `st` and the message `msg` when `ok` is false
struct ArgCheck { bool ok; const char* msg; spotv2_status st = SPOTV2_ERR_INVALID_ARG; };
// Input checks of the attention entry points after check_desc, in order: `own_args`; edge rows, table and v if Fe > 0; edge
// mode 1's edge terms (backward: and d_edge_terms); `own_layout`; H, Fe limits; edge-term alignment.  `who` prefixes messages.
int check_attn_inputs(const char* who, const spotv2_gat_desc* d, std::initializer_list<ArgCheck> own_args,
                      std::initializer_list<ArgCheck> own_layout, const AttnEdgeArgs& e);
// The kernels' view of a descriptor and its edge inputs; p_format 1 adds the head pitch, ld16 of the planes and the forward's
// record flag.  The caller sets the projection's pointers (P_aug, or P_hi / P_lo / p_blk / sd32).
AttnParams attn_params_of(const spotv2_gat_desc* d, const AttnEdgeArgs& e);
// p_format 1 forward (attn_fwd16.cu): P as an fp16 operand pair, aggregation on m16n8k16 from ldmatrix fragments
int attn_fwd16_dispatch(const AttnFwdArgs& a, cudaStream_t st);
bool attn_fwd16_fits(const AttnParams& p);                        // its shared-memory plan fits this problem
int fwd16_diag_add(unsigned long long* host_out, int reset);     // adds its role counters into host_out[0..15]

// Byte offset of (row r, 16-byte chunk q) in a tile of 64-byte rows under the TMA 64B swizzle (chunk ^= (r >> 1) & 3);
// eight consecutive rows of one chunk column land in eight distinct 16-byte bank groups (conflict-free ldmatrix).
__device__ __host__ __forceinline__ uint32_t sw64(int r, int q) { return (uint32_t)(r * 64 + ((q ^ ((r >> 1) & 3)) << 4)); }

struct AttnBwdArgs {
  AttnParams p;
  const float* dout;
  float* dP_aug;       // fp32 gradient [B*N, ldp] (CUDA-core GEMM path), or null
  // tensor-core path: dP emitted as scaled fp16 hi/lo pairs [B*N, ldp16] (operand format of gemm_f16.cu);
  // the scale comes from max|dout| (dout_blk[0], bit pattern) times `bound` >= max|dP| / max|dout|.
  // ds | dd have their own magnitude: they go to dsd [B*N, 2H] in fp32 and are split by the caller.
  __half* dP_hi16;
  __half* dP_lo16;
  int ldp16;
  const float* dout_blk;   // [0] = bit pattern of max |dout| (always set for the pipelined kernel)
  const float* p_amax;     // [0] = bit pattern of max |P| over the H*C projection columns (pipelined kernel)
  float bound;
  float* dsd;
  unsigned* dsd_amax;  // pipelined / tcgen05 kernels: receives (atomicMax) the bit pattern of max |ds|, |dd|; null = off
  float* dp_blk;       // receives inverse scale [2] and scale [4] of the dP group
  float* dv_part;      // [grid][H*Fe]
  float* dbias_part;   // [grid][ldo]
  // p_format 1: dout as an fp16 operand pair made by dout_pair_prepass (attn_prep.cu): planes [B*N, ldo16], one power-of-two
  // scale per unit (graph, or (graph, head) for concat layers: units_per_graph = H); the kernel then forms no dbias.
  const __half* dO_hi = nullptr;
  const __half* dO_lo = nullptr;
  const float* dO_scale = nullptr;
  int ldo16 = 0, units_per_graph = 1;
  const float* prep_dbias_part = nullptr;   // the prepass's per-CTA column sums [prep_dbias_n][ldo], reduced with the dv partials
  int prep_dbias_n = 0;
};
int dout_pair_grid(int n_units, int upg);
// dbias != null: reduce the partials here (one more launch); dbias == null with dbias_part != null: leave the partials
// ([*n_parts][upg * C]) to the caller
int dout_pair_prepass(const float* dout, int B, int N, int C, int upg, __half* hi, __half* lo, int ld16, float* scales, float* blk,
                      float* dbias, float* dbias_part, cudaStream_t st, int* n_parts = nullptr);

__device__ __forceinline__ float dp_scale_from_amax(float amax) {   // same rule as gemm_f16.cu
  if (!(amax > 0.f) || !(amax < INFINITY)) return 1.f;
  int ex;
  frexpf(amax, &ex);
  return exp2f((float)(15 - ex));
}

// out[k] = sum_c part[c][k] in a fixed order (deterministic)
int reduce_partials(const float* part, int nparts, int len, float* out, cudaStream_t st);
// two such reductions in one launch (either may be empty: out == nullptr or len == 0)
int reduce_partials2(const float* part_a, int nparts_a, int len_a, float* out_a, const float* part_b, int nparts_b, int len_b,
                     float* out_b, cudaStream_t st);

// Pipelined kernel.  Returns SPOTV2_ERR_UNSUPPORTED (without setting an error) when the plan does not fit.
bool attn_bwd2_fits(const AttnParams& p);
// d_alpha (null = none): [B, H, N, N] gradient w.r.t. the coefficients the forward returned (spotv2_gat_attn_bwd_dalpha);
// the launchers below take it the same way
int launch_attn_bwd2(AttnBwdArgs& a, float* dv, float* dbias, void* ws, size_t ws_bytes, cudaStream_t st,
                     const float* d_alpha = nullptr);
size_t attn_bwd2_partials_bytes(const spotv2_gat_desc* d);
int bwd2_diag_add(unsigned long long* host_out, int reset);      // adds its phase counters into host_out[0..5]

// tcgen05 kernel (attn_bwd3.cu): head-mean layers, N <= 31, edge terms kept by the forward.
bool attn_bwd3_applies(const AttnParams& p);
int launch_attn_bwd3(AttnBwdArgs& a, float* dv, float* dbias, void* ws, size_t ws_bytes, cudaStream_t st,
                     const float* d_alpha = nullptr);
size_t attn_bwd3_partials_bytes(const spotv2_gat_desc* d);
int bwd3_diag_add(unsigned long long* host_out, int reset);     // adds its 16 wait / work counters into host_out[0..15]

// Large-universe path (attn_large.cu): N > 32, several CTAs per graph, attention tile in HBM.
bool attn_large_applies(const spotv2_gat_desc* d);
size_t attn_large_fwd_ws_bytes(const spotv2_gat_desc* d);
size_t attn_large_bwd_ws_bytes(const spotv2_gat_desc* d);
int attn_large_fwd(const AttnParams& p, const float* bias, float* out, float* alpha_out, void* ws, size_t ws_bytes,
                   cudaStream_t st);
int attn_large_bwd(const spotv2_gat_desc* d, AttnBwdArgs& a, float* dv, float* dbias, void* ws, size_t ws_bytes,
                   cudaStream_t st, const float* d_alpha = nullptr);

}  // namespace spotv2
