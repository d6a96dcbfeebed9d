// Fused GAT attention backward, pipelined version (the default; attn_bwd.cu is the any-shape fallback of p_format 0).
// Same mathematics as attn_bwd.cu (SURVEY.md Appendix A.3, attention recomputed, nothing of size E x H stored), organised
// like the forward kernel: one persistent CTA per SM, 12 compute warps + 1 producer warp, every operand arrives through
// asynchronous copies that run ahead of the arithmetic, across phases and across graphs, and every product runs on the
// tensor cores (mma.sync; fp16 operand pairs on m16n8k16 for the two big products, 3xTF32 on m16n8k8 for logits and dv).
//
//   producer warp   ONE in-order stream of fixed-size slots (28 KB each, 5 of them at the default geometry), filled in
//                   exactly the order the compute warps consume them, as far ahead as the ring allows:
//                   * the forward's record (one bulk copy: its signed attention coefficients, or - with attention dropout -
//                     its edge terms) - or, without it, the edge rows a first time (logits)
//                   * phase A slots: the dout tile and the P tiles of all heads for one 32-channel block
//                   * edge rows: 1-D bulk copies, 48-row chunks (for dv)
//                   * phase D slots: groups of up to 7 dout tiles
//   compute warps   per graph
//     L  the record: copied from the slot (or edge terms recomputed: g[e,h] = <edge row, v_h>, 3xTF32, two half-groups of 6 warps)
//     S  self-loop mean fill, LeakyReLU, softmax -> alpha[h][j][i], z>0 masks       (thread per (h, i)) - skipped when the
//        record already is +-alpha (sign = LeakyReLU side; AttnParams::alpha_rec)
//     A  dalpha_h = g dO_h P_h^T         warp = (head, 16-target tile); K = channels streamed slot by slot;
//        softmax/LeakyReLU backward directly on the accumulator fragments (row sums by 4-lane shuffles),
//        dd -> global, ds partials, dz' (mean-fill redistributed) -> shared D tile
//     V  dv^T[f,h] += T^T dz'            warp = two 16-feature tiles of one 16-row group (shared dz' fragments) over the edge rows
//     D  dP_h = g alpha_h^T dO_h         warp = (head, 16-source tile), alpha^T fragments in registers
//
// Two instantiation families (template parameter P16):
//   p_format 0  P_aug and dout are fp32 (128B-swizzled fp32 tiles); every warp converts its fragments into fp16 pairs in
//               registers; dP leaves as fp16 pairs (or fp32) through per-lane global stores; dbias column sums in phase D.
//   p_format 1  P and dout arrive as fp16 operand pairs (P from the GEMM epilogue, dout from attn_prep.cu with a scale per
//               graph | (graph, head)): head-aware 4-D tensor maps bring a whole phase-A slot part with one TMA load and
//               zero-fill past a head's C, every fragment comes out of ldmatrix, dP leaves through TMA stores from per-warp
//               staging tiles (sector-aligned boxes), the bias gradient comes from the prepass.  SINGLE: hi planes only.
// Measured mma.sync facts this layout relies on (profiles/history/r1_mma_sync_latency_throughput.txt): 21-cycle
// dependent latency, one MMA per 8 cycles per SM sub-partition, so 3 chains per warp keep a tensor unit busy.
#include <string.h>

#include "attn_bwd.cuh"
#include "tma.cuh"

namespace spotv2 {

namespace {

constexpr int kW = 12;                  // compute warps
constexpr int kCT = kW * 32;            // compute threads
constexpr int kB2Threads = kCT + 32;    // + producer warp
constexpr int kTile = 4096;             // 32 rows x 32 fp32, 128B-swizzled
constexpr int kGrpTiles = 7;            // tiles per group slot
constexpr int kNS2 = 36;                // alpha / D tile row stride: (g*4 + t) fragment reads hit 32 banks
constexpr int kMaxDvUnits = 2;          // (feature tile, row group) units per warp in phase V

__device__ unsigned long long g_bwd2_counters[kNumCounters];

struct Bwd2Plan {
  int KS, chunk_rows, nchunks, n_cb, hpr, n_rounds, n_mt_chunk, ksplit;
  int n_mtiles, dv_rg, dv_rpu, dv_units, cbs_per_grp_d, tma_ok, n_slots;
  int hb;      // p_format 1: heads per TMA box of a phase-A slot (min(hpr, H))
  int stage_ok;   // p_format 1: the dz' tile (idle during phase D) can hold every warp's 2 KB dP staging tile for TMA stores
  uint32_t off_bar, off_table, off_vfrag, off_sd, off_mask, off_dspart, off_dbias, off_tile, off_D, off_slots,
      slot_bytes, total;
};

constexpr int kMaxSlots = 8;

Bwd2Plan make_plan(const AttnParams& p) {
  Bwd2Plan s{};
  const int N = p.N, H = p.H, C = p.C, Fe = p.Fe;
  s.KS = ((Fe + 7) / 8 + 7) / 8 * 8;
  s.n_cb = (C + 31) / 32;
  s.hpr = p.concat ? 3 : 6;
  s.n_rounds = (H + s.hpr - 1) / s.hpr;
  const int nh_max = H < s.hpr ? H : s.hpr;
  s.cbs_per_grp_d = p.concat ? (kGrpTiles / nh_max > 0 ? kGrpTiles / nh_max : 1) : kGrpTiles;
  s.tma_ok = (C % 4 == 0) ? 1 : 0;
  s.hb = nh_max;
  uint32_t o = 0;
  s.off_bar = o;    o += 128;
  s.off_table = o;  o += (uint32_t)round_up((size_t)(p.R > 0 ? p.R : 1) * 4, 16);
  s.off_vfrag = o;  o += (uint32_t)((Fe > 0 ? s.KS : 0) * 32 * 16);
  s.off_sd = o;     o += (uint32_t)round_up((size_t)N * 2 * H * 4, 16);
  s.off_mask = o;   o += 2 * (uint32_t)round_up((size_t)H * N * 4, 16);      // z > 0 bits | dropout keep bits
  s.off_dspart = o; o += (uint32_t)(2 * H * 32 * 4);
  s.off_dbias = o;  o += (uint32_t)round_up((size_t)p.ldo * 4, 16);
  s.off_tile = o;   o += (uint32_t)round_up((size_t)H * N * kNS2 * 4, 16);
  o = (uint32_t)round_up(o, 1024);       // (the dP staging tiles of phase D live here: swizzled TMA boxes want 512-byte alignment)
  s.off_D = o;      o += (uint32_t)round_up((size_t)H * N * kNS2 * 4, 16);
  s.stage_ok = ((size_t)H * N * kNS2 * 4 >= (size_t)kW * 2048) ? 1 : 0;
  s.off_slots = (uint32_t)round_up(o, 1024);
  // a slot holds one tile group (7 tiles) or one edge chunk (a multiple of 16 rows, at most 96)
  s.slot_bytes = kGrpTiles * kTile;
  if (Fe > 0 && (uint32_t)round_up((size_t)16 * Fe * 4, 1024) > s.slot_bytes) s.slot_bytes = (uint32_t)round_up((size_t)16 * Fe * 4, 1024);
  const uint32_t avail = 227 * 1024 - 256 > s.off_slots ? 227 * 1024 - 256 - s.off_slots : 0;
  s.n_slots = (int)(avail / s.slot_bytes);
  if (s.n_slots > kMaxSlots) s.n_slots = kMaxSlots;
  if (s.n_slots < 3) { s.total = 0xffffffffu; return s; }
  s.total = s.off_slots + (uint32_t)s.n_slots * s.slot_bytes + 256;     // + slack: k-steps padded past Fe read a few floats on
  if (Fe > 0) {
    s.chunk_rows = (int)(s.slot_bytes / ((uint32_t)Fe * 4)) / 16 * 16;
    if (s.chunk_rows > 96) s.chunk_rows = 96;
    if (s.chunk_rows > p.R) s.chunk_rows = (p.R + 15) / 16 * 16;
    s.nchunks = (p.R + s.chunk_rows - 1) / s.chunk_rows;
  }
  // phase L: a half-group of 6 warps covers one chunk: n_mt_chunk row tiles x ksplit k halves
  s.n_mt_chunk = s.chunk_rows / 16;
  s.ksplit = (s.n_mt_chunk > 0 && 2 * s.n_mt_chunk <= kW / 2 && s.KS >= 16) ? 2 : 1;
  // phase V units: (16-feature tile, row group)
  s.n_mtiles = (Fe + 15) / 16;
  if (Fe > 0) {
    int rg = (kMaxDvUnits * kW) / s.n_mtiles;
    const int rg_max = (s.chunk_rows + 7) / 8;
    if (rg > rg_max) rg = rg_max;
    if (rg > 3) rg = 3;
    if (rg < 1) { s.total = 0xffffffffu; return s; }
    s.dv_rg = rg;
    s.dv_rpu = ((s.chunk_rows + rg - 1) / rg + 7) / 8 * 8;
    s.dv_units = s.n_mtiles * rg;
  }
  return s;
}

// Two fp32 values -> packed fp16 "hi" pair and "lo" pair of the scaled values (hi + lo resolves 22 bits; s is a
// power of two that maps the tensor's largest magnitude below 2^15).  The big products of this kernel run as
// 3 x m16n8k16 on these pairs: same accuracy as the 3xTF32 split at half the tensor-pipe time (measured:
// m16n8k16.f16 and m16n8k8.tf32 both issue once per 8 cycles per sub-partition).
__device__ __forceinline__ void cvt_pair(float x0, float x1, float s, uint32_t& hi, uint32_t& lo) {
  const float y0 = x0 * s, y1 = x1 * s;
  const __half2 h = __floats2half2_rn(y0, y1);
  const float2 b = __half22float2(h);
  const __half2 l = __floats2half2_rn(y0 - b.x, y1 - b.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}
// FIX = true: the reference's default geometry (config/GNN_param.yaml: N=30, H=6, C=500, Fe=3*42, head mean) with
// every size a compile-time constant: index arithmetic folds, loops get fixed trip counts and the kernel stops
// re-reading its parameter block inside the hot loops.  FIX = false: the same code with run-time sizes.
struct FixedGeom {
  static constexpr int N = 30, H = 6, C = 500, Fe = 126, R = 870, ldp = 3012, ldo = 500;
  static constexpr int KS = 16, chunk_rows = 48, nchunks = 19, n_cb = 16, hpr = 6, n_rounds = 1, n_mt_chunk = 3, ksplit = 2;
  static constexpr int n_mtiles = 8, dv_rg = 3, dv_rpu = 16, dv_units = 24, cbs_per_grp_d = 7, n_slots = 5;
  static constexpr uint32_t slot_bytes = kGrpTiles * kTile;
};

bool plan_is_fixed_geom(const AttnParams& p, const Bwd2Plan& s) {
  using F = FixedGeom;
  return p.N == F::N && p.H == F::H && p.C == F::C && p.Fe == F::Fe && p.R == F::R && p.ldp == F::ldp && p.ldo == F::ldo &&
         !p.concat && p.bulk_ok && p.vec2_ok && s.KS == F::KS && s.chunk_rows == F::chunk_rows && s.nchunks == F::nchunks &&
         s.n_cb == F::n_cb && s.hpr == F::hpr && s.n_rounds == F::n_rounds && s.n_mt_chunk == F::n_mt_chunk &&
         s.ksplit == F::ksplit && s.n_mtiles == F::n_mtiles && s.dv_rg == F::dv_rg && s.dv_rpu == F::dv_rpu &&
         s.dv_units == F::dv_units && s.cbs_per_grp_d == F::cbs_per_grp_d && s.n_slots == F::n_slots &&
         s.slot_bytes == F::slot_bytes && s.tma_ok == 1;
}

// DROP: attention dropout in training mode (the mask is regenerated from the descriptor's Philox key, see attn_common.cuh);
// a separate instantiation so that the default path carries none of it.
// P16: p_format 1 - P AND dout arrive as fp16 operand pairs (32 x 32 tiles of 64-byte rows, 64B swizzle; P from the GEMM
// epilogue, dout from dout_pair_prepass with one scale per graph | (graph, head)): every MMA operand fragment of phases A
// and D comes out of ldmatrix, nothing is converted in registers, no tail masks (the head-aware tensor maps zero-fill
// columns past a head's C), one TMA load per phase-A slot part (all heads of a channel block in one box); the bias gradient
// comes from the prepass; dP leaves in the padded head pitch.  SINGLE (with P16): the half-precision class - hi planes only,
// one product per MMA step.  In P16 tmP = P seen head by head (box: hb heads), tmG = dout pair (box: one head),
// tmPl = dout pair (box: hb heads; concat layers' phase A).
// The kernel without and with the gradient through the returned coefficients (spotv2_gat_attn_bwd_dalpha / _pair_dalpha)
#define SPOTV2_KERNEL_NAME gat_attn_bwd2_kernel
#define SPOTV2_GA 0
#include "attn_bwd2_kernel.cuh"
#undef SPOTV2_KERNEL_NAME
#undef SPOTV2_GA
#define SPOTV2_KERNEL_NAME gat_attn_bwd2_dalpha_kernel
#define SPOTV2_GA 1
#include "attn_bwd2_kernel.cuh"
#undef SPOTV2_KERNEL_NAME
#undef SPOTV2_GA

}  // namespace

bool attn_bwd2_fits(const AttnParams& p) {
  if (p.N > 32 || p.H > kMaxHeads || p.Fe > kMaxFe) return false;
  const Bwd2Plan pl = make_plan(p);
  return pl.total <= 227 * 1024;
}

size_t attn_bwd2_partials_bytes(const spotv2_gat_desc* d) {
  const size_t ctas = (size_t)sm_count();
  const size_t ldo = d->concat ? (size_t)d->H * d->C : (size_t)d->C;
  return round_up(ctas * (3 * (size_t)d->H * d->Fe + ldo) * sizeof(float), 256);
}

int launch_attn_bwd2(AttnBwdArgs& a, float* dv, float* dbias, void* ws, size_t ws_bytes, cudaStream_t st, const float* d_alpha) {
  const AttnParams& p = a.p;
  const Bwd2Plan pl = make_plan(p);
  if (pl.total > 227 * 1024) return fail(SPOTV2_ERR_UNSUPPORTED, "attn_bwd2: shared-memory plan does not fit");
  int grid = sm_count();
  if (grid > p.B) grid = p.B;
  const int rg = p.Fe > 0 ? pl.dv_rg : 0;
  const size_t need = ((size_t)grid * ((size_t)rg * p.H * p.Fe + p.ldo)) * sizeof(float);
  if (!ws || ws_bytes < need) return fail(SPOTV2_ERR_WORKSPACE, "attn_bwd needs %zu B of workspace, got %zu", need, ws_bytes);
  a.dv_part = static_cast<float*>(ws);
  a.dbias_part = a.dv_part + (size_t)grid * rg * p.H * p.Fe;
  CUtensorMap tmP, tmG, tmPl;
  memset(&tmP, 0, sizeof(tmP));
  memset(&tmG, 0, sizeof(tmG));
  memset(&tmPl, 0, sizeof(tmPl));
  const bool p16 = p.P_hi != nullptr, single = p16 && p.P_lo == nullptr;
  if (p16) {
    if (!a.dO_hi || !a.dO_scale) return fail(SPOTV2_ERR_INVALID_ARG, "attn_bwd (p_format 1): the dout pair is missing");
    if (p.concat && p.C % 8 != 0) return fail(SPOTV2_ERR_UNSUPPORTED, "attn_bwd (p_format 1): concat layers need C %% 8 == 0");
    const uint64_t rows = (uint64_t)p.B * p.N;
    const uint32_t planes = single ? 1 : 2;
    const uint64_t p_stride = single ? 0 : (uint64_t)(p.P_lo - p.P_hi), g_stride = single ? 0 : (uint64_t)(a.dO_lo - a.dO_hi);
    if (!single && (p.P_lo <= p.P_hi || a.dO_lo <= a.dO_hi || p_stride % 8 != 0 || g_stride % 8 != 0))
      return fail(SPOTV2_ERR_INVALID_ARG, "attn_bwd (p_format 1): lo planes must follow their hi planes at multiples of 16 bytes");
    const uint64_t upg = (uint64_t)a.units_per_graph;
    // P head by head (box: hb heads); dout head by head (one head per box; hb heads per box for concat layers' phase A)
    if (int rc = make_tmap_heads_f16(&tmP, p.P_hi, p_stride, planes, rows, (uint64_t)p.C, (uint64_t)p.hp, (uint64_t)p.H, (uint64_t)p.ldp16,
                                     (uint32_t)pl.hb, CU_TENSOR_MAP_L2_PROMOTION_L2_256B))
      return rc;
    if (int rc = make_tmap_heads_f16(&tmG, a.dO_hi, g_stride, planes, rows, (uint64_t)p.C, (uint64_t)p.C, upg, (uint64_t)a.ldo16, 1)) return rc;
    if (int rc = make_tmap_heads_f16(&tmPl, a.dO_hi, g_stride, planes, rows, (uint64_t)p.C, (uint64_t)p.C, upg, (uint64_t)a.ldo16,
                                     p.concat ? (uint32_t)pl.hb : 1))
      return rc;
  } else if (pl.tma_ok) {
    // no L2 promotion: the 128-byte tile rows start anywhere in a 12 KB / 2 KB row, and fetching the enclosing 256-byte
    // blocks cost 0.4 GB of extra DRAM reads per launch (ncu: 5.02 -> 4.61 GB) for no gain in time
    if (int rc = make_tmap(&tmP, p.P_aug, (uint64_t)p.B * p.N, (uint64_t)p.ldp, (uint64_t)p.ldp, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_NONE))
      return rc;
    if (int rc = make_tmap(&tmG, a.dout, (uint64_t)p.B * p.N, (uint64_t)p.ldo, (uint64_t)p.ldo, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_NONE))
      return rc;
  }
  CUtensorMap tmD0, tmD1;
  memset(&tmD0, 0, sizeof(tmD0));
  memset(&tmD1, 0, sizeof(tmD1));
  if (p16 && pl.stage_ok) {
    // dP planes head by head with the padded pitch as the head's width (the pad columns are written, as zeros); boxes of
    // 16 (first source tile) and N - 16 (second) rows
    const uint64_t rows = (uint64_t)p.B * p.N;
    const uint64_t d_stride = single ? 0 : (uint64_t)(a.dP_lo16 - a.dP_hi16);
    if (!single && (a.dP_lo16 <= a.dP_hi16 || d_stride % 8 != 0))
      return fail(SPOTV2_ERR_INVALID_ARG, "attn_bwd (p_format 1): the dP lo plane must follow the hi plane at a multiple of 16 bytes");
    if (int rc = make_tmap_heads_f16(&tmD0, a.dP_hi16, d_stride, single ? 1 : 2, rows, (uint64_t)p.hp, (uint64_t)p.hp, (uint64_t)p.H,
                                     (uint64_t)a.ldp16, 1, CU_TENSOR_MAP_L2_PROMOTION_NONE, (uint32_t)(p.N < 16 ? p.N : 16)))
      return rc;
    if (p.N > 16)
      if (int rc = make_tmap_heads_f16(&tmD1, a.dP_hi16, d_stride, single ? 1 : 2, rows, (uint64_t)p.hp, (uint64_t)p.hp, (uint64_t)p.H,
                                       (uint64_t)a.ldp16, 1, CU_TENSOR_MAP_L2_PROMOTION_NONE, (uint32_t)(p.N - 16)))
        return rc;
  }
  const bool fixg = plan_is_fixed_geom(p, pl) && (!p16 || p.hp == 504), drop = p.drop.p > 0.f;
  if (d_alpha) {
    auto kern = drop ? (fixg ? gat_attn_bwd2_dalpha_kernel<true, true, false, false> : gat_attn_bwd2_dalpha_kernel<false, true, false, false>)
                     : (fixg ? gat_attn_bwd2_dalpha_kernel<true, false, false, false> : gat_attn_bwd2_dalpha_kernel<false, false, false, false>);
    if (p16 && !single)
      kern = drop ? (fixg ? gat_attn_bwd2_dalpha_kernel<true, true, true, false> : gat_attn_bwd2_dalpha_kernel<false, true, true, false>)
                  : (fixg ? gat_attn_bwd2_dalpha_kernel<true, false, true, false> : gat_attn_bwd2_dalpha_kernel<false, false, true, false>);
    else if (p16)
      kern = drop ? gat_attn_bwd2_dalpha_kernel<false, true, true, true> : gat_attn_bwd2_dalpha_kernel<false, false, true, true>;
    SPOTV2_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.total));
    kern<<<grid, kB2Threads, pl.total, st>>>(a, pl, tmP, tmG, tmPl, tmD0, tmD1, d_alpha);
  } else {
    auto kern = drop ? (fixg ? gat_attn_bwd2_kernel<true, true, false, false> : gat_attn_bwd2_kernel<false, true, false, false>)
                     : (fixg ? gat_attn_bwd2_kernel<true, false, false, false> : gat_attn_bwd2_kernel<false, false, false, false>);
    if (p16 && !single)
      kern = drop ? (fixg ? gat_attn_bwd2_kernel<true, true, true, false> : gat_attn_bwd2_kernel<false, true, true, false>)
                  : (fixg ? gat_attn_bwd2_kernel<true, false, true, false> : gat_attn_bwd2_kernel<false, false, true, false>);
    else if (p16)
      kern = drop ? gat_attn_bwd2_kernel<false, true, true, true> : gat_attn_bwd2_kernel<false, false, true, true>;
    SPOTV2_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.total));
    kern<<<grid, kB2Threads, pl.total, st>>>(a, pl, tmP, tmG, tmPl, tmD0, tmD1);
  }
  SPOTV2_CUDA_OK(cudaGetLastError());
  // (p_format 1: the bias gradient was formed by dout_pair_prepass)
  if (p16)
    return reduce_partials2(a.dv_part, grid * rg, (dv && p.Fe > 0) ? p.H * p.Fe : 0, dv, a.prep_dbias_part, a.prep_dbias_n,
                            (dbias && a.prep_dbias_part) ? p.ldo : 0, dbias, st);
  return reduce_partials2(a.dv_part, grid * rg, (dv && p.Fe > 0) ? p.H * p.Fe : 0, dv, a.dbias_part, grid, dbias ? p.ldo : 0, dbias, st);
}

int bwd2_diag_add(unsigned long long* host_out, int reset) {
  return diag_add(host_out, g_bwd2_counters, reset);
}

}  // namespace spotv2
