// Fused GAT attention forward for batches of small complete graphs (N <= 32).
// Replaces, per graph, PyG 2.3.0 GATConv's edge_update (gathers, lin_edge, leaky_relu),
// utils.softmax, message + 'add' aggregation, head mean/concat and bias
// ([PyG] nn/conv/gat_conv.py; reached from /root/reference/utils/models.py:146).
//
// One persistent CTA per SM, 384 threads (12 warps, 168 registers each), warp-specialised and pipelined ACROSS graphs:
//
//   group A (warps 0-2)   for graph b+1: edge rows stream through a 2-stage shared-memory ring
//                         (cp.async.bulk + mbarrier, issued two chunks ahead, across graph boundaries);
//                         g[e,h] = <edge_attr[e], v_h> on mma.sync m16n8k8 with a 3xTF32 split, scattered
//                         by the row table into tile[buf] (double buffered).
//   group B (warps 3-10)  for graph b: self-loop mean fill, s_j + d_i + g_ij, LeakyReLU, softmax over
//                         sources (one (head,target) row per thread, in place); then O_h[32 x C] = alpha_h[32 x 32] . P_h[32 x C] on mma.sync m16n8k8
//                         (3xTF32, fp32-accurate).  P arrives as TMA tiles of 32 source rows x 32 channels
//                         (128B-swizzled, conflict-free fragment reads); a warp owns two channel blocks and
//                         keeps the alpha fragments of the current head in registers.  Per-head accumulators
//                         are folded into the running sum with round-to-nearest adds.
//   warp 11               TMA producer: per graph one tile holding the s|d columns of P_aug, then the P
//                         tiles (24-slot ring; 8 slots where 24 do not fit), running ahead across graphs.
//
// Why tensor cores here: with CUDA-core FFMA2 every lane needs the whole alpha row in registers, and the
// shared-memory return path (512 B per LDS.128 per warp) bounded that version at 38 % of HBM peak
// (profiles/).  MMA fragments spread alpha and P across the lanes, cutting shared-memory traffic ~8x.
#include "attn_bwd.cuh"
#include "tma.cuh"

namespace spotv2 {

constexpr int kGroupA = 96;           // 3 logit/softmax warps (48-row edge chunks)
constexpr int kGroupB = 256;          // 8 MMA warps
constexpr int kFwdThreads = kGroupA + kGroupB + 32;
constexpr int kFwdChunkRows3 = 48;    // edge rows per ring stage: one m16 tile per group-A warp
constexpr int kCbPerPass = 8;         // channel blocks per pass: one per MMA warp
constexpr int kPSlots = 24;           // P-tile ring depth
// P-tile ring depth of the kernel for shapes whose plan does not fit with 24 slots (N x H x Fe large: at N = 32, H = 8,
// Fe = 512 the 24-slot plan needs 287 744 B).  Any depth >= kCbPerPass keeps the stale-fill guard valid: within a graph
// a warp's consecutive tiles are at most kCbPerPass apart in the ring's fill order (G tiles per head, G <= 8), so when it
// reaches fill r of a slot, fill r - 1 of that slot is at or before its own previous tile and has landed; across graphs
// the CTA barrier behind the softmax orders everything.
constexpr int kPSlotsLean = kCbPerPass;
constexpr int kPTileBytes = 32 * 128; // 32 source rows x 32 channels fp32, 128B-swizzled

// wait-cycle diagnostics of this kernel (see spotv2_diag_counters)
__device__ unsigned long long g_diag_counters[kNumCounters];

// The kernel with the 24-slot P ring and, for the shapes whose plan does not fit with it, the 8-slot one
#define SPOTV2_KERNEL_NAME gat_attn_fwd_kernel
#define SPOTV2_PSLOTS kPSlots
#include "attn_fwd_kernel.cuh"
#undef SPOTV2_KERNEL_NAME
#undef SPOTV2_PSLOTS
#define SPOTV2_KERNEL_NAME gat_attn_fwd_lean_kernel
#define SPOTV2_PSLOTS kPSlotsLean
#include "attn_fwd_kernel.cuh"
#undef SPOTV2_KERNEL_NAME
#undef SPOTV2_PSLOTS

template <int NPAIRS, bool VEC2>
static int launch_fwd(const AttnFwdArgs& a, cudaStream_t st) {
  const AttnParams& p = a.p;
  // alpha tile stride 36 floats: a fragment read touches source rows 2t (t = 0..3) x 8 consecutive targets;
  // 72 floats between those rows = 8 banks, so the 32 lanes hit 32 distinct banks
  const int NS = 36;
  const size_t tile_bytes = round_up((size_t)p.H * p.N * NS * 4, 16);
  const size_t sd_bytes = round_up((size_t)p.N * 2 * p.H * 4, 16);
  auto finish = [&](AttnSmem s) {                 // the common plan reserves one tile + one sd; double-buffer both
    s.NS = NS;
    s.off_tile = s.off_sd + 2 * sd_bytes;
    s.off_ring = round_up(s.off_tile + 2 * tile_bytes, 128);
    s.base_total = s.off_ring;
    return s;
  };
  // + 256: zero pad behind the ring (k-steps padded past Fe read up to 63 floats beyond the last staged row)
  auto ptile_off = [&](const AttnSmem& s) { return round_up(s.off_ring + 2 * s.ring_stage_bytes + 256, 1024); };
  auto total = [&](const AttnSmem& s, int slots) { return ptile_off(s) + (size_t)(slots + 2) * kPTileBytes; };
  auto plan = [&](int slots) {                    // the largest ring stage (48, 32 or 16 rows) that fits, else 16 rows
    AttnSmem s = finish(attn_smem_plan(p.N, p.Fe, p.H, p.R, NPAIRS, kFwdChunkRows3));
    for (int rows = kFwdChunkRows3 - 16; rows >= 16 && total(s, slots) > 227 * 1024; rows -= 16)
      s = finish(attn_smem_plan(p.N, p.Fe, p.H, p.R, NPAIRS, rows));
    return s;
  };
  AttnSmem sm = plan(kPSlots);
  const bool lean = total(sm, kPSlots) > 227 * 1024;       // the 8-slot kernel: only where 24 slots do not fit
  if (lean) sm = plan(kPSlotsLean);
  const size_t smem = total(sm, lean ? kPSlotsLean : kPSlots);
  if (smem > 227 * 1024)
    return fail(SPOTV2_ERR_UNSUPPORTED, "attn_fwd needs %zu B shared memory (> 227 KB)", smem);
  CUtensorMap tmP;      // P_aug as [B*N rows, ldp cols]; tiles of 32 rows x 32 channels
  if (int rc = make_tmap(&tmP, p.P_aug, (uint64_t)p.B * p.N, (uint64_t)p.ldp, (uint64_t)p.ldp, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B))
    return rc;
  const bool fix = NPAIRS == 15 && VEC2 && p.N == 30 && p.H == 6 && p.C == 500 && p.Fe == 126 && p.R == 870 && !p.concat && p.ldp == 3012 &&
                   p.ldo == 500 && p.bulk_ok && sm.NS == 36 && sm.KS == 16 && sm.chunk_rows == kFwdChunkRows3;
  auto kern = lean  ? gat_attn_fwd_lean_kernel<NPAIRS, VEC2, false>
              : fix ? gat_attn_fwd_kernel<NPAIRS, VEC2, (NPAIRS == 15 && VEC2)> : gat_attn_fwd_kernel<NPAIRS, VEC2, false>;
  SPOTV2_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int grid = sm_count();
  if (grid > p.B) grid = p.B;
  kern<<<grid, kFwdThreads, smem, st>>>(a, sm, (uint32_t)ptile_off(sm), tmP);
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

template <int NPAIRS>
static int dispatch_vec(const AttnFwdArgs& a, cudaStream_t st) {
  return a.p.vec2_ok ? launch_fwd<NPAIRS, true>(a, st) : launch_fwd<NPAIRS, false>(a, st);
}

int attn_fwd_dispatch(const AttnFwdArgs& a, cudaStream_t st) {
  const int np = (a.p.N + 1) / 2;
  if (np <= 4) return dispatch_vec<4>(a, st);
  if (np <= 8) return dispatch_vec<8>(a, st);
  if (np <= 15) return dispatch_vec<15>(a, st);
  if (np <= 16) return dispatch_vec<16>(a, st);
  return fail(SPOTV2_ERR_UNSUPPORTED, "N=%d > 32: the one-CTA-per-graph kernel covers N <= 32", a.p.N);
}

}  // namespace spotv2

namespace spotv2 { int bwd_diag_add(unsigned long long* host_out, int reset); }
using namespace spotv2;

extern "C" int spotv2_diag_counters(unsigned long long* host_out, int reset) {
  SPOTV2_REQUIRE(host_out, "diag_counters: null pointer");
  SPOTV2_CUDA_OK(cudaDeviceSynchronize());
  for (int k = 0; k < 2 * kNumCounters; ++k) host_out[k] = 0;
  if (int rc = diag_add(host_out, g_diag_counters, reset)) return rc;
  if (int rc = fwd16_diag_add(host_out, reset)) return rc;      // whichever forward ran contributes; the other adds zeros
  return bwd_diag_add(host_out + kNumCounters, reset);       // entries 16..31: backward phase times
}

extern "C" int spotv2_gat_attn_fwd(const spotv2_gat_desc* d, const float* P_aug,
                                   const float* edge_rows, const int32_t* table, const float* v,
                                   const float* bias_or_null, float* out, float* alpha_or_null,
                                   float* edge_terms_or_null, void* ws, size_t ws_bytes, void* stream) {
  if (int rc = check_desc(d)) return rc;
  const AttnEdgeArgs e{edge_rows, table, v, edge_terms_or_null, nullptr, false};
  if (int rc = check_attn_inputs("attn_fwd", d, {{P_aug && out, "attn_fwd: P_aug and out must be non-null"}},
                                 {{aligned16(P_aug) && aligned16(out), "attn_fwd: P_aug/out must be 16-byte aligned"}}, e))
    return rc;
  AttnFwdArgs a{attn_params_of(d, e), bias_or_null, out, alpha_or_null};
  a.p.P_aug = P_aug;
  if (attn_large_applies(d))       // several CTAs per graph, attention tile in the workspace (or alpha_or_null)
    return attn_large_fwd(a.p, bias_or_null, out, alpha_or_null, ws, ws_bytes, as_stream(stream));
  return attn_fwd_dispatch(a, as_stream(stream));
}
