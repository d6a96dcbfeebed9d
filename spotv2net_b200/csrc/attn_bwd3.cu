// Fused GAT attention backward on the 5th-generation tensor cores (tcgen05 + TMEM + TMA).  OPT-IN (attn_bwd_algo = 3):
// parity-green on every case the pipelined mma.sync kernel (attn_bwd2.cu) passes, but measured SLOWER on B200 at the
// default geometry (2.0 - 2.4 ms against 1.95 ms per 4096-graph batch), so attn_bwd2.cu stays the default.  Same
// mathematics as the other two kernels (SURVEY.md Appendix A.3; attention recomputed from P_aug and the forward's edge
// terms, nothing of size E x H stored).
//
// What it does differently: no thread touches an MMA operand fragment.  Operands are TMA tiles in shared memory, one
// thread issues tcgen05.mma, accumulators live in TMEM, and the per-element work that remains (the "lo" halves of the
// split operands, the dP epilogue, dv) is spread once over the CTA instead of being repeated per warp.
//
// What bounds it (profiles/r2_bwd3_*): the shared-memory port.  With fp32 inputs in HBM, an fp32-accurate product on
// tf32 tensor cores needs each operand as hi + lo; per element of P that is 4 B written by TMA, 4 B read and 4 B
// written by the lo pass, and 8 B x 4/3 read by the MMAs (K = 8 per instruction, 128-row blocks of which a quarter is
// padding): ~23 B of shared-memory traffic per 4 B that arrive from HBM, i.e. ~2.8 MB per graph for phase A alone at
// 128 B/clk, on top of the edge-row chunks, the alpha tiles and the epilogue staging - at or above the time the same
// graph's bytes take to arrive from HBM.  The fix is upstream, not here: the projection GEMM has to emit P already as
// an operand pair (then phase A costs 8 B per element and no lo pass); see DESIGN.md section 9.
//
// fp32 accuracy on tf32 tensor cores: every operand is hi + lo; hi is the TMA tile as it is (the tensor core reads the
// top 19 bits of an fp32 pattern - measured, tools/bwd3_rawhi.py), lo = RN_tf32(x - trunc_tf32(x)) is written to a
// second buffer of the same layout, and a product is lo*hi + hi*lo + hi*hi.
//
// One persistent CTA per SM, 16 warps (128 registers per thread), five roles connected by mbarriers; every role walks
// the graphs of this CTA in the same order:
//   producer (1 warp)   ONE in-order stream of shared-memory slots, per graph:
//                         T  the forward's edge-term tile                         (1-D bulk copies)
//                         A  per 16 channels: P tiles of all heads + the dout tile (K-major, 64-byte swizzled rows)
//                         G  per 128 channels: dout tiles in MN-major form         (128B/32B-atom swizzle)
//                         V  edge-row chunks                                       (1-D bulk copies; not in edge_mode 1)
//   stream group (2 w)  A/G slots: the lo pass; warp w owns lo buffer w and every second slot
//   MMA warp (1 thread) phase A  dalpha[(h,j), i] = sum_c P[j,h,c] dout[i,c]      M = (head, source) rows, N = targets;
//                                B = [dout_lo ; dout_hi] so that one MMA yields hi*lo and hi*hi, a second adds lo*hi
//                       phase D  dP[(h,j), c] = sum_i alpha_h[i,j] dout[i,c]      M = (head, source) rows, N = 128 channels
//                       (one spare source row of head 0 holds ones, so the same product yields the bias gradient)
//   softmax group (8 w) thread = (head, target): self-loop mean fill, LeakyReLU, softmax -> alpha as a tf32 hi/lo pair
//                       in UMMA layout; dalpha from TMEM -> shared; softmax / LeakyReLU backward; ds, dd, dz';
//                       then V: dv += dz'^T . edge rows on the CUDA cores (exact fp32, FFMA2, two-level sums)
//   epilogue group (4w) dP from TMEM (thread = one (head, source) row, 32 channels per tcgen05.ld): scale, fp16 hi/lo
//                       pair by packed converts, a 4 KB staging tile per warp, 64-byte row pieces to global
#include <string.h>

#include "attn_bwd.cuh"
#include "tc.cuh"
#include "tma.cuh"

namespace spotv2 {

namespace {

constexpr int kSmWarps = 8, kDeWarps = 4, kStWarps = 2;
constexpr int kSmT = kSmWarps * 32, kDeT = kDeWarps * 32, kStT = kStWarps * 32;
constexpr int kWarpDe0 = kSmWarps, kWarpSt0 = kSmWarps + kDeWarps, kWarpProd = kWarpSt0 + kStWarps, kWarpMma = kWarpProd + 1;
constexpr int kB3Threads = (kWarpMma + 1) * 32;      // 512: 16 warps, 128 registers per thread
constexpr int kNS3 = kEdgeTermNS;                    // work-tile row stride (the forward's edge-term layout)
constexpr int kKB = 16;                              // channels per A slot (64-byte rows)
constexpr int kPTile = 32 * kKB * 4;                 // one (head, k-block) tile: 32 source rows x 64 B
constexpr int kCB = 128;                             // channels per G slot / phase-D block
constexpr int kGTile = 32 * 32 * 4;                  // one MN-major dout box: 32 target rows x 32 channels
constexpr int kMaxSlots3 = 8;
constexpr int kMaxChunkRows = 64;

// barrier block layout (uint64 each)
enum { kBarFull = 0, kBarEmpty = kMaxSlots3, kBarLoFull = 2 * kMaxSlots3, kBarLoEmpty = kBarLoFull + 2, kBarDAFull = kBarLoEmpty + 2,
       kBarDAEmpty, kBarAlphaFull, kBarAlphaEmpty, kBarDTFull, kBarDTEmpty, kBarVDone, kBarTDone, kNumBars };

struct Bwd3Plan {
  int n_kb, n_cb, chunk_rows, nchunks, t_pieces, n_slots, slots_per_graph, n_blk;
  uint32_t slot_bytes, lo_bytes, a_bytes, tile_bytes, alpha_bytes;
  uint32_t off_bar, off_table, off_sd, off_stage, off_dbias, off_work, off_ahi, off_alo, off_lo, off_slots, total;
};

Bwd3Plan make_plan3(const AttnParams& p) {
  Bwd3Plan s{};
  const int N = p.N, H = p.H, C = p.C, Fe = p.Fe;
  s.n_kb = (C + kKB - 1) / kKB;
  s.n_cb = (C + kCB - 1) / kCB;
  s.n_blk = (32 * H + 127) / 128;
  s.a_bytes = (uint32_t)(H + 1) * kPTile;
  s.lo_bytes = (uint32_t)round_up(s.a_bytes + kPTile > 4u * kGTile ? s.a_bytes + kPTile : 4u * kGTile, 1024);
  // block 1 of phase A reads 128 rows from row 128 on whatever H is: keep that inside the buffers
  if (s.lo_bytes < (uint32_t)s.n_blk * 128 * 64) s.lo_bytes = (uint32_t)s.n_blk * 128 * 64;
  s.slot_bytes = s.lo_bytes;
  s.tile_bytes = (uint32_t)(H * N * kNS3 * 4);
  s.alpha_bytes = (uint32_t)(32 * H * 128);
  s.t_pieces = (int)((s.tile_bytes + s.slot_bytes - 1) / s.slot_bytes);
  if (!p.terms_in) {
    int rows = (int)(s.slot_bytes / ((uint32_t)Fe * 4u)) / 8 * 8;
    if (rows > kMaxChunkRows) rows = kMaxChunkRows;
    if (rows < 8) { s.total = 0xffffffffu; return s; }
    s.chunk_rows = rows;
    s.nchunks = (p.R + rows - 1) / rows;
  }
  s.slots_per_graph = s.t_pieces + s.n_kb + s.n_cb + s.nchunks;
  uint32_t o = 0;
  s.off_bar = o;    o += 512;
  s.off_table = o;  o += (uint32_t)round_up((size_t)(p.R > 0 ? p.R : 1) * 4, 16);
  s.off_sd = o;     o += (uint32_t)round_up((size_t)N * 2 * H * 4, 16);
  s.off_stage = o;  o += (uint32_t)(kDeWarps * 4096);          // per epilogue warp: [32 sources][64 B] fp16, hi | lo
  s.off_dbias = o;  o += (uint32_t)round_up((size_t)s.n_cb * kCB * 4, 16);
  s.off_work = o;   o += (uint32_t)round_up(s.tile_bytes, 16);
  o = (uint32_t)round_up(o, 1024);
  s.off_ahi = o;    o += s.alpha_bytes;
  s.off_alo = o;    o += s.alpha_bytes;
  s.off_lo = o;     o += 2 * s.lo_bytes;
  s.off_slots = o;
  const uint32_t cap = 227 * 1024;
  const uint32_t avail = cap > o ? cap - o : 0;
  s.n_slots = (int)(avail / s.slot_bytes);
  if (s.n_slots > kMaxSlots3) s.n_slots = kMaxSlots3;
  if (s.n_slots < 3) { s.total = 0xffffffffu; return s; }
  s.total = o + (uint32_t)s.n_slots * s.slot_bytes;
  return s;
}

// round-to-nearest (ties away) onto the tf32 grid: what the tensor core would see of x, made explicit
__device__ __forceinline__ float rn_tf32(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u); }
// what the tensor core reads of an fp32 bit pattern handed to it as tf32: the top 19 bits
__device__ __forceinline__ float tr_tf32(float x) { return __uint_as_float(__float_as_uint(x) & 0xffffe000u); }
// mbarrier wait of this kernel: up to kWaitSpins polls, then the shared bounded wait with kWaitSleepNs sleeps.  The polls
// are a loop of their own because in this form they stay a loop; inside mbar_wait_bounded the compiler unrolls all 64.
constexpr int kWaitSpins = 64;
constexpr unsigned kWaitSleepNs = 32;
__device__ __forceinline__ void bar_wait(uint32_t bar, uint32_t parity) {
  bool ok = false;
  for (int spin = 0; spin < kWaitSpins && !ok; ++spin) ok = mbar_try_wait(bar, parity);
  if (!ok) mbar_wait_bounded<0, kWaitSleepNs, kWaitTrapCycles>(bar, parity);
}

// Diagnostics (spotv2_diag_counters, entries 16..31 when this kernel ran): cycles one sampling thread per role spent
// waiting on each class of barrier / inside each block of work, summed over CTAs.
//  0 producer: slot empty     1 MMA: lo buffer ready (phase A; incl. TMEM free)   2 epilogue: dP^T ready   3 MMA: alpha ready
//  4 MMA: phase D operands    5 stream: A/G slot full    6 stream: lo buffer free   7 stream: lo pass      8 stream: dz' ready
//  9 stream: V slot full     10 stream: dv arithmetic   11 softmax: T slot / tile / alpha free              12 epilogue: work
// 13 softmax: softmax        14 softmax: dalpha ready   15 softmax: TMEM dump + softmax backward
__device__ unsigned long long g_bwd3_counters[kNumCounters];
__device__ __forceinline__ void bar_wait_t(uint32_t bar, uint32_t parity, long long& acc) {
  wait_timed(acc, [&] { bar_wait(bar, parity); });
}

// a cursor over the slot ring: every role steps through the producer's slot order
struct SlotCursor {
  int slot;
  uint32_t ph;
  int n;
  __device__ __forceinline__ void advance(int k = 1) {
    slot += k;
    while (slot >= n) { slot -= n; ph ^= 1u; }
  }
};

// DROP: attention dropout in training mode (mask regenerated from the descriptor's Philox key); a separate instantiation.
// HT: the head count as a compile-time constant (0 = run-time H; the default geometry's 6 gets its own instantiation).
// The kernel without and with the gradient through the returned coefficients (spotv2_gat_attn_bwd_dalpha)
#define SPOTV2_KERNEL_NAME gat_attn_bwd3_kernel
#define SPOTV2_GA 0
#include "attn_bwd3_kernel.cuh"
#undef SPOTV2_KERNEL_NAME
#undef SPOTV2_GA
#define SPOTV2_KERNEL_NAME gat_attn_bwd3_dalpha_kernel
#define SPOTV2_GA 1
#include "attn_bwd3_kernel.cuh"
#undef SPOTV2_KERNEL_NAME
#undef SPOTV2_GA

}  // namespace

// Head-mean layers on graphs of up to 31 nodes with the forward's edge terms at hand; everything else stays on the
// mma.sync kernels.
bool attn_bwd3_applies(const AttnParams& p) {
  if (p.N > 31 || p.N < 1 || p.H > kMaxHeads || p.concat || p.C % 4 != 0 || p.ldp % 4 != 0) return false;
  if (p.Fe <= 0 || !p.edge_terms) return false;
  if (!p.terms_in && (p.Fe > 128 || p.Fe % 2 != 0 || !p.bulk_ok || !p.edge_rows || !p.table)) return false;
  if (!tma_available()) return false;
  return make_plan3(p).total <= 227 * 1024;
}

size_t attn_bwd3_partials_bytes(const spotv2_gat_desc* d) {
  const size_t ctas = (size_t)sm_count();
  const size_t ldo = d->concat ? (size_t)d->H * d->C : (size_t)d->C;
  return round_up(ctas * (kSmWarps * (size_t)d->H * d->Fe + ldo) * sizeof(float), 256);
}

int launch_attn_bwd3(AttnBwdArgs& a, float* dv, float* dbias, void* ws, size_t ws_bytes, cudaStream_t st, const float* d_alpha) {
  const AttnParams& p = a.p;
  const Bwd3Plan pl = make_plan3(p);
  if (pl.total > 227 * 1024) return fail(SPOTV2_ERR_UNSUPPORTED, "attn_bwd3: shared-memory plan does not fit");
  int grid = sm_count();
  if (grid > p.B) grid = p.B;
  const int rg = p.terms_in ? 0 : kSmWarps;
  const size_t need = ((size_t)grid * ((size_t)rg * p.H * p.Fe + p.ldo)) * sizeof(float);
  if (!ws || ws_bytes < need) return fail(SPOTV2_ERR_WORKSPACE, "attn_bwd needs %zu B of workspace, got %zu", need, ws_bytes);
  a.dv_part = static_cast<float*>(ws);
  a.dbias_part = a.dv_part + (size_t)grid * rg * p.H * p.Fe;
  CUtensorMap tmP, tmG, tmGt;
  // P_aug and dout as [graph][node][column] so that the two node rows a 32-row box reaches past a graph read as zeros
  // (columns past H*C + 2H are row padding that may hold anything: outside the map, they read as zeros too)
  if (int rc = make_tmap3_f32(&tmP, p.P_aug, (uint64_t)(p.H * p.C + 2 * p.H), (uint64_t)p.N, (uint64_t)p.B, (uint64_t)p.ldp, (uint64_t)p.N * p.ldp, kKB, 32,
                              CU_TENSOR_MAP_SWIZZLE_64B))
    return rc;
  if (int rc = make_tmap3_f32(&tmG, a.dout, (uint64_t)p.ldo, (uint64_t)p.N, (uint64_t)p.B, (uint64_t)p.ldo, (uint64_t)p.N * p.ldo, kKB, 32,
                              CU_TENSOR_MAP_SWIZZLE_64B))
    return rc;
  if (int rc = make_tmap3_f32(&tmGt, a.dout, (uint64_t)p.ldo, (uint64_t)p.N, (uint64_t)p.B, (uint64_t)p.ldo, (uint64_t)p.N * p.ldo, 32, 32,
                              CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B))
    return rc;
  const bool drop = p.drop.p > 0.f;
  if (d_alpha) {
    auto kern = p.H == 6 ? (drop ? gat_attn_bwd3_dalpha_kernel<true, 6> : gat_attn_bwd3_dalpha_kernel<false, 6>)
                         : (drop ? gat_attn_bwd3_dalpha_kernel<true, 0> : gat_attn_bwd3_dalpha_kernel<false, 0>);
    SPOTV2_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.total));
    kern<<<grid, kB3Threads, pl.total, st>>>(a, pl, tmP, tmG, tmGt, d_alpha);
  } else {
    auto kern = p.H == 6 ? (drop ? gat_attn_bwd3_kernel<true, 6> : gat_attn_bwd3_kernel<false, 6>)
                         : (drop ? gat_attn_bwd3_kernel<true, 0> : gat_attn_bwd3_kernel<false, 0>);
    SPOTV2_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.total));
    kern<<<grid, kB3Threads, pl.total, st>>>(a, pl, tmP, tmG, tmGt);
  }
  SPOTV2_CUDA_OK(cudaGetLastError());
  return reduce_partials2(a.dv_part, grid * rg, (dv && rg > 0) ? p.H * p.Fe : 0, dv, a.dbias_part, grid, dbias ? p.ldo : 0, dbias, st);
}

int bwd3_diag_add(unsigned long long* host_out, int reset) {
  return diag_add(host_out, g_bwd3_counters, reset);
}

}  // namespace spotv2
