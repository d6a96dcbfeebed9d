// fp32-accurate projection GEMM on tcgen05 with fp16 operand pairs ("3xFP16").
//
//   C[m,n] = sum_k A(m,k) B(n,k)        A = (A_hi + A_lo) / sA,  B = (B_hi + B_lo) / sB
//   acc   += A_lo*B_hi + A_hi*B_lo + A_hi*B_hi   (kind::f16 MMAs, fp32 accumulate in TMEM)
//   C      = acc * (1/sA) * (1/sB)
//
// Why fp16 pairs instead of tf32 pairs (gemm_tc.cu): an fp16 significand carries the same 11 bits as
// tf32, so hi + lo still resolves 22 bits, but kind::f16 issues at twice the tf32 rate and the operands
// take half the bytes in HBM, L2 and shared memory.  fp16's narrow exponent is handled by a power-of-two
// scale per operand group (exact to apply and to remove): the group's largest magnitude is mapped into
// [2^14, 2^15); elements more than ~2^17 below it lose relative precision but their ABSOLUTE error stays
// below 2^-39 of the group maximum, far inside the 1e-5 max-norm parity budget (fp16 subnormals are
// honoured by the tensor core).  A group is "rows of the operand below / at-or-above split_at" along its
// M|N dimension: W_aug = [W ; u] and dP_aug = [dP | ds | dd] carry two magnitudes, x carries one.
//
// The accumulation-chain limit of gemm_tc.cu applies unchanged (the tensor core's fp32 adder truncates):
// TMEM holds 128-element K chunks, eight consumer warps fold them into fp32 registers round-to-nearest.
//
// Output: fp32 C (or split-K partials) through 3-D TMA stores - or, for the forward projection of p_format 1, the fp16
// operand PAIR of C * s (hi | lo planes; s from an a-priori bound, see pair_out_scale), split in the epilogue registers and
// stored through the same TMA path; the second column group (the logit terms s | d) additionally in fp32.
//
// Kernel shape: persistent clusters of two CTAs (one per SM), 384 threads each (warp 0 TMA, warp 1 MMA issue, warp 2 TMEM
// allocator, warps 4-11 accumulate + epilogue).  A work item is a PAIR tile of 256 x BN x TBK: CTA rank r loads A rows
// pair_mt * 256 + r * 128 and half of B's BN columns, the leader (rank 0) issues cta_group::2 MMAs of M = 256 that read
// both CTAs' shared memory, and each CTA drains its own 128 rows from its own TMEM.  Against a CTA that computes a 128 x BN
// tile alone this cuts the TMA loads and the tensor core's shared-memory operand reads per SM by a third (B is no longer
// loaded twice).  The single-product half-precision class runs the same template as one CTA per 128 x BN tile (see
// gemm3x_f16).  TBK = 64 | 32 fp16 elements.
#include <cuda_fp16.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "gemm.cuh"
#include "tc.cuh"
#include "tma.cuh"

namespace spotv2 {

namespace {

constexpr int HBM_ = 128;        // UMMA M
constexpr int HUMMA_K = 16;      // fp16
constexpr int kHThreads = 384;
constexpr int kHEpiWarps = 8;

struct HParams {
  int M, N, K;
  int ldc;
  float* C;
  int pm_tiles, n_tiles, splits, kb_per_split, kb_total, kb_per_chunk;   // pm_tiles: 256-row pair tiles
  size_t split_stride;
  const float* a_inv;   // 2 inverse scales of A's groups (null = 1)
  const float* b_inv;
  int a_split, b_split;
  int scale_in_kernel;  // 0 when a split-K reduce applies the scales
  unsigned* amax_out;   // optional: bit pattern of max |C[m, n]| over n < amax_cols (splits == 1 only)
  int amax_cols;
  int single;           // 1: half-precision class (gemm_algo 3): only the A_hi * B_hi product, lo tiles not even loaded
  int pair_out;         // 0: fp32 C; 1: C leaves as an fp16 hi | lo pair (planes of tmC); 2: hi plane only
  const float* out_scale;   // pair_out: 2 power-of-two scales of the output's column groups (col < / >= b_split)
  float* tail32;            // pair_out: fp32 copy of the columns >= b_split, [M, tail_ld] (null: none)
  int tail_ld;
  int tma_store;        // 1: C tiles / split-K partials leave through TMA bulk stores (16-byte aligned rows); 0: st.global
  int dbg;              // bring-up probe, compiled in only with -DSPOTV2_BRINGUP (env SPOTV2_GEMM_DBG): bit 0 skip the
                        // global stores, bit 1 skip scale + amax, bit 2 skip the per-chunk register accumulation
                        // (results are then wrong: timing only).  The product library carries none of it.
};
#ifdef SPOTV2_BRINGUP
#define SPOTV2_DBG(p) ((p).dbg)
#else
#define SPOTV2_DBG(p) 0
#endif

template <int BN, int TBK, bool A_KM, bool B_KM, int CTAS>
struct HSmem {
  static constexpr int kAOp = HBM_ * TBK * 2;              // this CTA's 128 rows of one A operand tile (hi or lo), bytes
  static constexpr int kBOp = (BN / CTAS) * TBK * 2;       // this CTA's share of the B tile's columns
  static constexpr int kStage = 2 * kAOp + 2 * kBOp;
  // K-major x K-major with 32-element k-blocks (the forward projection): three stages and FOUR 2 KB store boxes per
  // epilogue warp.  With two boxes the pair epilogue waited on the copy engine before six of its eight pieces (the stores
  // queue behind the operand loads); the MMA warp, which can run only two accumulation chunks ahead, stalled for it: 0.17 ms
  // of the K = 1260 product (bring-up probe, tools/gemm_dbg_probe.sh).  Pair tiles keep the ring depths in k-blocks of the
  // 1-CTA tiles (3, 4 at TBK = 32, 2 at TBK = 64), whose stages are half as large again.
  static constexpr bool kWideEpi = (TBK == 32) && A_KM && B_KM;
  static constexpr int kRingBytes = CTAS == 2 ? 160 * 1024 : 200 * 1024, kMaxStages = CTAS == 2 ? 4 : 6;
  static constexpr int kStages = kWideEpi ? 3 : (kRingBytes / kStage > kMaxStages ? kMaxStages : kRingBytes / kStage);
  static constexpr int kBarOff = kStages * kStage;
  static constexpr int kEpiOff = kBarOff + 1024;                     // 8 epilogue warps x 4224 B: a 32 x 32 fp32 output block each
  static constexpr int kEpiWarpBytes = kWideEpi ? 8192 : 32 * 33 * 4;    // ([32][33] transpose, or 2 KB swizzled TMA store boxes)
  static constexpr int kBoxStride = kWideEpi ? 8192 : 4096;         // store boxes of one warp
  static constexpr int kPairBoxes = kWideEpi ? 4 : 2;
  static constexpr int kEpiBytes = kHEpiWarps * kEpiWarpBytes;
  static constexpr int kTotal = kEpiOff + kEpiBytes + 1024;
  static constexpr uint32_t kTxBytes = CTAS * kStage;        // both CTAs' loads complete on the leader's full barrier
};

// Bounded wait that names the barrier that starved before it traps: a lost arrival from the other CTA of the pair must
// fail loudly instead of hanging the GPU.
enum { kWaitFull = 0, kWaitEmpty, kWaitTempty, kWaitPeerEmpty };
__device__ __noinline__ void gemm_wait_report(int id, uint32_t parity) {
  const char* const names[] = {"full (operands landed)", "empty (stage consumed)", "tempty (accumulator drained)",
                               "empty at exit (last stage released)"};
  printf("gemm3x_f16: wait on %s timed out (block %d rank %u thread %d parity %u)\n", names[id], (int)blockIdx.x,
         cluster_ctarank(), (int)threadIdx.x, parity);
}
constexpr int kWaitSpins = 16;
constexpr unsigned kWaitSleepNs = 64;
__device__ __forceinline__ void hwait(uint64_t* bar, uint32_t parity, int id) {
  mbar_wait_bounded<kWaitSpins, kWaitSleepNs, kWaitTrapCycles>(smem_u32(bar), parity, [=] { gemm_wait_report(id, parity); });
}

// CTAS = 2: pair tiles on a cluster of two CTAs (launched with cluster dimension 2); CTAS = 1: every CTA computes a
// 128 x BN tile alone (see gemm3x_f16 for which products take which).
template <int BN, int TBK, bool A_KM, bool B_KM, int CTAS>
__global__ void __launch_bounds__(kHThreads, 1)
gemm3x_f16_kernel(const __grid_constant__ CUtensorMap tmAh, const __grid_constant__ CUtensorMap tmAl,
                  const __grid_constant__ CUtensorMap tmBh, const __grid_constant__ CUtensorMap tmBl,
                  const __grid_constant__ CUtensorMap tmC, const HParams p) {
  using S = HSmem<BN, TBK, A_KM, B_KM, CTAS>;
  constexpr int kStages = S::kStages;
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + S::kBarOff);
  uint64_t* empty = full + kStages;
  uint64_t* tfull = empty + kStages;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = CTAS == 2 ? cluster_ctarank() : 0;
  const int pair_id = blockIdx.x / CTAS, num_pairs = gridDim.x / CTAS;
  const int total_items = p.pm_tiles * p.n_tiles * p.splits;
  constexpr uint32_t kTmemCols = 2 * BN;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmAh); prefetch_tmap(&tmAl); prefetch_tmap(&tmBh); prefetch_tmap(&tmBl);
  }
  if (warp == 1 && lane == 0) {
    // full and tempty are used in the leader only: full completes on both CTAs' loads, tempty on both CTAs' drains
    for (int s = 0; s < kStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&tfull[s], 1); mbar_init(&tempty[s], CTAS * kHEpiWarps); }
    fence_mbar_init();
  }
  if constexpr (CTAS == 2) {
    if (warp == 2) tmem_alloc_pair(tmem_slot, kTmemCols);
    tc_fence_before();
    cluster_sync();           // the peer's barriers are initialised before anything signals them
  } else {
    if (warp == 2) tmem_alloc(tmem_slot, kTmemCols);
    tc_fence_before();
    __syncthreads();
  }
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // n fastest: the pairs of one wave share the A rows (x / dP tiles) through L2, B (weights) is small.  This CTA's
  // 128-row tile of the pair tile is mt; when m_tiles is odd the last pair's second half reads zeros (TMA fills rows >= M)
  // and stores nothing.
  auto tile_coords = [&](int item, int& mt, int& nt, int& sp) {
    nt = item % p.n_tiles;
    const int r = item / p.n_tiles;
    mt = CTAS * (r % p.pm_tiles) + (int)rank;
    sp = r / p.pm_tiles;
  };

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (elect_one()) {
      const uint32_t full_leader = CTAS == 2 ? mapa_shared(full, 0) : 0;
      int stage = 0; uint32_t phase = 0;
      for (int item = pair_id; item < total_items; item += num_pairs) {
        int mt, nt, sp; tile_coords(item, mt, nt, sp);
        const int kb0 = sp * p.kb_per_split;
        const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        const int n0 = nt * BN + (int)rank * (BN / CTAS);
        for (int kb = kb0; kb < kb1; ++kb) {
          hwait(&empty[stage], phase ^ 1, kWaitEmpty);
          unsigned char* st = smem + stage * S::kStage;
          const bool lo = !p.single;
          const uint32_t fb = full_leader + stage * (uint32_t)sizeof(uint64_t);
          if (rank == 0) mbar_expect_tx(&full[stage], lo ? S::kTxBytes : S::kTxBytes / 2);
          auto tma_load = [&](void* dst, const CUtensorMap* tm, int c0, int c1) {
            if constexpr (CTAS == 2) tma_load_2d_pair(dst, tm, c0, c1, fb);
            else tma_load_2d(dst, tm, c0, c1, &full[stage]);
          };
          const int k = kb * TBK;
          if (A_KM) {
            tma_load(st, &tmAh, k, mt * HBM_);
            if (lo) tma_load(st + S::kAOp, &tmAl, k, mt * HBM_);
          } else {
#pragma unroll
            for (int blk = 0; blk < HBM_ / 64; ++blk) {
              tma_load(st + blk * (TBK * 128), &tmAh, mt * HBM_ + blk * 64, k);
              if (lo) tma_load(st + S::kAOp + blk * (TBK * 128), &tmAl, mt * HBM_ + blk * 64, k);
            }
          }
          unsigned char* sb = st + 2 * S::kAOp;
          if (B_KM) {
            tma_load(sb, &tmBh, k, n0);
            if (lo) tma_load(sb + S::kBOp, &tmBl, k, n0);
          } else {
#pragma unroll
            for (int blk = 0; blk < BN / CTAS / 64; ++blk) {
              tma_load(sb + blk * (TBK * 128), &tmBh, n0 + blk * 64, k);
              if (lo) tma_load(sb + S::kBOp + blk * (TBK * 128), &tmBl, n0 + blk * 64, k);
            }
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
      // the leader's last commits to this CTA's empty barriers must land before the CTA exits (pairs)
      for (int s = 0; s < kStages; ++s) {
        hwait(&empty[stage], phase ^ 1, kWaitPeerEmpty);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (rank == 0 && elect_one()) {
      auto mma = [&](uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
        if constexpr (CTAS == 2) umma_f16_pair(d, a, b, idesc, acc);
        else umma_f16(d, a, b, idesc, acc);
      };
      auto commit = [&](uint64_t* bar) {
        if constexpr (CTAS == 2) umma_commit_pair(bar, 0x3);
        else umma_commit(bar);
      };
      // instruction descriptor: D = f32 (1 << 4), A/B = f16 (0), majors, N >> 3, M >> 4 (pairs: M = 256, both CTAs' rows)
      constexpr uint32_t idesc = (1u << 4) | ((A_KM ? 0u : 1u) << 15) | ((B_KM ? 0u : 1u) << 16) |
                                 ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((CTAS * HBM_) >> 4) << 24);
      // K-major: rows of TBK*2 bytes (128 B -> SWIZZLE_128B, 64 B -> SWIZZLE_64B), 8-row atoms.
      // MN-major: 64-element (128 B) rows along M|N, 8 k-rows per 1024 B atom (SBO), LBO = one 64-wide block.
      constexpr uint32_t k_sbo = 8 * TBK * 2, k_lt = (TBK == 64) ? 2 : 4;
      constexpr uint32_t a_lbo = A_KM ? 16 : TBK * 128, b_lbo = B_KM ? 16 : TBK * 128;
      constexpr uint32_t a_sbo = A_KM ? k_sbo : 1024, b_sbo = B_KM ? k_sbo : 1024;
      constexpr uint32_t a_lt = A_KM ? k_lt : 2, b_lt = B_KM ? k_lt : 2;
      constexpr uint32_t a_kstep = A_KM ? HUMMA_K * 2 : HUMMA_K * 128;   // bytes per k-step of 16
      constexpr uint32_t b_kstep = B_KM ? HUMMA_K * 2 : HUMMA_K * 128;
      int stage = 0; uint32_t phase = 0;
      uint32_t chunk_ctr = 0;
      for (int item = pair_id; item < total_items; item += num_pairs) {
        int mt, nt, sp; tile_coords(item, mt, nt, sp);
        const int kb0 = sp * p.kb_per_split;
        const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        for (int kc = kb0; kc < kb1; kc += p.kb_per_chunk, ++chunk_ctr) {
          const int as = chunk_ctr & 1;
          hwait(&tempty[as], ((chunk_ctr >> 1) & 1) ^ 1, kWaitTempty);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + (uint32_t)(as * BN);
          uint32_t accum = 0;
          const int kce = min(kb1, kc + p.kb_per_chunk);
          for (int kb = kc; kb < kce; ++kb) {
            hwait(&full[stage], phase, kWaitFull);
            tc_fence_after();
            const uint32_t sa = smem_u32(smem + stage * S::kStage);
            const uint32_t sb = sa + 2 * S::kAOp;
#pragma unroll
            for (int ks = 0; ks < TBK / HUMMA_K; ++ks) {
              const uint64_t ah = make_desc(sa + ks * a_kstep, a_lbo, a_sbo, a_lt);
              const uint64_t al = make_desc(sa + S::kAOp + ks * a_kstep, a_lbo, a_sbo, a_lt);
              const uint64_t bh = make_desc(sb + ks * b_kstep, b_lbo, b_sbo, b_lt);
              const uint64_t bl = make_desc(sb + S::kBOp + ks * b_kstep, b_lbo, b_sbo, b_lt);
              if (!p.single) {
                mma(d_tmem, al, bh, idesc, accum);
                mma(d_tmem, ah, bl, idesc, 1);
                accum = 1;
              }
              mma(d_tmem, ah, bh, idesc, accum);
              accum = 1;
            }
            commit(&empty[stage]);
            if (++stage == kStages) { stage = 0; phase ^= 1; }
          }
          commit(&tfull[as]);
        }
      }
    }
  } else if (warp >= 4) {
    // ===================== accumulate + epilogue (both CTAs, each its own 128 rows) =====================
    constexpr int HALF = BN / 2;
    const int q = warp & 3;
    const int ch = (warp - 4) >> 2;
    const uint32_t tempty_leader = CTAS == 2 ? mapa_shared(tempty, 0) : 0;
    uint32_t chunk_ctr = 0;
    for (int item = pair_id; item < total_items; item += num_pairs) {
      int mt, nt, sp; tile_coords(item, mt, nt, sp);
      const int kb0 = sp * p.kb_per_split;
      const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
      float acc[HALF];
#pragma unroll
      for (int e = 0; e < HALF; ++e) acc[e] = 0.f;
      for (int kc = kb0; kc < kb1; kc += p.kb_per_chunk, ++chunk_ctr) {
        const int as = chunk_ctr & 1;
        // plain bounded wait: a report call here costs the register-bound epilogue spills, and a lost tfull in either CTA
        // starves the leader's tempty wait, which names it
        mbar_wait(&tfull[as], (chunk_ctr >> 1) & 1);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * BN + ch * HALF);
#pragma unroll
        for (int c0 = 0; c0 < HALF; c0 += 32) {
          uint32_t r[32];
          tmem_ld32(taddr + c0, r);
#pragma unroll
          if (!(SPOTV2_DBG(p) & 4))
#pragma unroll
            for (int e = 0; e < 32; ++e) acc[c0 + e] += __uint_as_float(r[e]);   // round-to-nearest adds
          else acc[c0] += __uint_as_float(r[0]);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if constexpr (CTAS == 2) mbar_arrive_cluster(tempty_leader + as * (uint32_t)sizeof(uint64_t));
          else mbar_arrive(&tempty[as]);
        }
      }
      const int row = mt * HBM_ + q * 32 + lane;
      const int col0 = nt * BN + ch * HALF;
      float row_amax = 0.f;
      if (row < p.M && col0 < p.N && !(SPOTV2_DBG(p) & 2)) {
        if (p.scale_in_kernel) {      // powers of two: exact
          const float ra = p.a_inv ? p.a_inv[row >= p.a_split ? 1 : 0] : 1.f;
          const float os0 = p.pair_out ? p.out_scale[0] : 1.f, os1 = p.pair_out ? p.out_scale[1] : 1.f;
          const float cb0 = ra * (p.b_inv ? p.b_inv[0] : 1.f) * os0, cb1 = ra * (p.b_inv ? p.b_inv[1] : 1.f) * os1;
#pragma unroll
          for (int e = 0; e < HALF; ++e) acc[e] *= (col0 + e >= p.b_split) ? cb1 : cb0;
        }
        if (p.amax_out) {             // the attention backward sizes its fp16 operand scale from this
          float mx = 0.f;
#pragma unroll
          for (int e = 0; e < HALF; ++e)
            if (col0 + e < p.amax_cols) mx = fmaxf(mx, fabsf(acc[e]));
          row_amax = mx;
        }
      }
      if (p.pair_out && p.tail32 && row < p.M && col0 + HALF > p.b_split && col0 < p.N) {
        // the second column group (s | d) also in fp32, free of the pair's scale (a power of two: exact)
        const float un = 1.f / p.out_scale[1];
        float* dst = p.tail32 + (size_t)row * p.tail_ld - p.b_split;
#pragma unroll
        for (int e = 0; e < HALF; ++e)
          if (col0 + e >= p.b_split && col0 + e < p.N) dst[col0 + e] = acc[e] * un;
      }
      if (p.pair_out && (SPOTV2_DBG(p) & 8)) {
        // (bring-up probe: no pair epilogue at all)
      } else if (p.pair_out) {
        // The tile leaves as the fp16 operand pair of the scaled result: 32 x 32 pieces, hi plane then lo plane, each a
        // 2 KB box (64-byte rows, 64B swizzle) handed to the TMA engine; the boxes of this warp rotate, and a box is
        // refilled once the engine has read the store issued from it kPairBoxes stores ago.
        unsigned char* box = smem + S::kEpiOff + (warp - 4) * S::kBoxStride;
        const int row_base = mt * HBM_ + q * 32;
#pragma unroll
        for (int cc = 0; cc < HALF / 32; ++cc) {
          uint32_t hi[16], lo[16];
#pragma unroll
          for (int e = 0; e < 16; ++e) {
            const float y0 = acc[cc * 32 + 2 * e], y1 = acc[cc * 32 + 2 * e + 1];
            const __half2 h = __floats2half2_rn(y0, y1);
            const float2 b = __half22float2(h);
            const __half2 l = __floats2half2_rn(y0 - b.x, y1 - b.y);
            hi[e] = *reinterpret_cast<const uint32_t*>(&h);
            lo[e] = *reinterpret_cast<const uint32_t*>(&l);
          }
#pragma unroll
          for (int pln = 0; pln < 2; ++pln) {
            if (pln == 1 && p.pair_out != 1) break;
            unsigned char* hb = box + ((p.pair_out == 1 ? 2 * cc + pln : cc) & (S::kPairBoxes - 1)) * 2048;
            if (lane == 0) bulk_wait_read<S::kPairBoxes - 1>();
            __syncwarp();
#pragma unroll
            for (int c = 0; c < 4; ++c)
              *reinterpret_cast<uint4*>(hb + lane * 64 + ((c ^ ((lane >> 1) & 3)) << 4)) =
                  pln ? make_uint4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3])
                      : make_uint4(hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
              if (col0 + cc * 32 < p.N && row_base < p.M && !(SPOTV2_DBG(p) & 1))
                tma_store_3d(&tmC, smem_u32(hb), col0 + cc * 32, row_base, pln);
              bulk_commit();
            }
          }
        }
      } else if (p.tma_store && !(SPOTV2_DBG(p) & 1)) {
        // Asynchronous stores (measured: with st.global the epilogue warps sat in the LSU queue for ~0.5 ms of the K = 1260
        // product while the MMA warp waited for them to drain TMEM).  Each warp parks 32 x 16 pieces of its block in two
        // alternating swizzled shared-memory boxes and one lane hands each to the TMA engine; the warp only waits for the
        // engine to have READ the box written two pieces ago before refilling it.  Rows >= M and columns >= N are clipped by the tensor map.
        unsigned char* box = smem + S::kEpiOff + (warp - 4) * S::kBoxStride;      // two 2 KB half-boxes (32 rows x 16 columns, 64B swizzle)
        const int row_base = mt * HBM_ + q * 32;
#pragma unroll
        for (int cc = 0; cc < HALF / 16; ++cc) {
          unsigned char* hb = box + (cc & 1) * 2048;
          if (lane == 0) bulk_wait_read<1>();                                             // the store before last has been read
          __syncwarp();
#pragma unroll
          for (int c = 0; c < 4; ++c)
            *reinterpret_cast<float4*>(hb + lane * 64 + ((c ^ ((lane >> 1) & 3)) << 4)) =
                make_float4(acc[cc * 16 + 4 * c], acc[cc * 16 + 4 * c + 1], acc[cc * 16 + 4 * c + 2], acc[cc * 16 + 4 * c + 3]);
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            if (col0 + cc * 16 < p.N && row_base < p.M)
              tma_store_3d(&tmC, smem_u32(hb), col0 + cc * 16, row_base, sp);
            bulk_commit();                                                  // always commit: keeps the group count in step with cc
          }
        }
      } else if (!(SPOTV2_DBG(p) & 1)) {
        // Stores: a lane owns an output ROW, so storing straight from registers makes every warp store touch 32 rows
        // (16 bytes each; ncu showed the LSU queue throttling the K = 1260 product).  Instead each 32 x 32 block goes
        // through a padded shared-memory transpose and leaves as 32 stores of 128 contiguous bytes.
        float* stage = reinterpret_cast<float*>(smem + S::kEpiOff + (warp - 4) * S::kEpiWarpBytes);
        const int row_base = mt * HBM_ + q * 32;
        float* cbase = p.C + (size_t)sp * p.split_stride + (size_t)row_base * p.ldc;
#pragma unroll
        for (int cc = 0; cc < HALF / 32; ++cc) {
#pragma unroll
          for (int j = 0; j < 32; ++j) stage[lane * 33 + j] = acc[cc * 32 + j];
          __syncwarp();
          const int col = col0 + cc * 32 + lane;
          if (col < p.N) {
#pragma unroll 8
            for (int rr = 0; rr < 32; ++rr)
              if (row_base + rr < p.M) cbase[(size_t)rr * p.ldc + col] = stage[rr * 33 + lane];
          }
          __syncwarp();
        }
      }
      if (p.amax_out) {
        for (int o = 16; o > 0; o >>= 1) row_amax = fmaxf(row_amax, __shfl_xor_sync(0xffffffffu, row_amax, o));
        if (lane == 0 && row_amax > 0.f) atomicMax(p.amax_out, __float_as_uint(row_amax));
      }
    }
  }

  if (warp >= 4 && lane == 0) bulk_wait();                                                // this lane's bulk stores have landed
  tc_fence_before();
  if constexpr (CTAS == 2) {
    cluster_sync();           // both CTAs have drained their TMEM and sent their last arrivals to the leader
    if (warp == 2) {
      tc_fence_after();
      tmem_dealloc_pair(tmem_base, kTmemCols);
    }
  } else {
    __syncthreads();
    if (warp == 2) {
      tc_fence_after();
      tmem_dealloc(tmem_base, kTmemCols);
    }
  }
}

__global__ void f16_splitk_reduce_kernel(const float* __restrict__ ws, int splits, size_t split_stride, int M, int N,
                                         float* __restrict__ C, int ldc, const float* __restrict__ a_inv, int a_split,
                                         const float* __restrict__ b_inv, int b_split) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)M * N) return;
  float s = 0.f;
  for (int z = 0; z < splits; ++z) s += ws[(size_t)z * split_stride + idx];
  const int m = (int)(idx / N), n = (int)(idx - (size_t)m * N);
  const float f = (a_inv ? a_inv[m >= a_split ? 1 : 0] : 1.f) * (b_inv ? b_inv[n >= b_split ? 1 : 0] : 1.f);
  C[(size_t)m * ldc + n] = s * f;
}

// CTA pairs of this instantiation that fit on the device at once (how the GPCs divide the SMs decides it, not just
// sm_count / 2); sets the kernel's shared-memory limit on the way.  Per device; 0 when the query fails.
template <int BN, int TBK, bool A_KM, bool B_KM>
int resident_pairs_h() {
  constexpr int CTAS = 2;
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  if (dev >= 0 && dev < 64 && cached[dev]) return cached[dev];
  using S = HSmem<BN, TBK, A_KM, B_KM, CTAS>;
  auto kern = gemm3x_f16_kernel<BN, TBK, A_KM, B_KM, CTAS>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, S::kTotal) != cudaSuccess) return 0;
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeClusterDimension;
  attr.val.clusterDim.x = CTAS; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(CTAS * sm_count());
  cfg.blockDim = dim3(kHThreads);
  cfg.dynamicSmemBytes = S::kTotal;
  cfg.attrs = &attr;
  cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess || n <= 0) return 0;
  if (dev >= 0 && dev < 64) cached[dev] = n;
  return n;
}

template <int BN, int TBK, bool A_KM, bool B_KM, int CTAS>
int launch_h(const CUtensorMap& tAh, const CUtensorMap& tAl, const CUtensorMap& tBh, const CUtensorMap& tBl,
             const CUtensorMap& tC, const HParams& p, cudaStream_t st) {
  using S = HSmem<BN, TBK, A_KM, B_KM, CTAS>;
  auto kern = gemm3x_f16_kernel<BN, TBK, A_KM, B_KM, CTAS>;
  int slots;                 // resident work-item slots: CTA pairs or single CTAs
  if constexpr (CTAS == 2) {
    slots = resident_pairs_h<BN, TBK, A_KM, B_KM>();
    if (slots <= 0) {
      cudaGetLastError();
      return fail(SPOTV2_ERR_CUDA, "gemm3x_f16: no cluster of two CTAs with %d B of shared memory fits on this device", S::kTotal);
    }
  } else {
    SPOTV2_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, S::kTotal));
    slots = sm_count();
  }
  const int total = p.pm_tiles * p.n_tiles * p.splits;
  if (slots > total) slots = total;
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeClusterDimension;
  attr.val.clusterDim.x = CTAS; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(CTAS * slots);
  cfg.blockDim = dim3(kHThreads);
  cfg.dynamicSmemBytes = S::kTotal;
  cfg.stream = st;
  cfg.attrs = &attr;
  cfg.numAttrs = CTAS == 2 ? 1 : 0;
  SPOTV2_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, tAh, tAl, tBh, tBl, tC, p));
  return SPOTV2_OK;
}

// ---- operand preparation ------------------------------------------------------------------------------
// Scale block (8 floats per operand): [0,1] bit patterns of the group maxima of |x * pre|, [2,3] inverse
// scales, [4,5] scales.
__device__ __forceinline__ float scale_from_amax(float amax) {
  if (!(amax > 0.f) || !(amax < INFINITY)) return 1.f;
  int ex;
  frexpf(amax, &ex);                         // amax = m * 2^ex, m in [0.5, 1)
  return exp2f((float)(15 - ex));            // amax * scale in [2^14, 2^15)
}

__global__ void amax_kernel(const float* __restrict__ src, int rows, int cols, size_t ld, int split_dim, int split_at,
                            const float* __restrict__ pre2, int pre_split, unsigned* __restrict__ out_bits) {
  float m0 = 0.f, m1 = 0.f;
  const size_t total = (size_t)rows * cols;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(idx / cols), c = (int)(idx - (size_t)r * cols);
    float v = fabsf(src[(size_t)r * ld + c]);
    if (pre2) v *= pre2[r >= pre_split ? 1 : 0];
    const bool g1 = (split_dim == 0 ? r : c) >= split_at;
    if (g1) m1 = fmaxf(m1, v); else m0 = fmaxf(m0, v);
  }
  for (int o = 16; o > 0; o >>= 1) {
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, o));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, o));
  }
  if ((threadIdx.x & 31) == 0) {
    if (m0 > 0.f) atomicMax(out_bits, __float_as_uint(m0));
    if (m1 > 0.f) atomicMax(out_bits + 1, __float_as_uint(m1));
  }
}

// hi = fp16(x * pre * s), lo = fp16(x * pre * s - hi); s from the group maxima (optionally widened by bound).
__global__ void split_f16_kernel(const float* __restrict__ src, int rows, int cols, size_t ld, int split_dim,
                                 int split_at, const float* __restrict__ pre2, int pre_split, float bound,
                                 __half* __restrict__ hi, __half* __restrict__ lo, size_t ld16, float* __restrict__ blk,
                                 int vec4) {
  const unsigned* bits = reinterpret_cast<const unsigned*>(blk);
  const float s0 = scale_from_amax(__uint_as_float(bits[0]) * bound);
  const float s1 = scale_from_amax(__uint_as_float(bits[1]) * bound);
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    blk[2] = 1.f / s0; blk[3] = 1.f / s1; blk[4] = s0; blk[5] = s1;
  }
  auto conv = [&](float x, int r, int c, __half& h, __half& l) {
    if (pre2) x *= pre2[r >= pre_split ? 1 : 0];
    x *= ((split_dim == 0 ? r : c) >= split_at) ? s1 : s0;
    h = __float2half_rn(x);
    l = __float2half_rn(x - __half2float(h));
  };
  if (vec4) {
    const int c4 = cols / 4;
    const size_t total = (size_t)rows * c4;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
      const int r = (int)(idx / c4), c = 4 * (int)(idx - (size_t)r * c4);
      const float4 v = *reinterpret_cast<const float4*>(src + (size_t)r * ld + c);
      __half h[4], l[4];
      conv(v.x, r, c, h[0], l[0]); conv(v.y, r, c + 1, h[1], l[1]);
      conv(v.z, r, c + 2, h[2], l[2]); conv(v.w, r, c + 3, h[3], l[3]);
      *reinterpret_cast<uint2*>(hi + (size_t)r * ld16 + c) = *reinterpret_cast<uint2*>(h);
      *reinterpret_cast<uint2*>(lo + (size_t)r * ld16 + c) = *reinterpret_cast<uint2*>(l);
    }
  } else {
    const size_t total = (size_t)rows * cols;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
      const int r = (int)(idx / cols), c = (int)(idx - (size_t)r * cols);
      __half h, l;
      conv(src[(size_t)r * ld + c], r, c, h, l);
      hi[(size_t)r * ld16 + c] = h;
      lo[(size_t)r * ld16 + c] = l;
    }
  }
}

// vec4 fast path: a block walks groups of four rows (grid stride), no index division; every thread has four 16-byte
// loads in flight (one per row) before it converts, 8-byte stores of 4 fp16 values
constexpr int kSplitRows = 4;
__global__ void __launch_bounds__(256)
split_f16_rows_kernel(const float* __restrict__ src, int rows, int cols4, size_t ld, int split_dim, int split_at,
                      const float* __restrict__ pre2, int pre_split, __half* __restrict__ hi, __half* __restrict__ lo,
                      size_t ld16, float* __restrict__ blk, float* __restrict__ out_blk = nullptr,
                      const float* __restrict__ x_blk = nullptr) {
  const unsigned* bits = reinterpret_cast<const unsigned*>(blk);
  const float s0 = scale_from_amax(__uint_as_float(bits[0])), s1 = scale_from_amax(__uint_as_float(bits[1]));
  if (blockIdx.x == 0 && threadIdx.x == 0) { blk[2] = 1.f / s0; blk[3] = 1.f / s1; blk[4] = s0; blk[5] = s1; }
  // optional: finish the scale block of a pair OUTPUT whose [0,1] hold the row-L1 maxima of this matrix (w_stats_kernel)
  if (out_blk && blockIdx.x == 0 && threadIdx.x >= 32 && threadIdx.x < 34) {
    const int gq = threadIdx.x - 32;
    const float xmax = __uint_as_float(reinterpret_cast<const unsigned*>(x_blk)[0]);
    const float bound = xmax * __uint_as_float(reinterpret_cast<const unsigned*>(out_blk)[gq]) * 1.0009765625f;
    const float so = scale_from_amax(bound);
    out_blk[gq] = bound; out_blk[2 + gq] = 1.f / so; out_blk[4 + gq] = so;
  }
  for (int r0 = blockIdx.x * kSplitRows; r0 < rows; r0 += gridDim.x * kSplitRows) {
    for (int c4 = threadIdx.x; c4 < cols4; c4 += 256) {
      float4 v[kSplitRows];
#pragma unroll
      for (int k = 0; k < kSplitRows; ++k)
        if (r0 + k < rows) v[k] = ldg_stream4(src + (size_t)(r0 + k) * ld + 4 * (size_t)c4);
#pragma unroll
      for (int k = 0; k < kSplitRows; ++k) {
        const int r = r0 + k;
        if (r >= rows) break;
        const float pre = pre2 ? pre2[r >= pre_split ? 1 : 0] : 1.f;
        const float row_scale = pre * ((split_dim == 0 && r >= split_at) ? s1 : s0);
        float sc[4] = {row_scale, row_scale, row_scale, row_scale};
        if (split_dim == 1) {
#pragma unroll
          for (int e = 0; e < 4; ++e) sc[e] = pre * ((4 * c4 + e >= split_at) ? s1 : s0);
        }
        const float x0 = v[k].x * sc[0], x1 = v[k].y * sc[1], x2 = v[k].z * sc[2], x3 = v[k].w * sc[3];
        const __half2 h01 = __floats2half2_rn(x0, x1), h23 = __floats2half2_rn(x2, x3);
        const float2 b01 = __half22float2(h01), b23 = __half22float2(h23);
        const __half2 l01 = __floats2half2_rn(x0 - b01.x, x1 - b01.y), l23 = __floats2half2_rn(x2 - b23.x, x3 - b23.y);
        reinterpret_cast<uint2*>(hi + (size_t)r * ld16)[c4] =
            make_uint2(*reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23));
        reinterpret_cast<uint2*>(lo + (size_t)r * ld16)[c4] =
            make_uint2(*reinterpret_cast<const uint32_t*>(&l01), *reinterpret_cast<const uint32_t*>(&l23));
      }
    }
  }
}

// Narrow matrices (a few float4 per row, e.g. the ds|dd block [B*N, 2H]): one thread per (row, float4), flat index.
__global__ void __launch_bounds__(256)
split_f16_narrow_kernel(const float* __restrict__ src, int rows, int cols4, size_t ld, int split_dim, int split_at,
                        const float* __restrict__ pre2, int pre_split, __half* __restrict__ hi, __half* __restrict__ lo,
                        size_t ld16, float* __restrict__ blk) {
  const unsigned* bits = reinterpret_cast<const unsigned*>(blk);
  const float s0 = scale_from_amax(__uint_as_float(bits[0])), s1 = scale_from_amax(__uint_as_float(bits[1]));
  if (blockIdx.x == 0 && threadIdx.x == 0) { blk[2] = 1.f / s0; blk[3] = 1.f / s1; blk[4] = s0; blk[5] = s1; }
  const size_t total = (size_t)rows * cols4;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(idx / cols4), c4 = (int)(idx - (size_t)r * cols4);
    const float4 v = ldg_stream4(src + (size_t)r * ld + 4 * (size_t)c4);
    const float pre = pre2 ? pre2[r >= pre_split ? 1 : 0] : 1.f;
    const float row_scale = pre * ((split_dim == 0 && r >= split_at) ? s1 : s0);
    float sc[4] = {row_scale, row_scale, row_scale, row_scale};
    if (split_dim == 1) {
#pragma unroll
      for (int e = 0; e < 4; ++e) sc[e] = pre * ((4 * c4 + e >= split_at) ? s1 : s0);
    }
    const float x0 = v.x * sc[0], x1 = v.y * sc[1], x2 = v.z * sc[2], x3 = v.w * sc[3];
    const __half2 h01 = __floats2half2_rn(x0, x1), h23 = __floats2half2_rn(x2, x3);
    const float2 b01 = __half22float2(h01), b23 = __half22float2(h23);
    const __half2 l01 = __floats2half2_rn(x0 - b01.x, x1 - b01.y), l23 = __floats2half2_rn(x2 - b23.x, x3 - b23.y);
    reinterpret_cast<uint2*>(hi + (size_t)r * ld16)[c4] =
        make_uint2(*reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23));
    reinterpret_cast<uint2*>(lo + (size_t)r * ld16)[c4] =
        make_uint2(*reinterpret_cast<const uint32_t*>(&l01), *reinterpret_cast<const uint32_t*>(&l23));
  }
}

}  // namespace

__global__ void amax_flat_kernel(const float* __restrict__ src, size_t n, unsigned* __restrict__ out_bits) {
  float m = 0.f;
  const size_t n4 = n / 4;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(src)[i];
    m = fmaxf(m, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
  }
  if (blockIdx.x == 0 && threadIdx.x == 0)
    for (size_t k = n4 * 4; k < n; ++k) m = fmaxf(m, fabsf(src[k]));
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(out_bits, __float_as_uint(m));
}

// ---- scale of a pair OUTPUT, known before the product runs ---------------------------------------------
// |sum_k x[i,k] W[j,k]| <= max|x| * ||W[j,:]||_1.  One warp per row of W; bits[g] <- max over the rows of group g
// (rows < / >= split_at) of the row's L1 norm (atomicMax on the bit pattern: all values are >= 0).
__global__ void __launch_bounds__(256)
row_l1_max_kernel(const float* __restrict__ W, int rows, int cols, int split_at, unsigned* __restrict__ bits) {
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float* w = W + (size_t)r * cols;
  float s = 0.f;
  for (int c = lane; c < cols; c += 32) s += fabsf(w[c]);
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0 && s > 0.f) atomicMax(bits + (r >= split_at ? 1 : 0), __float_as_uint(s));
}
// blk: [0,1] hold the row-L1 maxima (bits) on entry; on exit [0,1] = bits of the bounds max|x| * L1 * (1 + 2^-10),
// [2,3] inverse scales, [4,5] scales (power of two: bound * scale in [2^14, 2^15))
__global__ void pair_out_scale_kernel(float* blk, const float* __restrict__ x_blk) {
  if (threadIdx.x >= 2) return;
  const float xmax = __uint_as_float(reinterpret_cast<const unsigned*>(x_blk)[0]);
  const float l1 = __uint_as_float(reinterpret_cast<const unsigned*>(blk)[threadIdx.x]);
  const float bound = xmax * l1 * 1.0009765625f;
  const float s = scale_from_amax(bound);
  blk[threadIdx.x] = bound;
  blk[2 + threadIdx.x] = 1.f / s;
  blk[4 + threadIdx.x] = s;
}

// One pass over W [rows, cols]: per group (rows < / >= split_at) the largest magnitude (-> amax_bits[g], sizes W's own operand
// scale) and the largest row L1 norm (-> l1_bits[g], bounds the pair output).  One warp per row.
__global__ void __launch_bounds__(256)
w_stats_kernel(const float* __restrict__ W, int rows, int cols, int split_at, unsigned* __restrict__ amax_bits, unsigned* __restrict__ l1_bits) {
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float* w = W + (size_t)r * cols;
  float s = 0.f, m = 0.f;
  for (int c = lane; c < cols; c += 32) {
    const float a = fabsf(w[c]);
    s += a;
    m = fmaxf(m, a);
  }
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  }
  if (lane == 0) {
    const int gq = r >= split_at ? 1 : 0;
    if (s > 0.f) atomicMax(l1_bits + gq, __float_as_uint(s));
    if (m > 0.f) atomicMax(amax_bits + gq, __float_as_uint(m));
  }
}

// W_aug [rows, cols] -> its fp16 operand pair (two row groups at split_at) AND the scale block of the pair output x . W^T, in
// two launches (statistics, split); falls back to split_f16 + pair_out_scale when the vectorised split does not apply.
int w_pair_and_out_scale(const float* W, int rows, int cols, int split_at, void* hi, void* lo, size_t ld16, float* wblk,
                         const float* x_blk, float* out_blk, cudaStream_t st) {
  const bool vec4 = (cols % 4 == 0) && (ld16 % 4 == 0) && aligned16(W) && ((reinterpret_cast<uintptr_t>(hi) & 7) == 0) &&
                    ((reinterpret_cast<uintptr_t>(lo) & 7) == 0) && cols / 4 >= 64;
  if (!vec4) {
    if (int rc = split_f16(W, rows, cols, (size_t)cols, 0, split_at, nullptr, 0, hi, lo, ld16, wblk, st)) return rc;
    return pair_out_scale(W, rows, cols, split_at, x_blk, out_blk, st);
  }
  SPOTV2_CUDA_OK(cudaMemsetAsync(wblk, 0, kScaleBlockFloats * sizeof(float), st));
  SPOTV2_CUDA_OK(cudaMemsetAsync(out_blk, 0, kScaleBlockFloats * sizeof(float), st));
  w_stats_kernel<<<(rows + 7) / 8, 256, 0, st>>>(W, rows, cols, split_at, reinterpret_cast<unsigned*>(wblk), reinterpret_cast<unsigned*>(out_blk));
  split_f16_rows_kernel<<<std::min((rows + kSplitRows - 1) / kSplitRows, 32 * 148), 256, 0, st>>>(
      W, rows, cols / 4, (size_t)cols, 0, split_at, nullptr, 0, static_cast<__half*>(hi), static_cast<__half*>(lo), ld16, wblk, out_blk, x_blk);
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

int pair_out_scale(const float* W, int rows, int cols, int split_at, const float* x_blk, float* blk, cudaStream_t st) {
  SPOTV2_CUDA_OK(cudaMemsetAsync(blk, 0, kScaleBlockFloats * sizeof(float), st));
  row_l1_max_kernel<<<(rows + 7) / 8, 256, 0, st>>>(W, rows, cols, split_at, reinterpret_cast<unsigned*>(blk));
  pair_out_scale_kernel<<<1, 32, 0, st>>>(blk, x_blk);
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

int amax_flat(const float* src, size_t n, float* blk, cudaStream_t st) {
  SPOTV2_CUDA_OK(cudaMemsetAsync(blk, 0, 8 * sizeof(float), st));
  const bool al = aligned16(src);
  const size_t work = al ? n / 4 : 0;
  if (!al) {        // rare: unaligned view; fall back to the generic kernel as a 1 x n matrix
    amax_kernel<<<(unsigned)std::min<size_t>((n + 255) / 256, 4096), 256, 0, st>>>(src, 1, (int)n, n, 0, 1 << 30, nullptr, 0,
                                                                                  reinterpret_cast<unsigned*>(blk));
  } else {
    amax_flat_kernel<<<(unsigned)std::min<size_t>((std::max<size_t>(work, 1) + 255) / 256, 8 * 148), 256, 0, st>>>(
        src, n, reinterpret_cast<unsigned*>(blk));
  }
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

int amax_2d(const float* src, int rows, int cols, size_t ld, float* blk, cudaStream_t st) {
  SPOTV2_CUDA_OK(cudaMemsetAsync(blk, 0, 8 * sizeof(float), st));
  const size_t total = (size_t)rows * cols;
  const unsigned blocks = (unsigned)std::min<size_t>((total + 1023) / 1024, 16 * 148);
  amax_kernel<<<blocks, 256, 0, st>>>(src, rows, cols, ld, 0, 0x7fffffff, nullptr, 0, reinterpret_cast<unsigned*>(blk));
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

static int launch_amax_flat(const float* src, size_t n, unsigned* out, cudaStream_t st) {
  if (n == 0) return SPOTV2_OK;
  amax_flat_kernel<<<(unsigned)std::min<size_t>((n / 4 + 255) / 256 + 1, 8 * 148), 256, 0, st>>>(src, n, out);
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

int split_f16(const float* src, int rows, int cols, size_t ld, int split_dim, int split_at, const float* pre2,
              int pre_split, void* hi, void* lo, size_t ld16, float* blk, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return SPOTV2_OK;
  SPOTV2_CUDA_OK(cudaMemsetAsync(blk, 0, 8 * sizeof(float), st));
  const size_t total = (size_t)rows * cols;
  const unsigned blocks = (unsigned)std::min<size_t>((total + 1023) / 1024, 16 * 148);
  unsigned* bits = reinterpret_cast<unsigned*>(blk);
  // group maxima: contiguous row ranges go through the vectorised flat kernel
  const bool flat_ok = !pre2 && ld == (size_t)cols && aligned16(src) && (split_dim == 0 || split_at >= cols);
  if (flat_ok) {
    const int r_split = (split_dim == 0 && split_at < rows) ? (split_at > 0 ? split_at : 0) : rows;
    const bool second_aligned = ((size_t)r_split * cols) % 4 == 0;
    if (r_split < rows && !second_aligned) {
      amax_kernel<<<blocks, 256, 0, st>>>(src, rows, cols, ld, split_dim, split_at, pre2, pre_split, bits);
    } else {
      if (int rc = launch_amax_flat(src, (size_t)r_split * cols, bits, st)) return rc;
      if (r_split < rows)
        if (int rc = launch_amax_flat(src + (size_t)r_split * cols, (size_t)(rows - r_split) * cols, bits + 1, st)) return rc;
    }
  } else {
    amax_kernel<<<blocks, 256, 0, st>>>(src, rows, cols, ld, split_dim, split_at, pre2, pre_split, bits);
  }
  const int vec4 = (cols % 4 == 0) && (ld % 4 == 0) && (ld16 % 4 == 0) && aligned16(src) &&
                   ((reinterpret_cast<uintptr_t>(hi) & 7) == 0) && ((reinterpret_cast<uintptr_t>(lo) & 7) == 0);
  if (vec4 && cols / 4 < 64)
    split_f16_narrow_kernel<<<(unsigned)std::min<size_t>(((size_t)rows * (cols / 4) + 255) / 256, (size_t)16 * 148), 256, 0, st>>>(
        src, rows, cols / 4, ld, split_dim, split_at, pre2, pre_split, static_cast<__half*>(hi), static_cast<__half*>(lo), ld16, blk);
  else if (vec4)
    split_f16_rows_kernel<<<std::min((rows + kSplitRows - 1) / kSplitRows, 32 * 148), 256, 0, st>>>(
        src, rows, cols / 4, ld, split_dim, split_at, pre2, pre_split, static_cast<__half*>(hi), static_cast<__half*>(lo), ld16, blk);
  else
    split_f16_kernel<<<blocks, 256, 0, st>>>(src, rows, cols, ld, split_dim, split_at, pre2, pre_split, 1.f,
                                             static_cast<__half*>(hi), static_cast<__half*>(lo), ld16, blk, 0);
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

// The weight-gradient product's kernel (MN-major x MN-major, 256 x 256 x 32 pair tiles) sizes the split-K factor.
int gemm3x_f16_resident_pairs() {
  const int n = resident_pairs_h<256, 32, false, false>();
  if (n > 0) return n;
  cudaGetLastError();
  return sm_count() / 2;      // no device: the pairs of a B200's 148 SMs
}

// C[M,N] = A . B^T with operands pre-split into scaled fp16 pairs.  bn: 256 -> TBK 64, 256 + 16 -> TBK 32.
// The 3-product (fp32-accurate) class runs on pair tiles; the single-product half-precision class keeps 1-CTA tiles: with
// a third of the MMA work per k-block it is bound by its operand pipeline, which the cross-CTA hand-offs lengthen (config C
// half mode on a B200: forward 2.17 -> 2.51 ms, dW 1.73 -> 2.29, dX 1.09 -> 1.34 on pair tiles; profiles/r3a_pair_gemm_ab.txt).
int gemm3x_f16(bool a_kc, bool b_kc, int M, int N, int K, const F16Operand& A, const F16Operand& B, float* C, int ldc,
               int splits, int bn, int kb_per_chunk, void* ws, size_t ws_bytes, cudaStream_t st, float* amax_out,
               int amax_cols, bool single, const PairOut* pair) {
  const int TBK = (bn & 16) ? 32 : 64;
  bn &= ~16;
  if (!tma_available()) return fail(SPOTV2_ERR_NO_DEVICE, "tensor-core GEMM: TMA descriptor encoding is not available");
  if (A.ld % 8 != 0 || B.ld % 8 != 0 || !aligned16(A.hi) || !aligned16(A.lo) || !aligned16(B.hi) || !aligned16(B.lo))
    return fail(SPOTV2_ERR_INVALID_ARG, "fp16 GEMM operands need 16-byte aligned bases and leading dimensions % 8 == 0");
  HParams p;
  p.M = M; p.N = N; p.K = K;
  const int ctas = single ? 1 : 2;
  p.pm_tiles = (M + ctas * HBM_ - 1) / (ctas * HBM_);
  p.n_tiles = (N + bn - 1) / bn;
  p.kb_total = (K + TBK - 1) / TBK;
  if (splits < 1) splits = 1;
  if (splits > p.kb_total) splits = p.kb_total;
  p.kb_per_split = (p.kb_total + splits - 1) / splits;
  p.splits = (p.kb_total + p.kb_per_split - 1) / p.kb_per_split;
  p.kb_per_chunk = kb_per_chunk < 1 ? 128 / TBK : kb_per_chunk;
  p.C = C; p.ldc = ldc; p.split_stride = 0;
  p.a_inv = A.inv; p.b_inv = B.inv; p.a_split = A.split_at; p.b_split = B.split_at;
  p.scale_in_kernel = 1;
  p.amax_out = reinterpret_cast<unsigned*>(amax_out);
  p.amax_cols = amax_cols;
  p.single = single ? 1 : 0;
  p.pair_out = 0; p.out_scale = nullptr; p.tail32 = nullptr; p.tail_ld = 0;
  if (pair) {
    if (splits > 1 || !pair->hi || !pair->scale || pair->ld % 8 != 0 || !aligned16(pair->hi) || (pair->lo && !aligned16(pair->lo)))
      return fail(SPOTV2_ERR_INVALID_ARG, "gemm3x_f16: pair output needs splits == 1, 16-byte aligned planes, ld %% 8 == 0 and a scale");
    p.pair_out = pair->lo ? 1 : 2;
    p.out_scale = pair->scale;
    p.tail32 = pair->tail32; p.tail_ld = pair->tail_ld;
  }
  p.dbg = 0;
#ifdef SPOTV2_BRINGUP
  {
    // bring-up probe (tools/gemm_fill_probe.py): skips parts of the epilogue to time them; results are WRONG when set
    static const int dbg = [] {
      const char* e = getenv("SPOTV2_GEMM_DBG");
      const int v = e ? atoi(e) : 0;
      if (v) fprintf(stderr, "libspotv2_gat: SPOTV2_GEMM_DBG=%d - timing probe active, GEMM results are invalid\n", v);
      return v;
    }();
    p.dbg = dbg;
  }
#endif
  if (amax_out) {
    if (splits > 1) return fail(SPOTV2_ERR_INVALID_ARG, "gemm3x_f16: amax_out needs splits == 1");
    SPOTV2_CUDA_OK(cudaMemsetAsync(amax_out, 0, sizeof(float), st));
  }
  if (p.splits > 1) {
    const size_t need = (size_t)p.splits * M * N * sizeof(float);
    if (!ws || ws_bytes < need)
      return fail(SPOTV2_ERR_WORKSPACE, "split-K tensor-core GEMM needs %zu B of workspace, got %zu", need, ws_bytes);
    p.C = static_cast<float*>(ws); p.ldc = N; p.split_stride = (size_t)M * N;
    p.scale_in_kernel = 0;
  }
  CUtensorMap tAh, tAl, tBh, tBl, tC;
  int rc;
  memset(&tC, 0, sizeof(tC));
  p.tma_store = 0;
  if (pair) {
    // planes [hi, lo] of [M, ld] fp16; 32 x 32 boxes with 64-byte rows
    const uint64_t plane_stride = pair->lo ? (uint64_t)((const __half*)pair->lo - (const __half*)pair->hi) : (uint64_t)M * pair->ld;
    if (pair->lo && ((const __half*)pair->lo <= (const __half*)pair->hi || plane_stride % 8 != 0))
      return fail(SPOTV2_ERR_INVALID_ARG, "gemm3x_f16: the lo plane must follow the hi plane at a multiple of 16 bytes");
    if ((rc = make_tmap3_f16(&tC, pair->hi, pair->lo ? 2 : 1, plane_stride, (uint64_t)M, (uint64_t)N, (uint64_t)pair->ld, 32, 32,
                             CU_TENSOR_MAP_SWIZZLE_64B)))
      return rc;
  } else if (aligned16(p.C) && p.ldc % 4 == 0 && (p.splits == 1 || p.split_stride % 4 == 0)) {
    // C tiles (or split-K partials: plane = split) through TMA bulk stores: 32-row x 16-column fp32 boxes, 64B swizzle
    if ((rc = make_tmap3(&tC, p.C, (uint64_t)p.splits, p.splits > 1 ? p.split_stride : (uint64_t)M * p.ldc, (uint64_t)M, (uint64_t)N,
                         (uint64_t)p.ldc, 16, 32, CU_TENSOR_MAP_SWIZZLE_64B)))
      return rc;
    p.tma_store = 1;
  }
  // K-major operand: tensor [rows = M|N, cols = K], box TBK(k) x this CTA's tile rows (128 of A, bn / ctas of B; rows of
  // 128 or 64 bytes).  MN-major operand: tensor [rows = K, cols = M|N], box 64(m|n) x TBK(k); one box per 64-wide block.
  const CUtensorMapSwizzle kSw = TBK == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  const CUtensorMapSwizzle mnSw = CU_TENSOR_MAP_SWIZZLE_128B;
  if (a_kc) {
    if ((rc = make_tmap_f16(&tAh, A.hi, M, K, A.ld, TBK, HBM_, kSw))) return rc;
    if ((rc = make_tmap_f16(&tAl, A.lo, M, K, A.ld, TBK, HBM_, kSw))) return rc;
  } else {
    if ((rc = make_tmap_f16(&tAh, A.hi, K, M, A.ld, 64, TBK, mnSw))) return rc;
    if ((rc = make_tmap_f16(&tAl, A.lo, K, M, A.ld, 64, TBK, mnSw))) return rc;
  }
  if (b_kc) {
    if ((rc = make_tmap_f16(&tBh, B.hi, N, K, B.ld, TBK, bn / ctas, kSw))) return rc;
    if ((rc = make_tmap_f16(&tBl, B.lo, N, K, B.ld, TBK, bn / ctas, kSw))) return rc;
  } else {
    if ((rc = make_tmap_f16(&tBh, B.hi, K, N, B.ld, 64, TBK, mnSw))) return rc;
    if ((rc = make_tmap_f16(&tBl, B.lo, K, N, B.ld, 64, TBK, mnSw))) return rc;
  }
#define SPOTV2_H(BN_, TBK_, AK, BK_) \
  rc = single ? launch_h<BN_, TBK_, AK, BK_, 1>(tAh, tAl, tBh, tBl, tC, p, st) : launch_h<BN_, TBK_, AK, BK_, 2>(tAh, tAl, tBh, tBl, tC, p, st)
#define SPOTV2_H_MAJ(BN_, TBK_)                            \
  do {                                                     \
    if (a_kc && b_kc) SPOTV2_H(BN_, TBK_, true, true);     \
    else if (a_kc) SPOTV2_H(BN_, TBK_, true, false);       \
    else if (b_kc) SPOTV2_H(BN_, TBK_, false, true);       \
    else SPOTV2_H(BN_, TBK_, false, false);                \
  } while (0)
  if (bn == 256 && TBK == 64) SPOTV2_H_MAJ(256, 64);
  else if (bn == 256 && TBK == 32) SPOTV2_H_MAJ(256, 32);
  else if (bn == 128 && TBK == 64) SPOTV2_H_MAJ(128, 64);
  else return fail(SPOTV2_ERR_INVALID_ARG, "bn must be 128, 256 or 256+16");
#undef SPOTV2_H_MAJ
#undef SPOTV2_H
  if (rc) return rc;
  if (p.splits > 1) {
    const size_t total = (size_t)M * N;
    f16_splitk_reduce_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(p.C, p.splits, p.split_stride, M, N, C, ldc,
                                                                             A.inv, A.split_at, B.inv, B.split_at);
    SPOTV2_CUDA_OK(cudaGetLastError());
  }
  return SPOTV2_OK;
}

}  // namespace spotv2
