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
//                         tiles (24-slot ring), running ahead across graphs.
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
constexpr int kPSlots = 24;           // P-tile ring depth
constexpr int kPTileBytes = 32 * 128; // 32 source rows x 32 channels fp32, 128B-swizzled
constexpr int kCbPerPass = 8;         // channel blocks per pass: one per MMA warp

// wait-cycle diagnostics of this kernel (see spotv2_diag_counters)
__device__ unsigned long long g_diag_counters[kNumCounters];

// FIX: the reference's default geometry (N=30, H=6, C=500, Fe=126, head mean, PyG edge order) as compile-time
// constants, so index arithmetic folds and the parameter block is not re-read inside the hot loops.
template <int NPAIRS, bool VEC2, bool FIX>
__global__ void __launch_bounds__(kFwdThreads, 1)
gat_attn_fwd_kernel(const AttnFwdArgs args, const AttnSmem sm_, const uint32_t off_ptile,
                    const __grid_constant__ CUtensorMap tmP) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  AttnParams p = args.p;
  AttnSmem sm = sm_;
  if (FIX) {
    p.N = 30; p.H = 6; p.C = 500; p.Fe = 126; p.R = 870; p.concat = 0; p.ldp = 3012; p.ldo = 500; p.bulk_ok = 1; p.vec2_ok = 1;
    sm.NS = 36; sm.KS = 16; sm.NT = 1; sm.chunk_rows = kFwdChunkRows3;
  }
  const int tid = threadIdx.x;
  const int N = p.N, H = p.H, C = p.C, NS = sm.NS;
  const int HC = H * C;
  const int tile_floats = H * N * NS;
  const int sd_floats = N * 2 * H;

  // [0,1] edge ring, [2,3] tile_full, [4,5] tile_empty, [6..6+kPSlots) ptile_full, then ptile_empty
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + sm.off_bar);
  uint64_t* tile_full = bars + 2;
  uint64_t* tile_empty = bars + 4;
  uint64_t* ptile_full = bars + 6;
  uint64_t* ptile_empty = bars + 6 + kPSlots;
  uint64_t* sd_full = bars + 6 + 2 * kPSlots;          // [2] s|d tile landed
  uint64_t* sd_empty = sd_full + 2;                     // [2] s|d tile consumed
  const uint32_t off_sdtile = off_ptile + kPSlots * kPTileBytes;
  const int n_cb = (C + 31) / 32;                                   // 32-channel blocks per head
  const int n_pass = (n_cb + kCbPerPass - 1) / kCbPerPass;
  int32_t* table_s = reinterpret_cast<int32_t*>(smem_raw + sm.off_table);
  float4* vfrag = reinterpret_cast<float4*>(smem_raw + sm.off_vfrag);
  float* sd0 = reinterpret_cast<float*>(smem_raw + sm.off_sd);
  float* tile0 = reinterpret_cast<float*>(smem_raw + sm.off_tile);

  const int nchunks = (p.Fe > 0 && !p.terms_in) ? (p.R + sm.chunk_rows - 1) / sm.chunk_rows : 0;
  const int my_graphs = (p.B - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    mbar_init(&tile_full[0], kGroupA);
    mbar_init(&tile_full[1], kGroupA);
    mbar_init(&tile_empty[0], kGroupB);
    mbar_init(&tile_empty[1], kGroupB);
    for (int r = 0; r < kPSlots; ++r) { mbar_init(&ptile_full[r], 1); mbar_init(&ptile_empty[r], 1); }
    for (int r = 0; r < 2; ++r) { mbar_init(&sd_full[r], 1); mbar_init(&sd_empty[r], 1); }
    fence_mbar_init();
  }
  // row -> byte offset of (source j, target i) inside one head of the alpha tile (-1: row skipped)
  for (int r = tid; r < p.R; r += kFwdThreads) {
    const int code = (p.Fe > 0 && !p.terms_in) ? p.table[r] : -1;
    table_s[r] = code >= 0 ? ((code & 0xffff) * NS + (code >> 16)) * 4 : -1;
  }
  // the edge ring starts zero-filled: k-steps padded past Fe and rows past the end of a short chunk read stale
  // bytes (multiplied by zero fragments / discarded), which must be finite numbers
  for (uint32_t idx = tid; idx < (off_ptile - (uint32_t)sm.off_ring) / 16; idx += kFwdThreads)
    reinterpret_cast<float4*>(smem_raw + sm.off_ring)[idx] = make_float4(0.f, 0.f, 0.f, 0.f);
  fence_proxy_async();
  if (p.Fe > 0 && !p.terms_in) build_vfrag(vfrag, p.v, H, p.Fe, sm.KS, sm.NT, tid, kFwdThreads);
  for (int idx = tid; idx < 2 * tile_floats; idx += kFwdThreads) tile0[idx] = 0.f;
  __syncthreads();

  if (tid < kGroupA) {
    // ================================ group A: logits + softmax ================================
    const int warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const uint32_t sbase = smem_u32(smem_raw);
    const uint32_t ring_a[2] = {sbase + (uint32_t)sm.off_ring, sbase + (uint32_t)(sm.off_ring + sm.ring_stage_bytes)};
    const uint32_t a_vfrag = sbase + (uint32_t)sm.off_vfrag, a_table = sbase + (uint32_t)sm.off_table;
    const uint32_t a_tile0 = sbase + (uint32_t)sm.off_tile, head_bytes = (uint32_t)(N * NS * 4);
    float* stage[2] = {reinterpret_cast<float*>(smem_raw + sm.off_ring),
                       reinterpret_cast<float*>(smem_raw + sm.off_ring + sm.ring_stage_bytes)};
    const int total_chunks = my_graphs * nchunks;      // this CTA's global chunk stream
    auto rows_in = [&](int c) { const int r = p.R - c * sm.chunk_rows; return r < sm.chunk_rows ? r : sm.chunk_rows; };
    auto issue = [&](int k) {                           // one thread: start the k-th chunk of the stream
      const int it = k / nchunks, c = k - it * nchunks;
      const int b = blockIdx.x + it * gridDim.x;
      const uint32_t bytes = (uint32_t)rows_in(c) * p.Fe * 4u;
      mbar_expect_tx(&bars[k & 1], bytes);
      bulk_g2s(stage[k & 1], p.edge_rows + ((size_t)b * p.R + (size_t)c * sm.chunk_rows) * p.Fe, bytes, &bars[k & 1]);
    };
    if (p.bulk_ok && tid == 0) {
      if (total_chunks > 0) issue(0);
      if (total_chunks > 1) issue(1);
    }
    int k = 0;                                          // global chunk counter (stage = k & 1, parity = (k >> 1) & 1)
    long long w_ring = 0, w_tile = 0, t_mma = 0, t_call = 0, t_bar = 0;
    const long long t_role = clock64();
    for (int it = 0; it < my_graphs; ++it) {
      const int b = blockIdx.x + it * gridDim.x;
      const int buf = it & 1;
      float* tile = tile0 + buf * tile_floats;
      mbar_wait_timed(&tile_empty[buf], ((it >> 1) & 1) ^ 1, w_tile);   // group B has finished reading this buffer
      if (p.terms_in) {
        // structured edge source: the caller computed the edge terms; one bulk copy drops them into the tile buffer.
        // Thread 0's arrive.expect_tx is its arrival on tile_full; the phase completes when the bytes have landed.
        if (tid == 0) {
          const uint32_t bytes = (uint32_t)tile_floats * 4u;
          mbar_expect_tx(&tile_full[buf], bytes);
          bulk_g2s(tile, p.edge_terms + (size_t)b * tile_floats, bytes, &tile_full[buf]);
        } else {
          mbar_arrive(&tile_full[buf]);
        }
        continue;
      }
      if (nchunks == 0) {
        for (int idx = tid; idx < tile_floats; idx += kGroupA) tile[idx] = 0.f;
      }
      for (int c = 0; c < nchunks; ++c, ++k) {
        const int s = k & 1;
        const int rows = rows_in(c);
        if (p.bulk_ok) {
          mbar_wait_timed(&bars[s], (k >> 1) & 1, w_ring);
        } else {
          const float* src = p.edge_rows + ((size_t)b * p.R + (size_t)c * sm.chunk_rows) * p.Fe;
          for (int idx = tid; idx < rows * p.Fe; idx += kGroupA) stage[s][idx] = src[idx];
          bar_sync<1, kGroupA>();
        }
        const long long tc0 = clock64();
        if (warp * 16 < rows) {
          // 16 rows x all k-steps, 3xTF32, 8 k-steps of loads in flight; no index clamps (see the zero fill above)
          // MMA row g <-> chunk row 2g, g+8 <-> 2g+1: with the 126-float pitch the 8 even (odd) rows start 4 banks apart
          const uint32_t r0 = ring_a[s] + (uint32_t)(((warp * 16 + 2 * g) * p.Fe + t) * 4), r1 = r0 + (uint32_t)(p.Fe * 4);
          float acc[3][4];
#pragma unroll
          for (int pr = 0; pr < 3; ++pr)
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[pr][q] = 0.f;
          for (int ks0 = 0; ks0 < sm.KS; ks0 += 8) {
            const uint32_t ko = (uint32_t)ks0 * 32u, vf = a_vfrag + ((uint32_t)ks0 * 32u + (uint32_t)lane) * 16u;
            float a[8][4];
            float4 bf[8];
#pragma unroll
            for (int sl = 0; sl < 8; ++sl) {
              a[sl][0] = ldsa(r0 + ko + sl * 32);
              a[sl][1] = ldsa(r1 + ko + sl * 32);
              a[sl][2] = ldsa(r0 + ko + sl * 32 + 16);
              a[sl][3] = ldsa(r1 + ko + sl * 32 + 16);
              bf[sl] = lds128a(vf + sl * 512);
            }
#pragma unroll
            for (int sl = 0; sl < 8; ++sl) {
              uint32_t ah[4], al[4];
#pragma unroll
              for (int q = 0; q < 4; ++q) split_lean(a[sl][q], ah[q], al[q]);
              const uint32_t bh[2] = {__float_as_uint(bf[sl].x), __float_as_uint(bf[sl].y)};
              const uint32_t bl[2] = {__float_as_uint(bf[sl].z), __float_as_uint(bf[sl].w)};
              mma_tf32_16x8x8(acc[0], al, bh);
              mma_tf32_16x8x8(acc[1], ah, bl);
              mma_tf32_16x8x8(acc[2], ah, bh);
            }
          }
          const int rl = warp * 16 + 2 * g, row_base = c * sm.chunk_rows + rl;
          const int to0 = rl < rows ? ldsa_s32(a_table + (uint32_t)row_base * 4u) : -1;
          const int to1 = rl + 1 < rows ? ldsa_s32(a_table + (uint32_t)(row_base + 1) * 4u) : -1;
          const uint32_t tb = a_tile0 + (uint32_t)(buf * tile_floats * 4) + (uint32_t)(2 * t) * head_bytes;
          if (to0 >= 0) {
            if (2 * t < H) stsa(tb + (uint32_t)to0, (acc[0][0] + acc[1][0]) + acc[2][0]);
            if (2 * t + 1 < H) stsa(tb + head_bytes + (uint32_t)to0, (acc[0][1] + acc[1][1]) + acc[2][1]);
          }
          if (to1 >= 0) {
            if (2 * t < H) stsa(tb + (uint32_t)to1, (acc[0][2] + acc[1][2]) + acc[2][2]);
            if (2 * t + 1 < H) stsa(tb + head_bytes + (uint32_t)to1, (acc[0][3] + acc[1][3]) + acc[2][3]);
          }
        }
        const long long tc1 = clock64();
        bar_sync<1, kGroupA>();                          // stage s consumed by all three warps
        t_call += tc1 - tc0;
        (void)t_mma;
        t_bar += clock64() - tc1;
        if (p.bulk_ok && tid == 0 && k + 2 < total_chunks) issue(k + 2);
      }
      if (p.edge_terms && !p.terms_in && NS == kEdgeTermNS) {
        // keep the edge terms for the backward (it then reads 6 floats per edge instead of the Fe-wide rows).  All of
        // group A's scatters are behind the chunk loop's last bar.sync; diagonal entries hold stale finite values
        // that no consumer reads.
        if (nchunks == 0) bar_sync<1, kGroupA>();
        float4* dst = reinterpret_cast<float4*>(p.edge_terms + (size_t)b * tile_floats);
        const float4* src = reinterpret_cast<const float4*>(tile);
        for (int idx = tid; idx < tile_floats / 4; idx += kGroupA) dst[idx] = src[idx];
      }
      mbar_arrive(&tile_full[buf]);                      // release: edge terms of this graph visible to group B
    }
    if (tid == 0) {
      atomicAdd(&g_diag_counters[kCntRingFull], (unsigned long long)w_ring);
      atomicAdd(&g_diag_counters[kCntTileEmpty], (unsigned long long)w_tile);
      atomicAdd(&g_diag_counters[kCntRoleA], (unsigned long long)(clock64() - t_role));
      atomicAdd(&g_diag_counters[kCntAux0], (unsigned long long)t_mma);
      atomicAdd(&g_diag_counters[kCntAux1], (unsigned long long)t_call);
      atomicAdd(&g_diag_counters[kCntAux2], (unsigned long long)t_bar);
    }
  } else if (tid < kGroupA + kGroupB) {
    // ================================ group B: aggregation on mma.sync ================================
    const int wb = (tid - kGroupA) >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const uint32_t a_ptiles = smem_u32(smem_raw) + off_ptile;
    // MMA k index t <-> source row 2t, t+4 <-> 2t+1 (alpha fragments below use the same permutation): the 4 x 2
    // chunk slots one fragment load touches in the swizzled tile are then all distinct (no bank conflicts)
    const uint32_t fb_k0 = (uint32_t)((2 * t) * 128 + ((((g >> 2) ^ (2 * t))) << 4) + ((g & 3) << 2));
    const uint32_t fb_k1 = (uint32_t)((2 * t + 1) * 128 + ((((g >> 2) ^ (2 * t + 1))) << 4) + ((g & 3) << 2));
    uint32_t q_base = 0;                                   // tiles issued before the current (pass, head) group
    long long w_tf = 0, w_pf = 0;
    const long long t_role = clock64();
    const float out_scale = p.concat ? 1.f : 1.f / (float)H;
    for (int it = 0; it < my_graphs; ++it) {
      const int b = blockIdx.x + it * gridDim.x;
      const int buf = it & 1;
      float* tile = tile0 + buf * tile_floats;
      mbar_wait_timed(&tile_full[buf], (it >> 1) & 1, w_tf);
      mbar_wait_timed(&sd_full[buf], (it >> 1) & 1, w_tf);
      softmax_phase(p, sm, tile, reinterpret_cast<const float*>(smem_raw + off_sdtile + buf * kPTileBytes), out_scale,
                    args.alpha_out ? args.alpha_out + (size_t)b * H * N * N : nullptr, nullptr, tid - kGroupA, kGroupB,
                    -1, /*sd_swizzled=*/1, nullptr, b);
      bar_sync<2, kGroupB>();                            // alpha tile complete
      if (tid == kGroupA) mbar_arrive(&sd_empty[buf]);
      for (int pass = 0; pass < n_pass; ++pass) {
        const int G = min(kCbPerPass, n_cb - pass * kCbPerPass);     // valid channel blocks in this pass
        const bool mine = wb < G;                          // this warp's channel block: pass * 8 + wb
        const int cb = pass * kCbPerPass + wb;
        // Two accumulator sets (hi*hi products / cross terms) so that consecutive MMAs never wait on each
        // other's ~300-cycle latency; in mean mode they run across all heads (alpha carries the 1/H).
        float cmain[2][4][4], ccorr[2][4][4];
        auto clear = [&]() {
#pragma unroll
          for (int m = 0; m < 2; ++m)
#pragma unroll
            for (int n = 0; n < 4; ++n)
#pragma unroll
              for (int e = 0; e < 4; ++e) cmain[m][n][e] = ccorr[m][n][e] = 0.f;
        };
        auto store = [&](int col0) {                       // out[i, col0 + c] = cmain + ccorr + bias
#pragma unroll
          for (int m = 0; m < 2; ++m)
#pragma unroll
            for (int n = 0; n < 4; ++n)
#pragma unroll
              for (int hf = 0; hf < 2; ++hf) {
                const int i = m * 16 + g + 8 * hf, c = cb * 32 + n * 8 + 2 * t;
                if (i < N && c < C) {
                  const int col = col0 + c;
                  float* dst = args.out + ((size_t)b * N + i) * p.ldo + col;
                  const float o0 = cmain[m][n][2 * hf] + ccorr[m][n][2 * hf] + (args.bias ? args.bias[col] : 0.f);
                  if (c + 1 < C) {
                    const float o1 = cmain[m][n][2 * hf + 1] + ccorr[m][n][2 * hf + 1] + (args.bias ? args.bias[col + 1] : 0.f);
                    if (VEC2) *reinterpret_cast<float2*>(dst) = make_float2(o0, o1);
                    else { dst[0] = o0; dst[1] = o1; }
                  } else {
                    dst[0] = o0;
                  }
                }
              }
        };
        clear();
        for (int h = 0; h < H; ++h, q_base += G) {
          if (!mine) continue;
          // A fragments of alpha_h (rows = targets i, cols = sources j), split once per (pass, head)
          uint32_t ah[2][4][4], al[2][4][4];
#pragma unroll
          for (int m = 0; m < 2; ++m)
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              const int i0 = m * 16 + g, j0 = ks * 8 + 2 * t;
              const float* base = tile + (size_t)h * N * NS;
              const float a0 = (j0 < N) ? base[j0 * NS + i0] : 0.f;
              const float a1 = (j0 < N) ? base[j0 * NS + i0 + 8] : 0.f;
              const float a2 = (j0 + 1 < N) ? base[(j0 + 1) * NS + i0] : 0.f;
              const float a3 = (j0 + 1 < N) ? base[(j0 + 1) * NS + i0 + 8] : 0.f;
              split_lean(a0, ah[m][ks][0], al[m][ks][0]);
              split_lean(a1, ah[m][ks][1], al[m][ks][1]);
              split_lean(a2, ah[m][ks][2], al[m][ks][2]);
              split_lean(a3, ah[m][ks][3], al[m][ks][3]);
            }
          const uint32_t q = q_base + wb;
          const int slot = q % kPSlots;
          // a slot's consecutive uses may belong to different warps when the tiles per step change between passes: a warp
          // running ahead must not take the slot's previous fill for its own (parity cannot tell fill r from r - 2), so it
          // first waits until the previous use has been released
          mbar_wait_timed(&ptile_empty[slot], ((q / kPSlots) & 1) ^ 1, w_pf);
          mbar_wait_timed(&ptile_full[slot], (q / kPSlots) & 1, w_pf);
          // k-major fragment (rows 8ks+t | +4 = sources, cols 8n+g = channels) of the 128B-swizzled tile:
          // (base ^ (n << 5)) + ks*1024, two per-lane bases for the +0 / +4 rows
          const uint32_t pt0 = a_ptiles + (uint32_t)slot * kPTileBytes + fb_k0, pt1 = a_ptiles + (uint32_t)slot * kPTileBytes + fb_k1;
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
            for (int n = 0; n < 4; ++n) {
              const float b0 = ldsa((pt0 ^ (n << 5)) + ks * 1024), b1 = ldsa((pt1 ^ (n << 5)) + ks * 1024);
              uint32_t bh[2], bl[2];
              split_lean(b0, bh[0], bl[0]);
              split_lean(b1, bh[1], bl[1]);
#pragma unroll
              for (int m = 0; m < 2; ++m) {
                mma_tf32_16x8x8(ccorr[m][n], al[m][ks], bh);
                mma_tf32_16x8x8(cmain[m][n], ah[m][ks], bh);
                mma_tf32_16x8x8(ccorr[m][n], ah[m][ks], bl);
              }
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&ptile_empty[slot]);            // tile consumed
          if (p.concat) {                                  // every head is its own output block
            store(h * C);
            clear();
          }
        }
        if (!p.concat && mine) store(0);                   // head mean (alpha pre-scaled by 1/H) + bias
      }
      if (p.terms_in) fence_proxy_async();               // our generic-proxy writes to the tile precede the next bulk copy into it
      mbar_arrive(&tile_empty[buf]);                     // this thread is done reading the alpha tile
    }
    if (tid == kGroupA) {
      atomicAdd(&g_diag_counters[kCntTileFull], (unsigned long long)w_tf);
      atomicAdd(&g_diag_counters[kCntPtileFull], (unsigned long long)w_pf);
      atomicAdd(&g_diag_counters[kCntRoleB], (unsigned long long)(clock64() - t_role));
    }
  } else {
    // ================================ warp 11: tile producer ================================
    // TMA when every tile starts on a 16-byte boundary (C % 4 == 0: the reference's shapes); otherwise the
    // warp gathers the tile itself into the same 128B-swizzled layout.
    const int lane = tid & 31;
    const bool tma_ok = (C % 4) == 0;
    if (lane == 0) prefetch_tmap(&tmP);
    auto produce = [&](unsigned char* dst, uint64_t* full_bar, int col0, int row0, long long& wacc, uint64_t* empty_bar,
                       uint32_t empty_parity) {
      if (lane == 0) mbar_wait_timed(empty_bar, empty_parity, wacc);
      __syncwarp();
      if (tma_ok) {
        if (lane == 0) {
          mbar_expect_tx(full_bar, kPTileBytes);
          tma_load_2d(dst, &tmP, col0, row0, full_bar);
        }
      } else {
        const long long n_rows = (long long)p.B * N;
        for (int idx = lane; idx < 32 * 32; idx += 32) {
          const int r = idx >> 5, c = idx & 31;
          float v = 0.f;
          if (row0 + r < n_rows && col0 + c < p.ldp) v = p.P_aug[((size_t)row0 + r) * p.ldp + col0 + c];
          *reinterpret_cast<float*>(dst + r * 128 + ((((c >> 2) ^ (r & 7)) << 4) | ((c & 3) << 2))) = v;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(full_bar);              // release: the tile is visible to the consumers
      }
    };
    uint32_t q = 0;
    long long w_pe = 0;
    const long long t_role = clock64();
    for (int it = 0; it < my_graphs; ++it) {
      const int b = blockIdx.x + it * gridDim.x;
      {                                                  // the s|d columns [HC, HC + 2H) of this graph's rows
        const int sb = it & 1;
        produce(smem_raw + off_sdtile + sb * kPTileBytes, &sd_full[sb], HC, b * N, w_pe, &sd_empty[sb],
                ((it >> 1) & 1) ^ 1);
      }
      for (int pass = 0; pass < n_pass; ++pass) {
        const int G = min(kCbPerPass, n_cb - pass * kCbPerPass);
        for (int h = 0; h < H; ++h) {
          for (int k = 0; k < G; ++k, ++q) {
            const int slot = q % kPSlots;
            produce(smem_raw + off_ptile + (size_t)slot * kPTileBytes, &ptile_full[slot],
                    h * C + (pass * kCbPerPass + k) * 32, b * N, w_pe, &ptile_empty[slot], ((q / kPSlots) & 1) ^ 1);
          }
        }
      }
    }
    if (lane == 0) {
      atomicAdd(&g_diag_counters[kCntPtileEmpty], (unsigned long long)w_pe);
      atomicAdd(&g_diag_counters[kCntRoleP], (unsigned long long)(clock64() - t_role));
    }
  }
}

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
  auto total = [&](const AttnSmem& s) { return ptile_off(s) + (size_t)(kPSlots + 2) * kPTileBytes; };
  AttnSmem sm = finish(attn_smem_plan(p.N, p.Fe, p.H, p.R, NPAIRS, kFwdChunkRows3));
  for (int rows = kFwdChunkRows3 - 16; rows >= 16 && total(sm) > 227 * 1024; rows -= 16)
    sm = finish(attn_smem_plan(p.N, p.Fe, p.H, p.R, NPAIRS, rows));
  const size_t smem = total(sm);
  if (smem > 227 * 1024)
    return fail(SPOTV2_ERR_UNSUPPORTED, "attn_fwd needs %zu B shared memory (> 227 KB)", smem);
  CUtensorMap tmP;      // P_aug as [B*N rows, ldp cols]; tiles of 32 rows x 32 channels
  if (int rc = make_tmap(&tmP, p.P_aug, (uint64_t)p.B * p.N, (uint64_t)p.ldp, (uint64_t)p.ldp, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B))
    return rc;
  const bool fix = NPAIRS == 15 && VEC2 && p.N == 30 && p.H == 6 && p.C == 500 && p.Fe == 126 && p.R == 870 && !p.concat && p.ldp == 3012 &&
                   p.ldo == 500 && p.bulk_ok && sm.NS == 36 && sm.KS == 16 && sm.chunk_rows == kFwdChunkRows3;
  auto kern = fix ? gat_attn_fwd_kernel<NPAIRS, VEC2, (NPAIRS == 15 && VEC2)> : gat_attn_fwd_kernel<NPAIRS, VEC2, false>;
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
