// Fused GAT attention forward, p_format 1: the projection arrives as the fp16 operand pair the GEMM epilogue wrote
// (attn_fwd.cu is the fp32-P version of the same operator; [PyG] gat_conv.py edge_update / softmax / propagate, reached
// from /root/reference/utils/models.py:146).
//
// Same roles as attn_fwd.cu - group A (3 warps) edge logits on 3xTF32 mma.sync, group B (8 warps) softmax + aggregation,
// one TMA producer warp, pipelined across graphs - but no thread converts an MMA operand in the aggregation:
//   * P tiles are 32 source rows x 32 channels of fp16 (64B swizzle); ONE TMA load brings four adjacent tiles of both
//     planes (a 4-D tensor map whose tile dimension overlaps the column dimension); the B fragments of mma.sync.m16n8k16
//     come out of ldmatrix.x4.trans (one instruction per k16 x n16 block);
//   * the softmax (row held in registers between its passes) is converted ONCE per graph into an fp16 hi/lo tile
//     [h][target i][source j]; the A fragments come out of ldmatrix.x4; the fp32 tile goes back to the logit group right
//     after that conversion;
//   * out[i, c] = (sum_h sum_j alpha_h[i,j] P[j, h, c]) with lo*hi + hi*lo + hi*hi per product (hi*hi only for the
//     half-precision class), 48 instead of 96 MMAs per (head, channel block) and 16 ldmatrix instead of ~130 loads/splits;
//   * the edge rows stream through a THREE-stage ring (two chunks in flight while one is consumed), the finished edge-term
//     tile leaves for the backward through one bulk store, the logit terms s|d come in fp32 one graph ahead.
// Every wait is bounded and reports which barrier starved before it traps.  Role cycle counters: -DSPOTV2_BRINGUP.
#include "attn_bwd.cuh"
#include "tma.cuh"

namespace spotv2 {

namespace {

constexpr int kGA = 96, kGB = 256, kF16Threads = kGA + kGB + 32;
constexpr int kChunkRows = 48;
constexpr int kEdgeStages = 3;        // edge-row ring depth: two chunks in flight while a third is consumed
constexpr int kSlotBytes = 4096;      // per tile: hi (2 KB) + lo (2 KB); a slot holds `grp` tiles: [hi tiles][lo tiles]
constexpr int kMaxPSlots = 24;
constexpr int kCbPass = 8;

struct Fwd16Plan {
  int NS, KS, chunk_rows, n_slots, grp;   // grp: tiles per TMA load / ring slot (4, or 1 when a 4-tile box could leave the last row)
  float s_alpha;                       // fp16 scale of the attention coefficients (alpha * dropout scale * s_alpha < 2^15)
  uint32_t off_bar, off_table, off_vfrag, off_sd, off_tile, off_ahi, off_alo, off_ring, ring_stage, off_sdslot, off_slots, total;
};

// cycle accounting per role (one sampling thread each; read through spotv2_diag_counters, entries [0, 16)):
// 0 A: edge ring wait, 1 A: tile buffer free, 2 B: edge terms ready, 3 B: P tiles, 4 P: slot free, 5/6/7 role totals,
// 8 A: logits arithmetic, 9 B: softmax, 10 B: conversions, 11 B: s|d tile, 12 A: chunk barriers, 13 A: edge-term copy-out
__device__ unsigned long long g_fwd16_counters[kNumCounters];

// bounded wait that says WHICH barrier starved before it traps (a lost arrival must fail loudly, never hang the box)
__device__ __noinline__ void wait_report(int id, int it, uint32_t parity) {
  printf("attn_fwd16: wait %d timed out (block %d thread %d graph-iteration %d parity %u)\n", id, (int)blockIdx.x, (int)threadIdx.x, it, parity);
}
constexpr int kWaitSpins = 16;
constexpr unsigned kWaitSleepNs = 64;
constexpr long long kWaitLimit = 400000000LL;         // ~0.2 s: a tenth of the ~2 s the other kernels allow
__device__ __forceinline__ void wait_id(uint64_t* bar, uint32_t parity, int id, int it) {
  mbar_wait_bounded<kWaitSpins, kWaitSleepNs, kWaitLimit>(smem_u32(bar), parity, [=] { wait_report(id, it, parity); });
}
// role counters cost ~4 K cycles per graph on the logit warps' critical path: compiled in with -DSPOTV2_BRINGUP only
// (tools/fwd16_waits.py reads them); the product build measures nothing
#ifdef SPOTV2_BRINGUP
constexpr bool kRoleCounters = true;
#else
constexpr bool kRoleCounters = false;
#endif
__device__ __forceinline__ long long tick() { return kRoleCounters ? clock64() : 0; }
__device__ __forceinline__ void wait_id_t(uint64_t* bar, uint32_t parity, int id, int it, long long& acc) {
  wait_timed<kRoleCounters>(acc, [&] { wait_id(bar, parity, id, it); });
}

template <bool FIX, bool SINGLE>
__global__ void __launch_bounds__(kF16Threads, 1)
gat_attn_fwd16_kernel(const AttnFwdArgs args, const Fwd16Plan pl_, const __grid_constant__ CUtensorMap tmH,
                      const __grid_constant__ CUtensorMap tmL, const __grid_constant__ CUtensorMap tmG) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  AttnParams p = args.p;
  Fwd16Plan pl = pl_;
  if (FIX) {
    p.N = 30; p.H = 6; p.C = 500; p.hp = 504; p.Fe = 126; p.R = 870; p.concat = 0; p.ldo = 500; p.bulk_ok = 1; p.vec2_ok = 1;
    pl.NS = 36; pl.KS = 16; pl.chunk_rows = kChunkRows; pl.grp = 4;
  }
  const int grp = pl.grp;
  const uint32_t slot_bytes = (uint32_t)grp * kSlotBytes;
  const int tid = threadIdx.x;
  const int N = p.N, H = p.H, C = p.C, NS = pl.NS, Cp = p.hp;
  const int tile_floats = H * N * NS;
  const int n_slots = pl.n_slots;

  // barriers: [0,3) edge ring, [4,5] tile_full, [6,7] tile_empty, then slot full / empty
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + pl.off_bar);
  uint64_t* tile_full = bars + 4;
  uint64_t* tile_empty = bars + 6;
  uint64_t* p_full = bars + 10;
  uint64_t* p_empty = p_full + kMaxPSlots;
  const int n_cb = (C + 31) / 32;
  const int n_pass = (n_cb + kCbPass - 1) / kCbPass;
  int32_t* table_s = reinterpret_cast<int32_t*>(smem_raw + pl.off_table);
  float4* vfrag = reinterpret_cast<float4*>(smem_raw + pl.off_vfrag);
  float* sd0 = reinterpret_cast<float*>(smem_raw + pl.off_sd);              // [2][N][2H] fp32
  float* tile0 = reinterpret_cast<float*>(smem_raw + pl.off_tile);          // [2][H][N][NS] fp32
  const int sd_floats = N * 2 * H;

  const int nchunks = (p.Fe > 0 && !p.terms_in) ? (p.R + pl.chunk_rows - 1) / pl.chunk_rows : 0;
  const int my_graphs = (p.B - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (tid == 0) {
    for (int r = 0; r < kEdgeStages; ++r) mbar_init(&bars[r], 1);
    for (int r = 0; r < 2; ++r) {
      mbar_init(&tile_full[r], kGA);
      mbar_init(&tile_empty[r], kGB);
    }
    for (int r = 0; r < n_slots; ++r) { mbar_init(&p_full[r], 1); mbar_init(&p_empty[r], grp); }
    fence_mbar_init();
  }
  for (int r = tid; r < p.R; r += kF16Threads) {
    const int code = (p.Fe > 0 && !p.terms_in) ? p.table[r] : -1;
    table_s[r] = code >= 0 ? ((code & 0xffff) * NS + (code >> 16)) * 4 : -1;
  }
  // the edge ring (+ its zero pad) starts zero-filled, and so do the alpha pair tiles: rows i >= N and columns j >= N of
  // the 32 x 32 operand blocks are never written and must read as zeros
  for (uint32_t idx = tid; idx < (pl.off_sdslot - pl.off_ahi) / 16; idx += kF16Threads)
    reinterpret_cast<float4*>(smem_raw + pl.off_ahi)[idx] = make_float4(0.f, 0.f, 0.f, 0.f);
  fence_proxy_async();
  if (p.Fe > 0 && !p.terms_in) build_vfrag(vfrag, p.v, H, p.Fe, pl.KS, 1, tid, kF16Threads);
  for (int idx = tid; idx < 2 * tile_floats; idx += kF16Threads) tile0[idx] = 0.f;
  __syncthreads();

  if (tid < kGA) {
    // ================================ group A: edge logits (as in attn_fwd.cu) ================================
    const int warp = tid >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const uint32_t sbase = smem_u32(smem_raw);
    const uint32_t ring_a0 = sbase + pl.off_ring;
    const uint32_t a_vfrag = sbase + pl.off_vfrag, a_table = sbase + pl.off_table;
    const uint32_t a_tile0 = sbase + pl.off_tile, head_bytes = (uint32_t)(N * NS * 4);
    auto stage = [&](int s_) { return reinterpret_cast<float*>(smem_raw + pl.off_ring + (size_t)s_ * pl.ring_stage); };
    const int total_chunks = my_graphs * nchunks;
    auto rows_in = [&](int c) { const int r = p.R - c * pl.chunk_rows; return r < pl.chunk_rows ? r : pl.chunk_rows; };
    auto issue = [&](int k) {
      const int it = k / nchunks, c = k - it * nchunks;
      const int b = blockIdx.x + it * gridDim.x;
      const uint32_t bytes = (uint32_t)rows_in(c) * p.Fe * 4u;
      mbar_expect_tx(&bars[k % kEdgeStages], bytes);
      bulk_g2s(stage(k % kEdgeStages), p.edge_rows + ((size_t)b * p.R + (size_t)c * pl.chunk_rows) * p.Fe, bytes, &bars[k % kEdgeStages]);
    };
    if (p.bulk_ok && tid == 0) {
      for (int k0 = 0; k0 < kEdgeStages && k0 < total_chunks; ++k0) issue(k0);
    }
    int k = 0;
    long long w_ring = 0, w_te = 0, t_log = 0, t_bar = 0, t_out = 0;
    const long long t_role = tick();
    for (int it = 0; it < my_graphs; ++it) {
      const int b = blockIdx.x + it * gridDim.x;
      const int buf = it & 1;
      float* tile = tile0 + buf * tile_floats;
      wait_id_t(&tile_empty[buf], ((it >> 1) & 1) ^ 1, 1, it, w_te);
      if (p.terms_in) {
        if (tid == 0) {
          const uint32_t bytes = (uint32_t)tile_floats * 4u;
          mbar_expect_tx(&tile_full[buf], bytes);
          bulk_g2s(tile, p.edge_terms + (size_t)b * tile_floats, bytes, &tile_full[buf]);
        } else {
          mbar_arrive(&tile_full[buf]);
        }
        continue;
      }
      if (nchunks == 0)
        for (int idx = tid; idx < tile_floats; idx += kGA) tile[idx] = 0.f;
      for (int c = 0; c < nchunks; ++c, ++k) {
        const int s = k % kEdgeStages;
        const int rows = rows_in(c);
        if (p.bulk_ok) {
          wait_id_t(&bars[s], (k / kEdgeStages) & 1, 2, it, w_ring);
        } else {
          const float* src = p.edge_rows + ((size_t)b * p.R + (size_t)c * pl.chunk_rows) * p.Fe;
          for (int idx = tid; idx < rows * p.Fe; idx += kGA) stage(s)[idx] = src[idx];
          bar_sync<1, kGA>();
        }
        const long long tl0 = tick();
        if (warp * 16 < rows) {
          const uint32_t r0 = ring_a0 + (uint32_t)s * pl.ring_stage + (uint32_t)(((warp * 16 + 2 * g) * p.Fe + t) * 4), r1 = r0 + (uint32_t)(p.Fe * 4);
          // (same summation order as attn_fwd.cu: the edge terms - and with them every LeakyReLU kink - are bit-identical in
          // both formats; two accumulator sets were tried and bought nothing: the phase is bound by per-warp issue)
          float acc[3][4];
#pragma unroll
          for (int pr = 0; pr < 3; ++pr)
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[pr][q] = 0.f;
          // software pipeline over batches of four k-steps: the operand loads of the next batch are in flight while this
          // batch is split and multiplied (one warp per scheduler has nobody else to hide its shared-memory latency);
          // k-steps and accumulators keep their order, so the sums are bit-identical to the un-pipelined loop
          float a0[4][4], a1[4][4];
          float4 b0[4], b1[4];
          auto load4 = [&](float (&a)[4][4], float4 (&bf)[4], int ks) {
            const uint32_t ko = (uint32_t)ks * 32u, vf = a_vfrag + ((uint32_t)ks * 32u + (uint32_t)lane) * 16u;
#pragma unroll
            for (int sl = 0; sl < 4; ++sl) {
              a[sl][0] = ldsa(r0 + ko + sl * 32);
              a[sl][1] = ldsa(r1 + ko + sl * 32);
              a[sl][2] = ldsa(r0 + ko + sl * 32 + 16);
              a[sl][3] = ldsa(r1 + ko + sl * 32 + 16);
              bf[sl] = lds128a(vf + sl * 512);
            }
          };
          auto mma4 = [&](const float (&a)[4][4], const float4 (&bf)[4]) {
#pragma unroll
            for (int sl = 0; sl < 4; ++sl) {
              uint32_t ah[4], al[4];
#pragma unroll
              for (int q = 0; q < 4; ++q) split_lean(a[sl][q], ah[q], al[q]);
              const uint32_t bh[2] = {__float_as_uint(bf[sl].x), __float_as_uint(bf[sl].y)};
              const uint32_t bl[2] = {__float_as_uint(bf[sl].z), __float_as_uint(bf[sl].w)};
              mma_tf32_16x8x8(acc[0], al, bh);
              mma_tf32_16x8x8(acc[1], ah, bl);
              mma_tf32_16x8x8(acc[2], ah, bh);
            }
          };
          load4(a0, b0, 0);
          for (int ks0 = 0; ks0 < pl.KS; ks0 += 8) {         // KS is a multiple of 8
            load4(a1, b1, ks0 + 4);
            mma4(a0, b0);
            if (ks0 + 8 < pl.KS) load4(a0, b0, ks0 + 8);
            mma4(a1, b1);
          }
          float res[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) res[q] = (acc[0][q] + acc[1][q]) + acc[2][q];
          const int rl = warp * 16 + 2 * g, row_base = c * pl.chunk_rows + rl;
          const int to0 = rl < rows ? ldsa_s32(a_table + (uint32_t)row_base * 4u) : -1;
          const int to1 = rl + 1 < rows ? ldsa_s32(a_table + (uint32_t)(row_base + 1) * 4u) : -1;
          const uint32_t tb = a_tile0 + (uint32_t)(buf * tile_floats * 4) + (uint32_t)(2 * t) * head_bytes;
          if (to0 >= 0) {
            if (2 * t < H) stsa(tb + (uint32_t)to0, res[0]);
            if (2 * t + 1 < H) stsa(tb + head_bytes + (uint32_t)to0, res[1]);
          }
          if (to1 >= 0) {
            if (2 * t < H) stsa(tb + (uint32_t)to1, res[2]);
            if (2 * t + 1 < H) stsa(tb + head_bytes + (uint32_t)to1, res[3]);
          }
        }
        const long long tl1 = tick();
        bar_sync<1, kGA>();
        t_log += tl1 - tl0;
        t_bar += tick() - tl1;
        if (p.bulk_ok && tid == 0 && k + kEdgeStages < total_chunks) issue(k + kEdgeStages);
      }
      if (p.edge_terms && !p.terms_in && NS == kEdgeTermNS && !p.alpha_rec) {
        // keep the edge terms for the backward (6 floats per edge instead of the Fe-wide rows): ONE bulk store of the tile
        // by the copy engine (a thread-by-thread copy sat in the LSU queue for ~12 K cycles per graph).  The generic-proxy
        // scatters are fenced and behind a barrier; thread 0 holds its arrival on tile_full until the engine has read
        // the tile, because the softmax group rewrites it in place.
        const long long to0 = tick();
        fence_proxy_async();
        bar_sync<1, kGA>();
        if (tid == 0) {
          bulk_s2g_commit(p.edge_terms + (size_t)b * tile_floats, smem_u32(tile), (uint32_t)tile_floats * 4u);
          bulk_wait_read();
        }
        t_out += tick() - to0;
      }
      mbar_arrive(&tile_full[buf]);
    }
    if (tid == 0) {
      atomicAdd(&g_fwd16_counters[0], (unsigned long long)w_ring);
      atomicAdd(&g_fwd16_counters[1], (unsigned long long)w_te);
      atomicAdd(&g_fwd16_counters[5], (unsigned long long)(tick() - t_role));
      atomicAdd(&g_fwd16_counters[8], (unsigned long long)t_log);
      atomicAdd(&g_fwd16_counters[12], (unsigned long long)t_bar);
      atomicAdd(&g_fwd16_counters[13], (unsigned long long)t_out);
    }
  } else if (tid < kGA + kGB) {
    // ================================ group B: softmax + aggregation ================================
    const int tb_ = tid - kGA;
    const int wb = tb_ >> 5, lane = tid & 31;
    const int g = lane >> 2, t = lane & 3;
    const uint32_t sbase = smem_u32(smem_raw);
    const uint32_t a_slots = sbase + pl.off_slots, a_ahi = sbase + pl.off_ahi, a_alo = sbase + pl.off_alo;
    // ldmatrix lane roles (identical for the alpha A fragments and the P B fragments): matrix = lane >> 3,
    // row = (lane & 7) + 8 * (matrix & 1), 16-byte chunk = matrix >> 1
    const int lm_row = (lane & 7) + ((lane >> 3) & 1) * 8, lm_chunk = lane >> 4;
    uint32_t lm_off[2][2];              // [row block of 16][chunk pair]: swizzled byte offset inside a 32 x 32 fp16 tile
#pragma unroll
    for (int rb = 0; rb < 2; ++rb)
#pragma unroll
      for (int cp = 0; cp < 2; ++cp) lm_off[rb][cp] = sw64(16 * rb + lm_row, 2 * cp + lm_chunk);
    // alpha_rec: the tile receives the exact signed coefficients (the backward's record); the head-mean factor then rides in
    // the accumulator scale instead of in alpha
    const bool rec = p.alpha_rec != 0 && p.edge_terms != nullptr && NS == kEdgeTermNS;
    const float head_scale = p.concat ? 1.f : 1.f / (float)H;
    const float out_scale = rec ? 1.f : head_scale;
    const float k_out = p.p_blk[2] / pl.s_alpha * (rec ? head_scale : 1.f);          // accumulator -> out
    uint32_t q_base = 0;
    long long w_tf = 0, w_pf = 0, w_sd = 0, t_smx = 0, t_cnv = 0;
    const long long t_role = tick();
    // s | d (fp32, as the GEMM accumulated them; N * 2H <= 512 values per graph): fetched one graph ahead into two registers
    // per thread, so that the global-load latency never sits in front of a softmax
    float sd_nx[2] = {0.f, 0.f};
    auto fetch_sd = [&](int b_) {
#pragma unroll
      for (int r_ = 0; r_ < 2; ++r_) {
        const int idx = tb_ + r_ * kGB;
        sd_nx[r_] = idx < sd_floats ? __ldg(p.sd32 + (size_t)b_ * sd_floats + idx) : 0.f;
      }
    };
    if (my_graphs > 0) fetch_sd(blockIdx.x);
    // slot cursor of this warp's next P-tile group: advanced by the groups of every (pass, head) step (no division in the loop)
    int cur_slot = 0;
    uint32_t cur_ph = 0;
    auto advance = [&](int k_) {
      cur_slot += k_;
      while (cur_slot >= n_slots) { cur_slot -= n_slots; cur_ph ^= 1u; }
    };
    for (int it = 0; it < my_graphs; ++it) {
      const int b = blockIdx.x + it * gridDim.x;
      const int buf = it & 1;
      float* tile = tile0 + buf * tile_floats;
      float* sd = sd0 + buf * sd_floats;
      const long long tc0 = tick();
#pragma unroll
      for (int r_ = 0; r_ < 2; ++r_)
        if (tb_ + r_ * kGB < sd_floats) sd[tb_ + r_ * kGB] = sd_nx[r_];
      if (it + 1 < my_graphs) fetch_sd(b + gridDim.x);
      const long long tc1 = tick();
      wait_id_t(&tile_full[buf], (it >> 1) & 1, 4, it, w_tf);
      const long long ts0 = tick();
      bar_sync<2, kGB>();                                // sd complete (and everyone is past the previous graph's MMAs)
      softmax_phase_regs(p, NS, tile, sd, out_scale, args.alpha_out ? args.alpha_out + (size_t)b * H * N * N : nullptr, nullptr, tb_,
                         kGB, nullptr, b, rec);
      if (rec) fence_proxy_async();                      // the copy engine reads what this thread wrote
      bar_sync<2, kGB>();                                // alpha tile complete
      if (rec && tb_ == 0) {
        // the backward's record: ONE bulk store of the finished tile (edge_mode 1: over the edge terms this graph came from)
        bulk_s2g_commit(p.edge_terms + (size_t)b * tile_floats, smem_u32(tile), (uint32_t)tile_floats * 4u);
      }
      const long long tc2 = tick();
      t_smx += tc2 - ts0;
      // alpha[h][j][i] fp32 -> fp16 hi | lo tiles [h][i][j] (64-byte rows, swizzled): the A operand of the aggregation
      {
        const int njp = (N + 1) / 2;
        for (int idx = tb_; idx < H * njp * N; idx += kGB) {
          const int i = idx % N, r = idx / N, jp = r % njp, h = r / njp;
          const float* base = tile + (size_t)h * N * NS + i;
          const float y0 = fabsf(base[(2 * jp) * NS]) * pl.s_alpha;               // (the record carries the LeakyReLU side in the sign)
          const float y1 = (2 * jp + 1 < N) ? fabsf(base[(2 * jp + 1) * NS]) * pl.s_alpha : 0.f;
          const __half2 hh = __floats2half2_rn(y0, y1);
          const uint32_t off = (uint32_t)h * 2048u + sw64(i, jp >> 2) + (uint32_t)(jp & 3) * 4u;
          *reinterpret_cast<__half2*>(smem_raw + pl.off_ahi + off) = hh;
          if (!SINGLE) {
            const float2 bk = __half22float2(hh);
            *reinterpret_cast<__half2*>(smem_raw + pl.off_alo + off) = __floats2half2_rn(y0 - bk.x, y1 - bk.y);
          }
        }
      }
      if (p.terms_in) fence_proxy_async();               // generic-proxy writes to the tile precede the next bulk copy into it
      if (rec && tb_ == 0) bulk_wait_read();                                                // the engine has read the record
      mbar_arrive(&tile_empty[buf]);                     // the fp32 tile is free for the logit group
      bar_sync<2, kGB>();                                // alpha pair tiles complete
      t_cnv += (tc1 - tc0) + (tick() - tc2);
      for (int pass = 0; pass < n_pass; ++pass) {
        const int G = min(kCbPass, n_cb - pass * kCbPass);
        const bool mine = wb < G;
        const int cb = pass * kCbPass + wb;
        float cmain[2][4][4], ccorr[2][4][4];
        auto clear = [&]() {
#pragma unroll
          for (int m = 0; m < 2; ++m)
#pragma unroll
            for (int n = 0; n < 4; ++n)
#pragma unroll
              for (int e = 0; e < 4; ++e) cmain[m][n][e] = ccorr[m][n][e] = 0.f;
        };
        // the bias of this warp's 8 output columns, fetched BEFORE the MMAs that produce them (a load per stored element
        // inside store() cost 12 % of the kernel's samples in long-scoreboard stalls)
        float bv[4][2];
        auto load_bias = [&](int col0) {
#pragma unroll
          for (int n = 0; n < 4; ++n)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int c = cb * 32 + n * 8 + 2 * t + e;
              bv[n][e] = (args.bias && mine && c < C) ? __ldg(args.bias + col0 + c) : 0.f;
            }
        };
        auto store = [&](int col0) {
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
                  const float o0 = (cmain[m][n][2 * hf] + ccorr[m][n][2 * hf]) * k_out + bv[n][0];
                  if (c + 1 < C) {
                    const float o1 = (cmain[m][n][2 * hf + 1] + ccorr[m][n][2 * hf + 1]) * k_out + bv[n][1];
                    if (p.vec2_ok) *reinterpret_cast<float2*>(dst) = make_float2(o0, o1);
                    else { dst[0] = o0; dst[1] = o1; }
                  } else {
                    dst[0] = o0;
                  }
                }
              }
        };
        clear();
        if (!p.concat) load_bias(0);
        const int n_g = (G + grp - 1) / grp;               // tile groups (ring slots) of one (pass, head) step
        const int gi = wb / grp, ti = wb - gi * grp;       // this warp's group and its tile inside it
        for (int h = 0; h < H; ++h, q_base += n_g, advance(n_g)) {
          if (gi >= n_g) continue;
          if (p.concat) load_bias(h * C);
          uint32_t ah[2][2][4], al[2][2][4];
          if (mine) {
#pragma unroll
            for (int m = 0; m < 2; ++m)
#pragma unroll
              for (int ks = 0; ks < 2; ++ks) {
                const uint32_t o = (uint32_t)h * 2048u + lm_off[m][ks];
                // matrices: (rows 0-7, chunk 2ks) (rows 8-15, chunk 2ks) (rows 0-7, chunk 2ks+1) (rows 8-15, chunk 2ks+1) = a0..a3
                ldsm_x4(a_ahi + o, ah[m][ks][0], ah[m][ks][1], ah[m][ks][2], ah[m][ks][3]);
                if (!SINGLE) ldsm_x4(a_alo + o, al[m][ks][0], al[m][ks][1], al[m][ks][2], al[m][ks][3]);
              }
          }
          int slot = cur_slot + gi;
          uint32_t sph = cur_ph;
          while (slot >= n_slots) { slot -= n_slots; sph ^= 1u; }
          // A slot's consecutive uses may belong to different warps: a warp that runs ahead must not take the slot's
          // PREVIOUS fill for its own (the parity test cannot tell fill r from fill r - 2), so it first waits until the
          // previous use has been released - only then can fill r be pending.
          wait_id_t(&p_empty[slot], sph ^ 1u, 8, it, w_pf);
          wait_id_t(&p_full[slot], sph, 5, it, w_pf);
          if (mine) {
            const uint32_t th = a_slots + (uint32_t)slot * slot_bytes + (uint32_t)ti * 2048u, tl = th + (uint32_t)grp * 2048u;
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
#pragma unroll
              for (int np = 0; np < 2; ++np) {
                // source rows 16ks.. (k), channel chunks 2np, 2np+1 (n blocks 2np, 2np+1): b0,b1 of n = 2np; b0,b1 of n = 2np+1
                uint32_t bh[4], bl[4];
                ldsm_x4_t(th + lm_off[ks][np], bh[0], bh[1], bh[2], bh[3]);
                if (!SINGLE) ldsm_x4_t(tl + lm_off[ks][np], bl[0], bl[1], bl[2], bl[3]);
#pragma unroll
                for (int nn = 0; nn < 2; ++nn) {
                  const int n = 2 * np + nn;
#pragma unroll
                  for (int m = 0; m < 2; ++m) {
                    if (!SINGLE) {
                      mma_f16_k16(ccorr[m][n], al[m][ks], bh[2 * nn], bh[2 * nn + 1]);
                      mma_f16_k16(ccorr[m][n], ah[m][ks], bl[2 * nn], bl[2 * nn + 1]);
                    }
                    mma_f16_k16(cmain[m][n], ah[m][ks], bh[2 * nn], bh[2 * nn + 1]);
                  }
                }
              }
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&p_empty[slot]);
          if (!mine) continue;
          if (p.concat) {
            store(h * C);
            clear();
          }
        }
        if (!p.concat && mine) store(0);
      }
    }
    if (tid == kGA) {
      atomicAdd(&g_fwd16_counters[2], (unsigned long long)w_tf);
      atomicAdd(&g_fwd16_counters[3], (unsigned long long)w_pf);
      atomicAdd(&g_fwd16_counters[6], (unsigned long long)(tick() - t_role));
      atomicAdd(&g_fwd16_counters[9], (unsigned long long)t_smx);
      atomicAdd(&g_fwd16_counters[10], (unsigned long long)t_cnv);
      atomicAdd(&g_fwd16_counters[11], (unsigned long long)w_sd);
    }
  } else {
    // ================================ producer warp ================================
    const int lane = tid & 31;
    if (lane == 0) {
      prefetch_tmap(&tmH);
      prefetch_tmap(&tmG);
      if (!SINGLE) prefetch_tmap(&tmL);
      uint32_t q = 0;
      long long w_pe = 0;
      const long long t_role = tick();
      for (int it = 0; it < my_graphs; ++it) {
        const int b = blockIdx.x + it * gridDim.x;
        for (int pass = 0; pass < n_pass; ++pass) {
          const int G = min(kCbPass, n_cb - pass * kCbPass);
          const int n_g = (G + grp - 1) / grp;
          for (int h = 0; h < H; ++h) {
            for (int k = 0; k < n_g; ++k, ++q) {
              const int slot = q % n_slots;
              unsigned char* dst = smem_raw + pl.off_slots + (size_t)slot * slot_bytes;
              wait_id_t(&p_empty[slot], ((q / n_slots) & 1) ^ 1, 7, it, w_pe);
              mbar_expect_tx(&p_full[slot], (uint32_t)grp * (SINGLE ? 2048u : 4096u));
              tma_load_4d(dst, &tmG, h * Cp + (pass * kCbPass + k * grp) * 32, b * N, 0, 0, &p_full[slot]);
            }
          }
        }
      }
      atomicAdd(&g_fwd16_counters[4], (unsigned long long)w_pe);
      atomicAdd(&g_fwd16_counters[7], (unsigned long long)(tick() - t_role));
    }
  }
}

}  // namespace

int fwd16_diag_add(unsigned long long* host_out, int reset) {
  return diag_add(host_out, g_fwd16_counters, reset);
}

// Shared-memory carve-up of the p_format 1 forward for a problem; n_slots * grp < 4 means it does not fit.
static Fwd16Plan fwd16_plan(const AttnParams& p) {
  Fwd16Plan pl{};
  pl.NS = 36;
  pl.KS = ((p.Fe + 7) / 8 + 7) / 8 * 8;
  // alpha (times the dropout scale 1/(1-p)) * s_alpha stays below 2^15
  int e = 14;
  for (float s = p.drop.scale; s > 1.f && e > -10; s *= 0.5f) --e;
  pl.s_alpha = ldexpf(1.f, e);
  const size_t tile_bytes = round_up((size_t)p.H * p.N * pl.NS * 4, 16);
  const size_t sd_bytes = round_up((size_t)p.N * 2 * p.H * 4, 16);
  auto layout = [&](int rows) {
    pl.chunk_rows = rows;
    size_t o = 0;
    pl.off_bar = (uint32_t)o;    o += 512;
    pl.off_table = (uint32_t)o;  o += round_up((size_t)(p.R > 0 ? p.R : 1) * 4, 16);
    pl.off_vfrag = (uint32_t)o;  o += (size_t)(p.Fe > 0 ? pl.KS : 0) * 32 * 16;
    pl.off_sd = (uint32_t)o;     o += 2 * sd_bytes;
    pl.off_tile = (uint32_t)o;   o += 2 * tile_bytes;
    o = round_up(o, 128);
    pl.off_ahi = (uint32_t)o;    o += (size_t)p.H * 2048;
    pl.off_alo = (uint32_t)o;    o += (size_t)p.H * 2048;
    pl.off_ring = (uint32_t)o;
    pl.ring_stage = (uint32_t)round_up((size_t)rows * p.Fe * 4, 128);
    o += (p.Fe > 0 && !p.terms_in) ? kEdgeStages * (size_t)pl.ring_stage + 256 : 0;     // + zero pad behind the ring (k-steps past Fe)
    o = round_up(o, 1024);
    pl.off_sdslot = (uint32_t)o;                           // (end of the zero-filled region; the P slots start here)
    pl.off_slots = (uint32_t)o;
    const size_t cap = 227 * 1024;
    pl.n_slots = o < cap ? (int)((cap - o) / ((size_t)pl.grp * kSlotBytes)) : 0;
    if (pl.n_slots > kMaxPSlots) pl.n_slots = kMaxPSlots;
    pl.total = (uint32_t)(o + (size_t)pl.n_slots * pl.grp * kSlotBytes);
  };
  // four tiles per load when the 4-tile box of the last head's last group stays inside a row of the planes (the tile
  // dimension of the tensor map overlaps the column dimension: nothing checks it against the row's end)
  const int n_cb_ = (p.C + 31) / 32;
  pl.grp = ((p.H - 1) * p.hp + (n_cb_ + 3) / 4 * 4 * 32 <= p.ldp16) ? 4 : 1;
  layout(kChunkRows);
  for (int rows = kChunkRows - 16; rows >= 16 && pl.n_slots * pl.grp < 12; rows -= 16) layout(rows);
  return pl;
}

bool attn_fwd16_fits(const AttnParams& p) {
  if (p.N > 32 || p.H > kMaxHeads || p.Fe > kMaxFe || p.hp % 8 != 0 || p.ldp16 % 8 != 0) return false;
  const Fwd16Plan pl = fwd16_plan(p);
  return pl.n_slots * pl.grp >= 4;
}

int attn_fwd16_dispatch(const AttnFwdArgs& a, cudaStream_t st) {
  const AttnParams& p = a.p;
  if (p.N > 32) return fail(SPOTV2_ERR_UNSUPPORTED, "attn_fwd (p_format 1): N=%d > 32", p.N);
  if (p.hp % 8 != 0 || p.ldp16 % 8 != 0) return fail(SPOTV2_ERR_INVALID_ARG, "attn_fwd (p_format 1): head pitch and ld16 must be multiples of 8");
  const bool single = p.P_lo == nullptr;
  Fwd16Plan pl = fwd16_plan(p);
  if (pl.n_slots * pl.grp < 4) return fail(SPOTV2_ERR_UNSUPPORTED, "attn_fwd (p_format 1): shared-memory plan does not fit (Fe=%d, H=%d)", p.Fe, p.H);
  CUtensorMap tmH, tmL;
  const uint64_t rows = (uint64_t)p.B * p.N, cols = (uint64_t)p.H * p.hp + 2 * p.H;
  if (int rc = make_tmap_f16(&tmH, p.P_hi, rows, cols, (uint64_t)p.ldp16, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B)) return rc;
  if (int rc = make_tmap_f16(&tmL, single ? p.P_hi : p.P_lo, rows, cols, (uint64_t)p.ldp16, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B)) return rc;
  CUtensorMap tmG;
  const uint64_t plane_stride = single ? 0 : (uint64_t)(p.P_lo - p.P_hi);
  if (!single && (p.P_lo <= p.P_hi || plane_stride % 8 != 0))
    return fail(SPOTV2_ERR_INVALID_ARG, "attn_fwd (p_format 1): the lo plane must follow the hi plane at a multiple of 16 bytes");
  if (int rc = make_tmap_tile_groups_f16(&tmG, p.P_hi, plane_stride, single ? 1 : 2, rows, cols, (uint64_t)p.ldp16, (uint32_t)pl.grp)) return rc;
  const bool fix = p.N == 30 && p.H == 6 && p.C == 500 && p.hp == 504 && p.Fe == 126 && p.R == 870 && !p.concat && p.ldo == 500 &&
                   p.bulk_ok && p.vec2_ok && pl.KS == 16 && pl.chunk_rows == kChunkRows && pl.grp == 4;
  auto kern = single ? (fix ? gat_attn_fwd16_kernel<true, true> : gat_attn_fwd16_kernel<false, true>)
                     : (fix ? gat_attn_fwd16_kernel<true, false> : gat_attn_fwd16_kernel<false, false>);
  SPOTV2_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.total));
  int grid = sm_count();
  if (grid > p.B) grid = p.B;
  kern<<<grid, kF16Threads, pl.total, st>>>(a, pl, tmH, tmL, tmG);
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

}  // namespace spotv2

using namespace spotv2;

extern "C" int spotv2_gat_attn_fwd_pair(const spotv2_gat_desc* d, const void* P_hi, const void* P_lo_or_null, const float* p_scale,
                                        const float* sd, const float* edge_rows, const int32_t* table, const float* v, const float* bias_or_null,
                                        float* out, float* alpha_or_null, float* edge_terms_or_null, void* stream) {
  if (int rc = check_desc(d)) return rc;
  const AttnEdgeArgs e{edge_rows, table, v, edge_terms_or_null, nullptr, false};
  if (int rc = check_attn_inputs(
          "attn_fwd_pair", d,
          {{d->p_format == 1, "attn_fwd_pair: the descriptor must say p_format 1"},
           {P_hi && p_scale && sd && out, "attn_fwd_pair: P_hi, p_scale, sd and out must be non-null"},
           {P_lo_or_null || d->gemm_algo == 3, "attn_fwd_pair: the lo plane may be omitted with gemm_algo 3 only"}},
          {{aligned16(P_hi) && (!P_lo_or_null || aligned16(P_lo_or_null)) && aligned16(out),
            "attn_fwd_pair: P planes / out must be 16-byte aligned"}},
          e))
    return rc;
  AttnFwdArgs a{attn_params_of(d, e), bias_or_null, out, alpha_or_null};
  a.p.P_hi = static_cast<const __half*>(P_hi);
  a.p.P_lo = d->gemm_algo == 3 ? nullptr : static_cast<const __half*>(P_lo_or_null);
  a.p.p_blk = p_scale;
  a.p.sd32 = sd;
  return attn_fwd16_dispatch(a, as_stream(stream));
}
