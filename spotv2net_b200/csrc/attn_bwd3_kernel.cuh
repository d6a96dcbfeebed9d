// Body of the tcgen05 attention backward (attn_bwd3.cu), included there twice: SPOTV2_KERNEL_NAME names the kernel and
// SPOTV2_GA = 1 makes the variant that takes d_alpha [B, H, N(j), N(i)], the gradient through the coefficients the forward
// returned (after dropout), which joins dalpha before the dropout factor.  Two kernels under their own names keep the
// machine code of the one without it exactly what it was.  No include guard: meant to be included more than once.
template <bool DROP, int HT>
__global__ void __launch_bounds__(kB3Threads, 1)
SPOTV2_KERNEL_NAME(const AttnBwdArgs args, const Bwd3Plan pl, const __grid_constant__ CUtensorMap tmP,
            const __grid_constant__ CUtensorMap tmG, const __grid_constant__ CUtensorMap tmGt
#if SPOTV2_GA
            , const float* __restrict__ d_alpha
#endif
) {
  constexpr bool GA = SPOTV2_GA != 0;
#if !SPOTV2_GA
  const float* const d_alpha = nullptr;
#endif
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  const AttnParams& p = args.p;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = p.N, H = HT ? HT : p.H, C = p.C, Fe = p.Fe, HC = H * C;
  const uint32_t sbase = smem_u32(smem_raw);
  const uint32_t a_bar = sbase + pl.off_bar, a_table = sbase + pl.off_table, a_sd = sbase + pl.off_sd;
  const uint32_t a_dbias = sbase + pl.off_dbias, a_work = sbase + pl.off_work, a_ahi = sbase + pl.off_ahi, a_alo = sbase + pl.off_alo;
  const uint32_t a_lo = sbase + pl.off_lo, a_slots = sbase + pl.off_slots;
  auto BAR = [&](int k) { return a_bar + (uint32_t)k * 8u; };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem_raw + pl.off_bar + kNumBars * 8);
  const int my_graphs = (p.B - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const bool has_v = !p.terms_in;
  const int tile_floats = H * N * kNS3;

  // ---------------------------------------------------------------- setup
  if (tid == 0) {
    for (int k = 0; k < kNumBars; ++k) mbar_init(reinterpret_cast<uint64_t*>(smem_raw + pl.off_bar) + k, 1);
    fence_mbar_init();
  }
  // zero everything the tensor core or a padded loop may read before it is written
  for (uint32_t o = pl.off_table + (uint32_t)tid * 16u; o < pl.total; o += kB3Threads * 16u)
    *reinterpret_cast<float4*>(smem_raw + o) = make_float4(0.f, 0.f, 0.f, 0.f);
  __syncthreads();
  // row -> float offset of (source j, target i) inside one head of the work tile (-1: row skipped)
  for (int r = tid; r < p.R && has_v; r += kB3Threads) {
    const int code = p.table[r];
    reinterpret_cast<int32_t*>(smem_raw + pl.off_table)[r] = code >= 0 ? (code & 0xffff) * kNS3 + (code >> 16) : -1;
  }
  // the ones row (head 0, spare source row 31): phase D then also produces sum_i dout[i, c] = the bias gradient
  if (tid < N) {
    const int r = 31, i = tid;
    *reinterpret_cast<float*>(smem_raw + pl.off_ahi + r * 128 + ((((i >> 2) ^ (r & 7)) << 4) | ((i & 3) << 2))) = 1.f;
  }
  fence_proxy_async();
  if (warp == kWarpMma) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tA = tmem_base, tD = tmem_base + 128u;        // phase A: 64 columns per 128-row block; phase D: 128 per block

  // Ring discipline.  A wait on a slot's "full" barrier tells phases apart by parity alone, so a role may start such a
  // wait only when the previous use of that slot has been filled already (else the wait returns at once) and before the
  // next one can be (else it never returns).  Every role therefore waits only on slots it consumes itself, and each
  // jump over slots consumed by others is gated by an event that implies the fills in between:
  //   softmax group  T(g): after alpha_empty(g-1) (all MMAs of g-1 done, so all its A/G fills) and its own V(g-1);
  //                  V(g): after dalpha_full(g) (all A(g) fills); the G(g) fills it jumps are issued before V(g)'s
  //   stream warps   A/G(g): after v_done(g-1) and t_done(g); inside the run, lo_empty of the warp's previous slot
  //                  (a commit, so every earlier MMA and with it every earlier fill) comes BEFORE the full wait
  if (warp == kWarpProd) {
    // =========================================== producer ===========================================
    if (lane == 0) {
      prefetch_tmap(&tmP); prefetch_tmap(&tmG); prefetch_tmap(&tmGt);
      SlotCursor cur{0, 0u, pl.n_slots};
      long long w_empty = 0;
      auto acquire = [&]() -> uint32_t {
        bar_wait_t(BAR(kBarEmpty + cur.slot), cur.ph ^ 1u, w_empty);
        return a_slots + (uint32_t)cur.slot * pl.slot_bytes;
      };
      for (int it = 0; it < my_graphs; ++it) {
        const int b = blockIdx.x + it * gridDim.x;
        for (int pc = 0; pc < pl.t_pieces; ++pc) {                               // T: the forward's edge terms
          const uint32_t dst = acquire(), full = BAR(kBarFull + cur.slot);
          const uint32_t off = (uint32_t)pc * pl.slot_bytes;
          const uint32_t bytes = min(pl.slot_bytes, pl.tile_bytes - off);
          mbar_expect_tx(full, bytes);
          bulk_g2s_hint(dst, reinterpret_cast<const unsigned char*>(p.edge_terms + (size_t)b * tile_floats) + off, bytes, full, kEvictFirst);
          cur.advance();
        }
        for (int kb = 0; kb < pl.n_kb; ++kb) {                                   // A: P tiles of all heads + dout, 16 channels
          const uint32_t dst = acquire(), full = BAR(kBarFull + cur.slot);
          mbar_expect_tx(full, pl.a_bytes);
          for (int h = 0; h < H; ++h) tma_load_3d_hint(dst + (uint32_t)h * kPTile, &tmP, h * C + kb * kKB, 0, b, full, kEvictFirst);
          tma_load_3d_hint(dst + (uint32_t)H * kPTile, &tmG, kb * kKB, 0, b, full, kEvictNormal);
          cur.advance();
        }
        for (int cb = 0; cb < pl.n_cb; ++cb) {                                   // G: dout again, MN-major boxes (L2 hits)
          const uint32_t dst = acquire(), full = BAR(kBarFull + cur.slot);
          mbar_expect_tx(full, 4u * kGTile);
          for (int k = 0; k < 4; ++k) tma_load_3d_hint(dst + (uint32_t)k * kGTile, &tmGt, cb * kCB + k * 32, 0, b, full, kEvictFirst);
          cur.advance();
        }
        for (int c = 0; c < pl.nchunks; ++c) {                                   // V: edge rows, once
          const uint32_t dst = acquire(), full = BAR(kBarFull + cur.slot);
          int rows = p.R - c * pl.chunk_rows;
          if (rows > pl.chunk_rows) rows = pl.chunk_rows;
          const uint32_t bytes = (uint32_t)rows * (uint32_t)Fe * 4u;
          mbar_expect_tx(full, bytes);
          bulk_g2s_hint(dst, p.edge_rows + ((size_t)b * p.R + (size_t)c * pl.chunk_rows) * Fe, bytes, full, kEvictFirst);
          cur.advance();
        }
      }
      atomicAdd(&g_bwd3_counters[0], (unsigned long long)w_empty);
    }
  } else if (warp == kWarpMma) {
    // =========================================== MMA issuer ===========================================
    if (lane == 0) {
      // instruction descriptors: D fp32, A/B tf32; bit 16 = B is MN-major; N >> 3 at bit 17, M >> 4 at bit 24
      const uint32_t id_base = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(128 >> 4) << 24);
      const uint32_t id_a64 = id_base | ((uint32_t)(64 >> 3) << 17), id_a32 = id_base | ((uint32_t)(32 >> 3) << 17);
      const uint32_t id_d = id_base | (1u << 16) | ((uint32_t)(kCB >> 3) << 17);
      SlotCursor cur{0, 0u, pl.n_slots};
      uint32_t lo_n = 0, d_n = 0;                       // lo-buffer uses and phase-D blocks so far
      long long w_a = 0, w_al = 0, w_d = 0;
      for (int it = 0; it < my_graphs; ++it) {
        const uint32_t gph = (uint32_t)it & 1u;
        cur.advance(pl.t_pieces);
        // ---- phase A: dalpha.  TMEM columns per 128-row block: [0,32) small terms (hi*lo + lo*hi), [32,64) hi*hi
        bar_wait_t(BAR(kBarDAEmpty), gph ^ 1u, w_a);
        tc_fence_after();
        for (int kb = 0; kb < pl.n_kb; ++kb, ++lo_n) {
          const uint32_t li = lo_n & 1u;
          bar_wait_t(BAR(kBarLoFull + li), (lo_n >> 1) & 1u, w_a);
          tc_fence_after();
          const uint32_t sa = a_slots + (uint32_t)cur.slot * pl.slot_bytes, lo = a_lo + li * pl.lo_bytes;
#pragma unroll
          for (int ks = 0; ks < kKB / 8; ++ks) {
            const uint64_t b_cat = make_desc(lo + (uint32_t)H * kPTile + ks * 32, 16, 512, 4);    // dout lo rows | hi rows
            const uint64_t b_hi = make_desc(sa + (uint32_t)H * kPTile + ks * 32, 16, 512, 4);
            for (int blk = 0; blk < pl.n_blk; ++blk) {
              const uint64_t a_hi = make_desc(sa + (uint32_t)blk * 8192u + ks * 32, 16, 512, 4);
              const uint64_t a_lo_ = make_desc(lo + (uint32_t)blk * 8192u + ks * 32, 16, 512, 4);
              umma_tf32(tA + (uint32_t)blk * 64u, a_hi, b_cat, id_a64, (kb | ks) ? 1u : 0u);
              umma_tf32(tA + (uint32_t)blk * 64u, a_lo_, b_hi, id_a32, 1u);
            }
          }
          umma_commit(BAR(kBarEmpty + cur.slot));
          umma_commit(BAR(kBarLoEmpty + li));
          cur.advance();
        }
        umma_commit(BAR(kBarDAFull));
        // ---- phase D: dP[(h,j), c] per block of 128 channels; A = alpha^T (K-major), B = dout (channel-major)
        bar_wait_t(BAR(kBarAlphaFull), gph, w_al);
        for (int cb = 0; cb < pl.n_cb; ++cb, ++lo_n, ++d_n) {
          const uint32_t li = lo_n & 1u;
          bar_wait_t(BAR(kBarLoFull + li), (lo_n >> 1) & 1u, w_d);
          bar_wait_t(BAR(kBarDTEmpty), (d_n & 1u) ^ 1u, w_d);
          tc_fence_after();
          const uint32_t sa = a_slots + (uint32_t)cur.slot * pl.slot_bytes, lo = a_lo + li * pl.lo_bytes;
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            const uint64_t b_hi = make_desc(sa + ks * 1024, kGTile, 512, 1);       // 8 target rows per k-step
            const uint64_t b_lo = make_desc(lo + ks * 1024, kGTile, 512, 1);
            for (int blk = 0; blk < pl.n_blk; ++blk) {
              const uint64_t a_hi = make_desc(a_ahi + (uint32_t)blk * 16384u + ks * 32, 16, 1024, 2);
              const uint64_t a_lo_ = make_desc(a_alo + (uint32_t)blk * 16384u + ks * 32, 16, 1024, 2);
              const uint32_t td = tD + (uint32_t)blk * kCB;
              umma_tf32(td, a_lo_, b_hi, id_d, ks ? 1u : 0u);                      // small terms first
              umma_tf32(td, a_hi, b_lo, id_d, 1u);
              umma_tf32(td, a_hi, b_hi, id_d, 1u);
            }
          }
          umma_commit(BAR(kBarEmpty + cur.slot));
          umma_commit(BAR(kBarLoEmpty + li));
          umma_commit(BAR(kBarDTFull));
          cur.advance();
        }
        umma_commit(BAR(kBarAlphaEmpty));
        cur.advance(pl.nchunks);
      }
      atomicAdd(&g_bwd3_counters[1], (unsigned long long)w_a);
      atomicAdd(&g_bwd3_counters[3], (unsigned long long)w_al);
      atomicAdd(&g_bwd3_counters[4], (unsigned long long)w_d);
    }
  } else if (warp >= kWarpSt0) {
    // =========================================== stream group: the lo pass ===========================================
    // Warp w owns lo buffer w and takes every second A / G slot: two slots are in flight and nothing but the warp itself
    // has to be synchronised before the MMA warp is told.  hi stays where TMA put it (the tensor core reads the top 19
    // bits of an fp32 pattern: measured, tools/bwd3_rawhi.py); lo = RN_tf32(x - trunc_tf32(x)) goes to the lo buffer.
    // 16-byte pieces at or past dup_from (the dout tile of an A slot) also copy hi one tile further into the lo buffer
    // (B operand "lo rows | hi rows").  Four pieces per lane per round, loads first.
    const int sw = warp - kWarpSt0;
    SlotCursor cur{0, 0u, pl.n_slots};
    uint32_t lo_n = 0;
    long long w_full = 0, w_loe = 0, t_lo = 0;
    auto lo_pass = [&](uint32_t src, uint32_t dst, int n16, int dup_from) {
      for (int base = 0; base < n16; base += 4 * 32) {
        float4 x[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int idx = base + u * 32 + lane;
          x[u] = idx < n16 ? lds128a(src + (uint32_t)idx * 16u) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int idx = base + u * 32 + lane;
          if (idx < n16) {
            const float4 lo = make_float4(rn_tf32(x[u].x - tr_tf32(x[u].x)), rn_tf32(x[u].y - tr_tf32(x[u].y)),
                                          rn_tf32(x[u].z - tr_tf32(x[u].z)), rn_tf32(x[u].w - tr_tf32(x[u].w)));
            sts128a(dst + (uint32_t)idx * 16u, lo);
            if (idx >= dup_from) sts128a(dst + (uint32_t)idx * 16u + kPTile, x[u]);
          }
        }
      }
    };
    for (int it = 0; it < my_graphs; ++it) {
      bar_sync<3, kStT>();                                                        // both warps know every fill either has seen
      if (has_v && it > 0) bar_wait_t(BAR(kBarVDone), (uint32_t)(it - 1) & 1u, w_full);
      bar_wait_t(BAR(kBarTDone), (uint32_t)it & 1u, w_full);
      cur.advance(pl.t_pieces);
      for (int kb = 0; kb < pl.n_kb + pl.n_cb; ++kb, ++lo_n) {                    // A slots, then G slots
        if ((int)(lo_n & 1u) == sw) {
          bar_wait_t(BAR(kBarLoEmpty + sw), ((lo_n >> 1) & 1u) ^ 1u, w_loe);
          bar_wait_t(BAR(kBarFull + cur.slot), cur.ph, w_full);
          const long long t0 = clock64();
          const uint32_t sa = a_slots + (uint32_t)cur.slot * pl.slot_bytes, lo = a_lo + (uint32_t)sw * pl.lo_bytes;
          if (kb < pl.n_kb) lo_pass(sa, lo, (int)(pl.a_bytes / 16u), H * (kPTile / 16));
          else lo_pass(sa, lo, 4 * kGTile / 16, 0x7fffffff);
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive(BAR(kBarLoFull + sw));
          t_lo += clock64() - t0;
        }
        cur.advance();
      }
      cur.advance(pl.nchunks);
    }
    if (lane == 0) {
      atomicAdd(&g_bwd3_counters[5], (unsigned long long)w_full);
      atomicAdd(&g_bwd3_counters[6], (unsigned long long)w_loe);
      atomicAdd(&g_bwd3_counters[7], (unsigned long long)t_lo);
    }
  } else if (warp >= kWarpDe0) {
    // =========================================== epilogue group: dP ===========================================
    // Warp q owns TMEM lanes [32q, 32q + 32) = the source rows of head q (block 0) and head 4 + q (block 1): a thread
    // holds one (head, source) row and takes 32 consecutive channels per tcgen05.ld, so the fp16 hi/lo pair of those
    // channels leaves as 64 contiguous bytes per array (8-byte stores: a head's columns start on 8-byte boundaries).
    const int de = tid - kWarpDe0 * 32, q = de >> 5;
    float dp_scale = 1.f;
    if (args.dP_hi16) {
      dp_scale = dp_scale_from_amax(__uint_as_float(*reinterpret_cast<const unsigned*>(args.dout_blk)) * args.bound);
      if (blockIdx.x == 0 && de == 0) { args.dp_blk[2] = 1.f / dp_scale; args.dp_blk[4] = dp_scale; }
    }
    const float k_dp = dp_scale / (float)H * (DROP ? p.drop.scale : 1.f);
    const uint32_t stg = sbase + pl.off_stage + (uint32_t)q * 4096u;
    uint32_t d_n = 0;
    long long w_dt = 0, t_de = 0;
    for (int it = 0; it < my_graphs; ++it) {
      const int b = blockIdx.x + it * gridDim.x;
      for (int cb = 0; cb < pl.n_cb; ++cb, ++d_n) {
        bar_wait_t(BAR(kBarDTFull), d_n & 1u, w_dt);
        const long long t0 = clock64();
        tc_fence_after();
        for (int blk = 0; blk < pl.n_blk; ++blk) {
          const int h = blk * 4 + q;
          if (h >= H) break;                                                      // warp-uniform
          const uint32_t tbase = tD + (uint32_t)blk * kCB + ((uint32_t)(q * 32) << 16);
          const size_t row = ((size_t)b * N + lane);                              // lane = source j
#pragma unroll 1
          for (int c0 = 0; c0 < kCB; c0 += 32) {
            const int c = cb * kCB + c0;
            if (c >= C) break;
            uint32_t r[32];
            tmem_ld32(tbase + (uint32_t)c0, r);
            if (h == 0 && lane == 31) {                                           // the ones row: column sums of dout
#pragma unroll
              for (int k = 0; k < 32; ++k)
                if (c + k < C) stsa(a_dbias + (uint32_t)(c + k) * 4u, ldsa(a_dbias + (uint32_t)(c + k) * 4u) + __uint_as_float(r[k]));
            }
            if (args.dP_hi16) {
              // the row's 32 channels as fp16 hi | lo (packed converts), parked in the warp's staging tile ([32 sources][64 B]
              // per array, 16-byte chunks XOR (j >> 1) & 3: conflict-free both ways) and read back so that 8 lanes cover one
              // row: a store instruction writes four 64-byte row pieces instead of thirty-two 8-byte ones
              uint32_t hi[16], lo[16];
#pragma unroll
              for (int k = 0; k < 16; ++k) {
                const float w0 = __uint_as_float(r[2 * k]) * k_dp, w1 = __uint_as_float(r[2 * k + 1]) * k_dp;
                const __half2 hh = __floats2half2_rn(w0, w1);
                const float2 bk = __half22float2(hh);
                const __half2 ll = __floats2half2_rn(w0 - bk.x, w1 - bk.y);
                hi[k] = *reinterpret_cast<const uint32_t*>(&hh);
                lo[k] = *reinterpret_cast<const uint32_t*>(&ll);
              }
              const uint32_t sw_ = (uint32_t)((lane >> 1) & 3);
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const uint32_t o = (uint32_t)lane * 64u + (((uint32_t)k ^ sw_) << 4);
                sts128a_b32(stg + o, hi[4 * k], hi[4 * k + 1], hi[4 * k + 2], hi[4 * k + 3]);
                sts128a_b32(stg + 2048u + o, lo[4 * k], lo[4 * k + 1], lo[4 * k + 2], lo[4 * k + 3]);
              }
              __syncwarp();
              const int pc = (lane & 7) * 4;                                        // first of this lane's 4 channels in the piece
              if (c + pc < C) {                                                    // C % 4 == 0: four channels are in or out together
                uint2 vh[8], vl[8];
#pragma unroll
                for (int it8 = 0; it8 < 8; ++it8) {
                  const int j = 4 * it8 + (lane >> 3);
                  const uint32_t o = (uint32_t)j * 64u + ((((uint32_t)(lane & 7) >> 1) ^ (uint32_t)((j >> 1) & 3)) << 4) + (uint32_t)(lane & 1) * 8u;
                  vh[it8] = lds64a_b32(stg + o);
                  vl[it8] = lds64a_b32(stg + 2048u + o);
                }
#pragma unroll
                for (int it8 = 0; it8 < 8; ++it8) {
                  const int j = 4 * it8 + (lane >> 3);
                  if (j < N) {
                    const size_t off = ((size_t)b * N + j) * args.ldp16 + (size_t)h * C + c + pc;
                    *reinterpret_cast<uint2*>(args.dP_hi16 + off) = vh[it8];
                    *reinterpret_cast<uint2*>(args.dP_lo16 + off) = vl[it8];
                  }
                }
              }
              __syncwarp();
            } else if (lane < N) {
              float* pf = args.dP_aug + row * p.ldp + (size_t)h * C + c;
#pragma unroll
              for (int k = 0; k < 32; k += 4)
                if (c + k < C)
                  *reinterpret_cast<float4*>(pf + k) = make_float4(__uint_as_float(r[k]) * k_dp, __uint_as_float(r[k + 1]) * k_dp,
                                                                   __uint_as_float(r[k + 2]) * k_dp, __uint_as_float(r[k + 3]) * k_dp);
            }
          }
        }
        tc_fence_before();
        bar_sync<2, kDeT>();
        if (de == 0) mbar_arrive(BAR(kBarDTEmpty));
        t_de += clock64() - t0;
      }
    }
    bar_sync<2, kDeT>();
    for (int c = de; c < C; c += kDeT) args.dbias_part[(size_t)blockIdx.x * p.ldo + c] = ldsa(a_dbias + (uint32_t)c * 4u);
    if (de == 0) {
      atomicAdd(&g_bwd3_counters[2], (unsigned long long)w_dt);
      atomicAdd(&g_bwd3_counters[12], (unsigned long long)t_de);
    }
  } else {
    // =========================================== softmax group ===========================================
    const int h = warp, i = lane;                     // thread = (head, target) for the column passes, (head, source) for rows
    const bool on = h < H && i < N;
    const float g_scale = 1.f / (float)H;
    const float inv_nm1 = 1.f / (float)(N > 1 ? N - 1 : 1);
    SlotCursor cur{0, 0u, pl.n_slots};
    long long w_t = 0, t_sm = 0, w_da = 0, t_sb = 0, w_vfull = 0, t_v = 0;
    float dsd_max = 0.f;                 // max |ds|, |dd| written by this thread
    // phase V: a warp takes every 8th row of a chunk; a lane owns features 2l, 2l+1, 64+2l, 64+2l+1 and all heads
    constexpr int kHP = HT ? (HT + 1) / 2 : kMaxHeads / 2;      // head pairs
    const int f0 = 2 * lane, f1 = 64 + 2 * lane;
    float2 run[4][kHP];
#pragma unroll
    for (int f = 0; f < 4; ++f)
#pragma unroll
      for (int k = 0; k < kHP; ++k) run[f][k] = make_float2(0.f, 0.f);
    const uint32_t col = a_work + (uint32_t)(h * N * kNS3 + i) * 4u;             // + j * kNS3 * 4
    // element (row r = 32 h + j, k = i) of the alpha operand tiles (128-byte rows, 16-byte chunks XOR (r & 7))
    auto aoff = [&](int j, int k) -> uint32_t {
      const int r = 32 * h + j;
      return (uint32_t)(r * 128 + ((((k >> 2) ^ (r & 7)) << 4) | ((k & 3) << 2)));
    };
    for (int it = 0; it < my_graphs; ++it) {
      const int b = blockIdx.x + it * gridDim.x;
      const uint32_t gph = (uint32_t)it & 1u;
      // s | d columns of this graph's nodes (2H floats per node behind the H*C projection columns)
      float sd_reg[2] = {0.f, 0.f};
      for (int k = 0; k < 2; ++k) {
        const int idx = tid + k * kSmT;
        if (idx < N * 2 * H) sd_reg[k] = p.P_aug[((size_t)b * N + idx / (2 * H)) * p.ldp + HC + idx % (2 * H)];
      }
      bar_wait_t(BAR(kBarAlphaEmpty), gph ^ 1u, w_t);     // every MMA of the previous graph is done: its slots were all filled
      for (int pc = 0; pc < pl.t_pieces; ++pc) {
        bar_wait_t(BAR(kBarFull + cur.slot), cur.ph, w_t);
        const uint32_t sa = a_slots + (uint32_t)cur.slot * pl.slot_bytes, off = (uint32_t)pc * pl.slot_bytes;
        const int n16 = (int)(min(pl.slot_bytes, pl.tile_bytes - off) / 16u);
        for (int idx = tid; idx < n16; idx += kSmT) sts128a(a_work + off + (uint32_t)idx * 16u, lds128a(sa + (uint32_t)idx * 16u));
        bar_sync<1, kSmT>();
        if (tid == 0) mbar_arrive(BAR(kBarEmpty + cur.slot));
        cur.advance();
      }
      if (tid == 0) mbar_arrive(BAR(kBarTDone));
      cur.advance(pl.n_kb + pl.n_cb);                                            // on to this graph's V slots
      for (int k = 0; k < 2; ++k) {
        const int idx = tid + k * kSmT;
        if (idx < N * 2 * H) stsa(a_sd + (uint32_t)idx * 4u, sd_reg[k]);
      }
      bar_sync<1, kSmT>();
      // ------------------------------------------------ softmax (thread = head h, target i) ------------------------------------------------
      const long long t_s0 = clock64();
      uint32_t mask = 0u, keep = 0xffffffffu;
      if (on) {
        float gsum = 0.f;
        for (int j = 0; j < N; ++j) gsum += (j != i) ? ldsa(col + (uint32_t)j * (kNS3 * 4)) : 0.f;
        const float gii = gsum / (float)(N > 1 ? N - 1 : 1);
        const float di = ldsa(a_sd + (uint32_t)(i * 2 * H + H + h) * 4u);
        float mx = -INFINITY;
        for (int j = 0; j < N; ++j) {
          const float z = (j == i ? gii : ldsa(col + (uint32_t)j * (kNS3 * 4))) + ldsa(a_sd + (uint32_t)(j * 2 * H + h) * 4u) + di;
          if (z > 0.f) mask |= 1u << j;
          const float l = z > 0.f ? z : z * p.slope;
          mx = fmaxf(mx, l);
          stsa(col + (uint32_t)j * (kNS3 * 4), l);
        }
        float sum = 0.f;
        for (int j = 0; j < N; ++j) {
          const float e = expf(ldsa(col + (uint32_t)j * (kNS3 * 4)) - mx);
          sum += e;
          stsa(col + (uint32_t)j * (kNS3 * 4), e);
        }
        const float inv = 1.f / (sum + 1e-16f);
        if (DROP) keep = dropout_keep_bits(p.drop, (((unsigned long long)b * H + h) * N + i) * N, N);
        for (int j = 0; j < N; ++j) {
          const float a = ldsa(col + (uint32_t)j * (kNS3 * 4)) * inv;
          stsa(col + (uint32_t)j * (kNS3 * 4), a);                              // un-dropped alpha stays in the work tile for now
          const float am = ((keep >> j) & 1u) ? a : 0.f;                         // the MMA operand carries the mask, not 1/(1-p)
          const float hi = tr_tf32(am);
          const uint32_t o = aoff(j, i);
          stsa(a_ahi + o, hi);
          stsa(a_alo + o, rn_tf32(am - hi));
        }
      }
      fence_proxy_async();
      bar_sync<1, kSmT>();
      if (tid == 0) mbar_arrive(BAR(kBarAlphaFull));
      // alpha column of this thread: kept in registers across the TMEM dump (which overwrites the work tile)
      float al[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) al[j] = (on && j < N) ? ldsa(col + (uint32_t)j * (kNS3 * 4)) : 0.f;
      // ------------------------------------------------ dalpha: TMEM -> work tile (thread = head h, source j) ------------------------------------------------
      t_sm += clock64() - t_s0;
      bar_wait_t(BAR(kBarDAFull), gph, w_da);
      const long long t_b0 = clock64();
      tc_fence_after();
      bar_sync<1, kSmT>();                                                       // every alpha column is in registers
      if (h < H) {
        const uint32_t taddr = tA + (uint32_t)(h >> 2) * 64u + ((uint32_t)((h & 3) * 32) << 16);
        const uint32_t row = a_work + (uint32_t)((h * N + lane) * kNS3) * 4u;    // lane = source j
#pragma unroll
        for (int c0 = 0; c0 < 32; c0 += 16) {
          uint32_t sm_[16], mn_[16];
          tmem_ld16(taddr + (uint32_t)c0, sm_);
          tmem_ld16(taddr + 32u + (uint32_t)c0, mn_);
          if (lane < N) {
#pragma unroll
            for (int e = 0; e < 16; e += 4)
              sts128a(row + (uint32_t)(c0 + e) * 4u,
                      make_float4((__uint_as_float(mn_[e]) + __uint_as_float(sm_[e])) * g_scale,
                                  (__uint_as_float(mn_[e + 1]) + __uint_as_float(sm_[e + 1])) * g_scale,
                                  (__uint_as_float(mn_[e + 2]) + __uint_as_float(sm_[e + 2])) * g_scale,
                                  (__uint_as_float(mn_[e + 3]) + __uint_as_float(sm_[e + 3])) * g_scale));
          }
        }
      }
      tc_fence_before();
      bar_sync<1, kSmT>();
      if (tid == 0) mbar_arrive(BAR(kBarDAEmpty));
      // ------------------------------------------------ softmax / LeakyReLU backward (thread = head h, target i) ------------------------------------------------
      float share = 0.f;
      if (on) {
        float dot = 0.f;
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (j < N) {
            float da = ldsa(col + (uint32_t)j * (kNS3 * 4));
            if (GA) {                                                          // (the second loop reads the sum back)
              da += __ldg(d_alpha + (((size_t)b * H + h) * N + j) * N + i);
              stsa(col + (uint32_t)j * (kNS3 * 4), da);
            }
            if (DROP) da = ((keep >> j) & 1u) ? da * p.drop.scale : 0.f;         // dalpha = m * d(alpha m)
            dot = fmaf(al[j], da, dot);
          }
        float dd = 0.f, dii = 0.f;
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (j < N) {
            float da = ldsa(col + (uint32_t)j * (kNS3 * 4));
            if (DROP) da = ((keep >> j) & 1u) ? da * p.drop.scale : 0.f;
            const float dl = al[j] * (da - dot);
            const float dz = ((mask >> j) & 1u) ? dl : dl * p.slope;
            stsa(col + (uint32_t)j * (kNS3 * 4), dz);
            dd += dz;
            if (j == i) dii = dz;
          }
        share = dii * inv_nm1;
        dsd_max = fmaxf(dsd_max, fabsf(dd));
        if (args.dsd) args.dsd[((size_t)b * N + i) * 2 * H + H + h] = dd;
        else args.dP_aug[((size_t)b * N + i) * p.ldp + HC + H + h] = dd;
      }
      bar_sync<1, kSmT>();
      if (on) {                                                                  // ds_j = row sum of dz (thread = head h, source j = lane)
        const uint32_t row = a_work + (uint32_t)((h * N + lane) * kNS3) * 4u;
        float ds = 0.f;
        for (int k = 0; k < N; ++k) ds += ldsa(row + (uint32_t)k * 4u);
        dsd_max = fmaxf(dsd_max, fabsf(ds));
        if (args.dsd) args.dsd[((size_t)b * N + lane) * 2 * H + h] = ds;
        else args.dP_aug[((size_t)b * N + lane) * p.ldp + HC + h] = ds;
      }
      bar_sync<1, kSmT>();
      if (on) {                                                                  // dz' = dz + dz_ii / (N - 1) off the diagonal, 0 on it
        for (int j = 0; j < N; ++j) {
          const uint32_t a = col + (uint32_t)j * (kNS3 * 4);
          stsa(a, j == i ? 0.f : ldsa(a) + share);
        }
      }
      bar_sync<1, kSmT>();
      if (p.dterms_out) {                                                        // edge_mode 1: d(edge terms) leaves in the tile layout
        float4* dst = reinterpret_cast<float4*>(p.dterms_out + (size_t)b * tile_floats);
        for (int idx = tid; idx < tile_floats / 4; idx += kSmT) dst[idx] = lds128a(a_work + (uint32_t)idx * 16u);
        bar_sync<1, kSmT>();
      }
      t_sb += clock64() - t_b0;
      // ------------------------------------------------ V: dv += dz'^T . edge rows (exact fp32 on the CUDA cores) ------------------------------------------------
      if (has_v) {
        // (a ring of fewer slots than G blocks + 2 could still hold an unfilled G block where the first V chunk goes)
        if (pl.n_slots <= pl.n_cb + 1) bar_wait_t(BAR(kBarAlphaEmpty), gph, w_vfull);
        float2 acc[4][kHP];
#pragma unroll
        for (int f = 0; f < 4; ++f)
#pragma unroll
          for (int k = 0; k < kHP; ++k) acc[f][k] = make_float2(0.f, 0.f);
        const uint32_t hstride = (uint32_t)(N * kNS3) * 4u;
        const bool f0_on = f0 < Fe, f1_on = f1 < Fe;
        for (int c = 0; c < pl.nchunks; ++c) {
          bar_wait_t(BAR(kBarFull + cur.slot), cur.ph, w_vfull);
          const long long t0 = clock64();
          const uint32_t sa = a_slots + (uint32_t)cur.slot * pl.slot_bytes;
          int rows = p.R - c * pl.chunk_rows;
          if (rows > pl.chunk_rows) rows = pl.chunk_rows;
          for (int rb = warp; rb < rows; rb += 2 * kSmWarps) {
            // two rows per round (rb, rb + 8), branch-free, loads first: table entries and the lane's four edge features, then
            // the H dz' values each entry points at.  A row past the chunk's end or skipped by the table contributes e = 0.
            int off[2];
            float2 e0[2], e1[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              const int r = min(rb + u * kSmWarps, rows - 1);
              off[u] = ldsa_s32(a_table + (uint32_t)(c * pl.chunk_rows + r) * 4u);
              e0[u] = f0_on ? lds64a(sa + (uint32_t)(r * Fe + f0) * 4u) : make_float2(0.f, 0.f);
              e1[u] = f1_on ? lds64a(sa + (uint32_t)(r * Fe + f1) * 4u) : make_float2(0.f, 0.f);
            }
            float z[2][2 * kHP];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              const bool ok = rb + u * kSmWarps < rows && off[u] >= 0;
              if (!ok) e0[u] = e1[u] = make_float2(0.f, 0.f);
              const uint32_t zb = a_work + (uint32_t)max(off[u], 0) * 4u;
#pragma unroll
              for (int hh = 0; hh < 2 * kHP; ++hh) z[u][hh] = hh < H ? ldsa(zb + (uint32_t)hh * hstride) : 0.f;
            }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
#pragma unroll
              for (int k = 0; k < kHP; ++k) {
                const float2 zz = make_float2(z[u][2 * k], z[u][2 * k + 1]);
                acc[0][k] = ffma2(make_float2(e0[u].x, e0[u].x), zz, acc[0][k]);
                acc[1][k] = ffma2(make_float2(e0[u].y, e0[u].y), zz, acc[1][k]);
                acc[2][k] = ffma2(make_float2(e1[u].x, e1[u].x), zz, acc[2][k]);
                acc[3][k] = ffma2(make_float2(e1[u].y, e1[u].y), zz, acc[3][k]);
              }
            }
          }
          bar_sync<1, kSmT>();
          if (tid == 0) mbar_arrive(BAR(kBarEmpty + cur.slot));
          cur.advance();
          t_v += clock64() - t0;
        }
        if (tid == 0) mbar_arrive(BAR(kBarVDone));
#pragma unroll
        for (int f = 0; f < 4; ++f)
#pragma unroll
          for (int k = 0; k < kHP; ++k) { run[f][k].x += acc[f][k].x; run[f][k].y += acc[f][k].y; }   // two-level sum
      }
    }
    if (args.dsd_amax) {
      for (int o = 16; o > 0; o >>= 1) dsd_max = fmaxf(dsd_max, __shfl_xor_sync(0xffffffffu, dsd_max, o));
      if (lane == 0 && dsd_max > 0.f) atomicMax(args.dsd_amax, __float_as_uint(dsd_max));
    }
    // per-CTA partials: dv_part[cta * kSmWarps + warp][h][f]
    if (has_v) {
      float* dst = args.dv_part + ((size_t)blockIdx.x * kSmWarps + warp) * H * Fe;
#pragma unroll
      for (int f = 0; f < 4; ++f) {
        const int feat = (f < 2 ? f0 : f1) + (f & 1);
        if (feat < Fe) {
#pragma unroll
          for (int k = 0; k < kHP; ++k) {
            if (2 * k < H) dst[(size_t)(2 * k) * Fe + feat] = run[f][k].x;
            if (2 * k + 1 < H) dst[(size_t)(2 * k + 1) * Fe + feat] = run[f][k].y;
          }
        }
      }
    }
    if (tid == 0) {
      atomicAdd(&g_bwd3_counters[9], (unsigned long long)w_vfull);
      atomicAdd(&g_bwd3_counters[10], (unsigned long long)t_v);
      atomicAdd(&g_bwd3_counters[11], (unsigned long long)w_t);
      atomicAdd(&g_bwd3_counters[13], (unsigned long long)t_sm);
      atomicAdd(&g_bwd3_counters[14], (unsigned long long)w_da);
      atomicAdd(&g_bwd3_counters[15], (unsigned long long)t_sb);
    }
  }
  // ---------------------------------------------------------------- teardown
  tc_fence_before();
  __syncthreads();
  if (warp == kWarpMma) tmem_dealloc(tmem_base, 512);
}
