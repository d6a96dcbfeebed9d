// Body of the pipelined attention backward (attn_bwd2.cu), included there twice: SPOTV2_KERNEL_NAME names the kernel and
// SPOTV2_GA = 1 makes the variant that takes d_alpha [B, H, N(j), N(i)], the gradient through the coefficients the forward
// returned (after dropout), which joins dalpha before the dropout factor.  Two kernels under their own names keep the
// machine code of the one without it exactly what it was.  No include guard: meant to be included more than once.
template <bool FIX, bool DROP, bool P16, bool SINGLE>
__global__ void __launch_bounds__(kB2Threads, 1)
SPOTV2_KERNEL_NAME(const AttnBwdArgs args, const Bwd2Plan pl_, const __grid_constant__ CUtensorMap tmP,
            const __grid_constant__ CUtensorMap tmG, const __grid_constant__ CUtensorMap tmPl,
            const __grid_constant__ CUtensorMap tmD0, const __grid_constant__ CUtensorMap tmD1
#if SPOTV2_GA
            , const float* __restrict__ d_alpha
#endif
) {
  constexpr bool GA = SPOTV2_GA != 0;
#if !SPOTV2_GA
  const float* const d_alpha = nullptr;
#endif
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  AttnParams p = args.p;
  Bwd2Plan pl = pl_;
  if (FIX) {
    using F = FixedGeom;
    p.N = F::N; p.H = F::H; p.C = F::C; p.Fe = F::Fe; p.R = F::R; p.ldp = F::ldp; p.ldo = F::ldo;
    p.concat = 0; p.bulk_ok = 1; p.vec2_ok = 1; p.hp = P16 ? 504 : F::C;
    pl.KS = F::KS; pl.chunk_rows = F::chunk_rows; pl.nchunks = F::nchunks; pl.n_cb = F::n_cb; pl.hpr = F::hpr;
    pl.n_rounds = F::n_rounds; pl.n_mt_chunk = F::n_mt_chunk; pl.ksplit = F::ksplit; pl.n_mtiles = F::n_mtiles;
    pl.dv_rg = F::dv_rg; pl.dv_rpu = F::dv_rpu; pl.dv_units = F::dv_units; pl.cbs_per_grp_d = F::cbs_per_grp_d;
    pl.n_slots = F::n_slots; pl.slot_bytes = F::slot_bytes; pl.tma_ok = 1;
  }
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = p.N, H = p.H, C = p.C, Fe = p.Fe;
  const int Cp = P16 ? p.hp : C;          // head pitch of the P / dP columns
  const int HC = H * Cp;
  constexpr int NS = kNS2;
  const int tile_floats = H * N * NS;

  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + pl.off_bar);
  uint64_t* full = bars;                // [kMaxSlots]
  uint64_t* empty = bars + kMaxSlots;   // [kMaxSlots]
  int32_t* table_s = reinterpret_cast<int32_t*>(smem_raw + pl.off_table);
  float4* vfrag = reinterpret_cast<float4*>(smem_raw + pl.off_vfrag);
  float* sd = reinterpret_cast<float*>(smem_raw + pl.off_sd);
  uint32_t* pos_mask = reinterpret_cast<uint32_t*>(smem_raw + pl.off_mask);
  uint32_t* keep_mask = pos_mask + ((H * N + 3) / 4) * 4;                  // [H][N] dropout keep bits (bit j = source j kept)
  float* ds_part = reinterpret_cast<float*>(smem_raw + pl.off_dspart);     // [2][H][32]
  float* dbias_s = reinterpret_cast<float*>(smem_raw + pl.off_dbias);
  float* tile = reinterpret_cast<float*>(smem_raw + pl.off_tile);          // alpha[h][j][i]
  float* D = reinterpret_cast<float*>(smem_raw + pl.off_D);                // dz'[h][j][i]
  unsigned char* slots = smem_raw + pl.off_slots;
  __builtin_assume(__isShared(table_s)); __builtin_assume(__isShared(vfrag)); __builtin_assume(__isShared(sd));
  __builtin_assume(__isShared(pos_mask)); __builtin_assume(__isShared(ds_part)); __builtin_assume(__isShared(dbias_s));
  __builtin_assume(__isShared(tile)); __builtin_assume(__isShared(D)); __builtin_assume(__isShared(slots));

  // edge_mode 1 (structured source): no edge rows at all - the edge terms come in, d(edge terms) goes out
  const int nchunks = p.terms_in ? 0 : pl.nchunks;
  // the forward kept the edge terms: phase L becomes a bulk copy of the tile (in slot-sized pieces) instead of a pass
  // over the edge rows
  const uint32_t tile_bytes = (uint32_t)tile_floats * 4u;
  const int term_pieces = (int)((tile_bytes + pl.slot_bytes - 1) / pl.slot_bytes);
  const bool use_terms = p.edge_terms != nullptr && (nchunks > 0 || p.terms_in);
  // the kept tile is the forward's record of signed attention coefficients (AttnParams::alpha_rec): phases L and S fall away
  const bool rec = P16 && !DROP && use_terms && p.alpha_rec != 0;
  const int my_graphs = (p.B - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const int n_cb = pl.n_cb;
  auto rows_in = [&](int c) { const int r = p.R - c * pl.chunk_rows; return r < pl.chunk_rows ? r : pl.chunk_rows; };

  if (tid == 0) {
    for (int s = 0; s < pl.n_slots; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], kW); }
    fence_mbar_init();
  }
  // row -> byte offset of (source j, target i) inside one head of the alpha / dz' tiles (-1: row skipped)
  for (int r = tid; r < p.R; r += kB2Threads) {
    const int code = (Fe > 0 && !p.terms_in) ? p.table[r] : -1;
    table_s[r] = code >= 0 ? ((code & 0xffff) * NS + (code >> 16)) * 4 : -1;
  }
  // slots start zero-filled: rows and tails a chunk does not cover must read as finite numbers
  for (uint32_t idx = tid; idx < (uint32_t)pl.n_slots * pl.slot_bytes / 16; idx += kB2Threads)
    reinterpret_cast<float4*>(smem_raw + pl.off_slots)[idx] = make_float4(0.f, 0.f, 0.f, 0.f);
  fence_proxy_async();                    // generic-proxy zero fill before the copy engine writes the same bytes
  if (Fe > 0 && !p.terms_in) build_vfrag(vfrag, p.v, H, Fe, pl.KS, 1, tid, kB2Threads);
  for (int idx = tid; idx < tile_floats; idx += kB2Threads) { tile[idx] = 0.f; D[idx] = 0.f; }
  for (int idx = tid; idx < p.ldo; idx += kB2Threads) dbias_s[idx] = 0.f;
  __syncthreads();

  if (warp == kW) {
    // =========================================== producer ===========================================
    if (lane == 0) { prefetch_tmap(&tmP); prefetch_tmap(&tmG); if (P16) { prefetch_tmap(&tmPl); prefetch_tmap(&tmD0); prefetch_tmap(&tmD1); } }
    const long long n_rows = (long long)p.B * N;
    // one tile: TMA, or (C % 4 != 0: tile starts are not 16-byte aligned) a cooperative gather into the
    // same swizzled layout
    auto put_tile = [&](unsigned char* dst, const CUtensorMap* tm, const float* base, int ld, int col0, int row0, uint64_t* full) {
      if (pl.tma_ok) {
        if (lane == 0) tma_load_2d_hint(dst, tm, col0, row0, full, kEvictFirst);
      } else {
        for (int idx = lane; idx < 32 * 32; idx += 32) {
          const int r = idx >> 5, c = idx & 31;
          float v = 0.f;
          if (row0 + r < n_rows && col0 + c < ld) v = base[((size_t)row0 + r) * ld + col0 + c];
          *reinterpret_cast<float*>(dst + r * 128 + ((((c >> 2) ^ (r & 7)) << 4) | ((c & 3) << 2))) = v;
        }
      }
    };
    int slot = 0;
    uint32_t sph = 0;
    auto acquire = [&]() -> unsigned char* {
      if (lane == 0) mbar_wait(&empty[slot], sph ^ 1);
      __syncwarp();
      return slots + (size_t)slot * pl.slot_bytes;
    };
    auto publish = [&](bool async_done) {          // async_done: completion comes from the copy engine's tx count
      if (!async_done) {
        __syncwarp();
        if (lane == 0) mbar_arrive(&full[slot]);
      }
      if (++slot == pl.n_slots) { slot = 0; sph ^= 1; }
    };
    auto edge_chunk = [&](int b, int c, uint64_t hint) {
      float* dst = reinterpret_cast<float*>(acquire());
      const int rows = rows_in(c);
      const float* src = p.edge_rows + ((size_t)b * p.R + (size_t)c * pl.chunk_rows) * Fe;
      if (p.bulk_ok) {
        if (lane == 0) {
          const uint32_t bytes = (uint32_t)rows * Fe * 4u;
          mbar_expect_tx(&full[slot], bytes);
          bulk_g2s_hint(dst, src, bytes, &full[slot], hint);
        }
      } else {
        for (int idx = lane; idx < rows * Fe; idx += 32) dst[idx] = src[idx];
      }
      publish(p.bulk_ok != 0);
    };
    const int n_grp_d = (n_cb + pl.cbs_per_grp_d - 1) / pl.cbs_per_grp_d;
    for (int it = 0; it < my_graphs; ++it) {
      const int b = blockIdx.x + it * gridDim.x;
      if (use_terms) {                                                          // phase L': the edge-term tile, slot-sized pieces
        for (int pc = 0; pc < term_pieces; ++pc) {
          float* dst = reinterpret_cast<float*>(acquire());
          if (lane == 0) {
            const uint32_t off = (uint32_t)pc * pl.slot_bytes;
            const uint32_t bytes = min(pl.slot_bytes, tile_bytes - off);
            mbar_expect_tx(&full[slot], bytes);
            bulk_g2s_hint(dst, reinterpret_cast<const unsigned char*>(p.edge_terms + (size_t)b * tile_floats) + off, bytes,
                          &full[slot], kEvictFirst);
          }
          publish(true);
        }
      } else {
        for (int c = 0; c < nchunks; ++c) edge_chunk(b, c, kEvictLast);         // phase L (kept in L2 for phase V)
      }
      for (int r = 0; r < pl.n_rounds; ++r) {                                   // phase A: one group per channel block
        const int h0 = r * pl.hpr;
        const int nh = min(pl.hpr, H - h0);
        for (int cb = 0; cb < n_cb; ++cb) {
          unsigned char* gb = acquire();
          if (P16) {
            // slot: [dout hi: hbd tiles][dout lo][P hi: hb tiles][P lo]   (hbd = hb for concat layers, 1 for the head mean)
            const int hbd = p.concat ? pl.hb : 1;
            const uint32_t planes = SINGLE ? 1u : 2u;
            if (lane == 0) {
              mbar_expect_tx(&full[slot], planes * (uint32_t)(hbd + pl.hb) * 2048u);
              tma_load_4d_hint(gb, p.concat ? &tmPl : &tmG, cb * 32, b * N, p.concat ? h0 : 0, 0, &full[slot], kEvictFirst);
              // (no eviction hint, 256-byte promotion: the 64-byte row pieces of heads that start mid-sector would otherwise be
              // fetched as two 64-byte DRAM bursts each; promoted lines are shared with the next channel block's box)
              tma_load_4d(gb + planes * (uint32_t)hbd * 2048u, &tmP, cb * 32, b * N, h0, 0, &full[slot]);
            }
          } else {
          const int ntiles = p.concat ? 2 * nh : 1 + nh;
          if (pl.tma_ok && lane == 0) mbar_expect_tx(&full[slot], (uint32_t)ntiles * kTile);
          if (p.concat) {
            for (int hl = 0; hl < nh; ++hl) {
              put_tile(gb + (2 * hl) * kTile, &tmG, args.dout, p.ldo, (h0 + hl) * C + cb * 32, b * N, &full[slot]);
              put_tile(gb + (2 * hl + 1) * kTile, &tmP, p.P_aug, p.ldp, (h0 + hl) * C + cb * 32, b * N, &full[slot]);
            }
          } else {
            put_tile(gb, &tmG, args.dout, p.ldo, cb * 32, b * N, &full[slot]);
            for (int hl = 0; hl < nh; ++hl)
              put_tile(gb + (1 + hl) * kTile, &tmP, p.P_aug, p.ldp, (h0 + hl) * C + cb * 32, b * N, &full[slot]);
          }
          }
          publish(pl.tma_ok != 0);
        }
      }
      for (int c = 0; c < nchunks; ++c) edge_chunk(b, c, kEvictFirst);          // phase V: second and last use
      for (int r = 0; r < pl.n_rounds; ++r) {                                   // phase D: groups of dO tiles
        const int h0 = r * pl.hpr;
        const int nh = min(pl.hpr, H - h0);
        for (int gi = 0; gi < n_grp_d; ++gi) {
          unsigned char* gb = acquire();
          const int cb0 = gi * pl.cbs_per_grp_d;
          const int ncb = min(pl.cbs_per_grp_d, n_cb - cb0);
          const int ntiles = p.concat ? ncb * nh : ncb;
          if (P16) {      // a tile = [hi 2 KB][lo 2 KB] from one load of the pair's one-head box
            if (lane == 0) {
              mbar_expect_tx(&full[slot], (uint32_t)ntiles * (SINGLE ? 2048u : 4096u));
              for (int k = 0; k < ncb; ++k) {
                if (p.concat) {
                  for (int hl = 0; hl < nh; ++hl)
                    tma_load_4d_hint(gb + (k * nh + hl) * kTile, &tmG, (cb0 + k) * 32, b * N, h0 + hl, 0, &full[slot], kEvictFirst);
                } else {
                  tma_load_4d_hint(gb + k * kTile, &tmG, (cb0 + k) * 32, b * N, 0, 0, &full[slot], kEvictFirst);
                }
              }
            }
          } else {
          if (pl.tma_ok && lane == 0) mbar_expect_tx(&full[slot], (uint32_t)ntiles * kTile);
          for (int k = 0; k < ncb; ++k) {
            if (p.concat) {
              for (int hl = 0; hl < nh; ++hl)
                put_tile(gb + (k * nh + hl) * kTile, &tmG, args.dout, p.ldo, (h0 + hl) * C + (cb0 + k) * 32, b * N, &full[slot]);
            } else {
              put_tile(gb + k * kTile, &tmG, args.dout, p.ldo, (cb0 + k) * 32, b * N, &full[slot]);
            }
          }
          }
          publish(pl.tma_ok != 0);
        }
      }
    }
    return;
  }

  // ============================================== compute ==============================================
  // All hot-loop addressing is done on 32-bit shared-window addresses computed once (generic pointers made
  // the compiler re-derive the window base before every access), swizzled tile offsets are folded into a
  // per-lane base plus an XOR with a compile-time constant, and table lookups return byte offsets.
  const int g = lane >> 2, t = lane & 3;
  const float g_scale = p.concat ? 1.f : 1.f / (float)H;
  const float inv_nm1 = 1.f / (float)(N > 1 ? N - 1 : 1);
  float dp_scale = 1.f;
  if (args.dP_hi16) {
    dp_scale = dp_scale_from_amax(__uint_as_float(*reinterpret_cast<const unsigned*>(args.dout_blk)) * args.bound);
    if (blockIdx.x == 0 && tid == 0) { args.dp_blk[2] = 1.f / dp_scale; args.dp_blk[4] = dp_scale; }
  }
  // fp16-pair operand scales of the two big products: dO and P from their tensors' maxima, alpha <= 1 fixed
  const float s_dO = dp_scale_from_amax(__uint_as_float(*reinterpret_cast<const unsigned*>(args.dout_blk)));
  const float s_P = P16 ? p.p_blk[4] : dp_scale_from_amax(__uint_as_float(*reinterpret_cast<const unsigned*>(args.p_amax)));
  constexpr float s_al = 16384.f;
  // (p_format 1: dout's pair carries one scale per graph | (graph, head): the two factors are rebuilt per unit)
  const float k_dalpha0 = g_scale / s_P, k_dp0 = g_scale * dp_scale / s_al * (DROP ? p.drop.scale : 1.f);
  float k_dalpha = k_dalpha0 / s_dO;                             // accumulator -> dalpha
  float k_dp = k_dp0 / s_dO;                                     // accumulator -> (scaled) dP
  const bool vec4_out = (C % 4 == 0);     // 8-byte aligned groups of 4 fp16 columns (ldp16 % 8 == 0)
  AttnSmem asm_{};                        // what softmax_phase reads
  asm_.NS = NS; asm_.KS = pl.KS; asm_.NT = 1;

  const uint32_t sbase = smem_u32(smem_raw);
  const uint32_t a_tile = sbase + pl.off_tile, a_D = sbase + pl.off_D, a_toff = sbase + pl.off_table;
  const uint32_t a_vfrag = sbase + pl.off_vfrag, a_slots = sbase + pl.off_slots, a_full = sbase + pl.off_bar;
  const uint32_t head_bytes = (uint32_t)(N * NS * 4);
  // fragment bases inside a 128B-swizzled 32x32 tile (row r, col c at r*128 + (((c>>2) ^ (r&7)) << 4) + (c&3)*4):
  //   row-major operand fragments (rows g / 8n+g, cols 8ks+t):  base ^ (ks << 5)  and  base ^ ((2ks+1) << 4)
  //   k-major operand fragments (rows 8ks+2t / +1, cols 8n+g):  base ^ (n << 5), + ks*1024
  //   row-major fp16-pair fragments (rows g / 8n+g, col pairs 16ks + 2t + 8hf):  base64 ^ ((4ks + 2hf) << 4)
  const uint32_t fb_row64 = (uint32_t)(g * 128 + ((g ^ (t >> 1)) << 4) + ((t & 1) << 3));
  // (MMA k index t <-> tile row 2t, t+4 <-> 2t+1: the 4 x 2 chunk slots of one load are then all distinct)
  const uint32_t fb_k0 = (uint32_t)((2 * t) * 128 + ((((g >> 2) ^ (2 * t))) << 4) + ((g & 3) << 2));
  const uint32_t fb_k1 = (uint32_t)((2 * t + 1) * 128 + ((((g >> 2) ^ (2 * t + 1))) << 4) + ((g & 3) << 2));

  // p_format 1, phase A: B fragments (k = channel pairs, n = source j) by ldmatrix.x4 from the [j][c] fp16 tile: matrix
  // = lane >> 3: (j 0-7, chunk 2ks) (j 0-7, chunk 2ks+1) (j 8-15, chunk 2ks) (j 8-15, chunk 2ks+1) = b0,b1 of n-block 2np
  // and b0,b1 of n-block 2np+1
  uint32_t lmB[2][2];                 // [k16 step][n pair]
#pragma unroll
  for (int ks = 0; ks < 2; ++ks)
#pragma unroll
    for (int np = 0; np < 2; ++np) lmB[ks][np] = sw64(16 * np + (lane & 7) + ((lane >> 4) & 1) * 8, 2 * ks + ((lane >> 3) & 1));
  // operand fragments of a [row][col] fp16 tile with 16 rows per block: matrix = lane >> 3, row = (lane & 7) + 8 * (matrix & 1),
  // chunk = matrix >> 1: A fragments (ldmatrix: rows = m, cols = k) and, transposed, B fragments of a [k][n] tile
  uint32_t lmX[2][2];                 // [16-row block][chunk pair]
#pragma unroll
  for (int rb = 0; rb < 2; ++rb)
#pragma unroll
    for (int cp = 0; cp < 2; ++cp) lmX[rb][cp] = sw64(16 * rb + (lane & 7) + ((lane >> 3) & 1) * 8, 2 * cp + (lane >> 4));
  // phase V units of this warp (feature tile, row group): fixed for the whole kernel
  int dv_mt[kMaxDvUnits], dv_rb[kMaxDvUnits];
  float dv_run[kMaxDvUnits][4];
#pragma unroll
  // (a warp's two units are neighbours: same row group whenever the feature-tile count is even, so that the dz' fragments
  // of a k-step are fetched and split once for both)
  for (int uu = 0; uu < kMaxDvUnits; ++uu) {
    const int u = warp * kMaxDvUnits + uu;
    const bool ok = u < pl.dv_units;
    dv_mt[uu] = ok ? u % pl.n_mtiles : -1;
    dv_rb[uu] = ok ? (u / pl.n_mtiles) * pl.dv_rpu : 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) dv_run[uu][q] = 0.f;
  }
  // phase L unit of this warp: half-group, row tile, k block start
  const int l_hg = warp / (kW / 2), l_w6 = warp - l_hg * (kW / 2);
  const int l_mt = pl.n_mt_chunk > 0 ? l_w6 % pl.n_mt_chunk : 0, l_kh = pl.n_mt_chunk > 0 ? l_w6 / pl.n_mt_chunk : 0;
  const bool l_on = pl.n_mt_chunk > 0 && l_kh < pl.ksplit;
  // MMA row g <-> chunk row 2g, row g+8 <-> 2g+1: with the 126-float row pitch the 8 even (odd) rows start 4 banks
  // apart, so the 32 lanes of a fragment load hit 32 distinct banks
  const uint32_t l_row0 = (uint32_t)(((l_mt * 16 + 2 * g) * Fe + t) * 4);
  const uint32_t l_hoff0 = (uint32_t)(2 * t) * head_bytes;

  // slot cursor: every compute warp walks the slots in the producer's order; the slot wait counts its polls (it reads no
  // clock) and traps after kSlotWaitSpins of them
  constexpr uint32_t kSlotWaitSpins = 1u << 24;
  int slot = 0;
  uint32_t sph = 0;
  auto wait_slot = [&]() -> uint32_t {
    const uint32_t bar = a_full + (uint32_t)slot * 8u;
    bool ok;
    uint32_t spins = 0;
    do {
      ok = mbar_try_wait(bar, sph);
      if (!ok && ++spins > kSlotWaitSpins) __trap();             // lost transaction: fail loudly, never hang the box
    } while (!ok);
    return a_slots + (uint32_t)slot * pl.slot_bytes;
  };
  auto release_slot = [&]() {
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[slot]);
    if (++slot == pl.n_slots) { slot = 0; sph ^= 1; }
  };

  float dsd_max = 0.f;                   // max |ds|, |dd| this thread wrote: sizes the fp16 scale of the ds|dd operand columns
  // phase cycle counters (spotv2_diag_counters, tools/fwd_waits.py): 14 registers that stay live across the whole kernel -
  // compiled in with -DSPOTV2_BRINGUP only (the product build spilled because of them)
#ifdef SPOTV2_BRINGUP
  long long ph[6] = {0, 0, 0, 0, 0, 0};
  long long t_ph = clock64();
  auto lap = [&](int k) { const long long now = clock64(); ph[k] += now - t_ph; t_ph = now; };
#else
  auto lap = [&](int) {};
#endif

  for (int it = 0; it < my_graphs; ++it) {
    const int b = blockIdx.x + it * gridDim.x;
    // ------------------------------------------------ L: edge logits ------------------------------------------------
    if (!rec)
    for (int idx = tid; idx < N * 2 * H; idx += kCT) {
      const int j = idx / (2 * H), k = idx - j * 2 * H;
      if (P16) {
        sd[idx] = p.sd32[((size_t)b * N + j) * 2 * H + k];
      } else {
        sd[idx] = p.P_aug[((size_t)b * N + j) * p.ldp + HC + k];
      }
    }
    for (int idx = tid; idx < 2 * H * 32; idx += kCT) ds_part[idx] = 0.f;
    if (use_terms) {
      for (int pc = 0; pc < term_pieces; ++pc) {
        const uint32_t sa = wait_slot();
        const uint32_t off = (uint32_t)pc * pl.slot_bytes;
        const int n16 = (int)(min(pl.slot_bytes, tile_bytes - off) / 16u);
        float4* dst = reinterpret_cast<float4*>(reinterpret_cast<unsigned char*>(tile) + off);
        for (int idx = tid; idx < n16; idx += kCT) dst[idx] = lds128a(sa + (uint32_t)idx * 16u);
        release_slot();
      }
    }
    for (int c = 0; c < (use_terms ? 0 : nchunks); ++c) {
      const uint32_t sa = wait_slot();
      const int rows = rows_in(c);
      if (l_on && (c & 1) == l_hg && l_mt * 16 < rows) {
        // 16 rows x this warp's k blocks (4 k-steps each), 3xTF32; features past Fe meet zero B fragments
        // (k-blocks reaching past Fe are masked below)
        float acc[3][4];
#pragma unroll
        for (int pr = 0; pr < 3; ++pr)
#pragma unroll
          for (int q = 0; q < 4; ++q) acc[pr][q] = 0.f;
        const uint32_t r0 = sa + l_row0, r1 = r0 + (uint32_t)(Fe * 4);
        for (int kb = l_kh; kb < pl.KS / 4; kb += pl.ksplit) {
          const uint32_t ko = (uint32_t)kb * 128u;                 // 4 k-steps x 8 features x 4 bytes
          const uint32_t vf = a_vfrag + ((uint32_t)(kb * 4) * 32u + (uint32_t)lane) * 16u;
          float a[4][4];
          float4 bf[4];
#pragma unroll
          for (int sl = 0; sl < 4; ++sl) {
            a[sl][0] = ldsa(r0 + ko + sl * 32);
            a[sl][1] = ldsa(r1 + ko + sl * 32);
            a[sl][2] = ldsa(r0 + ko + sl * 32 + 16);
            a[sl][3] = ldsa(r1 + ko + sl * 32 + 16);
            bf[sl] = lds128a(vf + sl * 512);
          }
          if ((kb + 1) * 32 > Fe) {
            // k-steps reaching past Fe: whatever lies there (stale slot bytes) must not meet the zero B
            // fragments as NaN/Inf
#pragma unroll
            for (int sl = 0; sl < 4; ++sl) {
              const int f = kb * 32 + sl * 8 + t;
              if (f >= Fe) a[sl][0] = a[sl][1] = 0.f;
              if (f + 4 >= Fe) a[sl][2] = a[sl][3] = 0.f;
            }
          }
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
        }
        // k half 0 stores into the alpha tile, k half 1 into the (idle) dz' tile; the softmax adds them: no atomics,
        // fixed summation order
        const int rl = l_mt * 16 + 2 * g, row_base = c * pl.chunk_rows + rl;
        const int to0 = rl < rows ? ldsa_s32(a_toff + (uint32_t)row_base * 4u) : -1;
        const int to1 = rl + 1 < rows ? ldsa_s32(a_toff + (uint32_t)(row_base + 1) * 4u) : -1;
        const float v0 = (acc[0][0] + acc[1][0]) + acc[2][0], v1 = (acc[0][1] + acc[1][1]) + acc[2][1];
        const float v2 = (acc[0][2] + acc[1][2]) + acc[2][2], v3 = (acc[0][3] + acc[1][3]) + acc[2][3];
        const uint32_t tb = (l_kh == 0 ? a_tile : a_D) + l_hoff0;
        if (to0 >= 0) {
          if (2 * t < H) stsa(tb + (uint32_t)to0, v0);
          if (2 * t + 1 < H) stsa(tb + head_bytes + (uint32_t)to0, v1);
        }
        if (to1 >= 0) {
          if (2 * t < H) stsa(tb + (uint32_t)to1, v2);
          if (2 * t + 1 < H) stsa(tb + head_bytes + (uint32_t)to1, v3);
        }
      }
      release_slot();
    }
    bar_sync<1, kCT>();
    lap(0);
    // ------------------------------------------------ S: softmax ------------------------------------------------
    // (the forward's record already IS the result of this phase: signed attention coefficients)
    if (!rec) {
      softmax_phase(p, asm_, tile, sd, 1.f, nullptr, pos_mask, tid, kCT, -1, 0, (nchunks > 0 && pl.ksplit == 2 && !use_terms) ? D : nullptr);
      bar_sync<1, kCT>();
    }
    lap(1);
    // ------------------------------------------------ A: dalpha + softmax backward ------------------------------------------------
    for (int r = 0; r < pl.n_rounds; ++r) {
      const int h0 = r * pl.hpr;
      const int nh = min(pl.hpr, H - h0);
      const int hl = warp >> 1, m = warp & 1;
      const bool active = (warp < 2 * nh) && (16 * m < N);
      const int h = h0 + hl;
      if (P16) {
        const float sdo = active ? args.dO_scale[(size_t)b * args.units_per_graph + (p.concat ? h : 0)] : 1.f;
        k_dalpha = k_dalpha0 / sdo;
      }
      const uint32_t d_off = (uint32_t)((p.concat ? 2 * hl : 0) * kTile + m * 2048) + fb_row64;
      const uint32_t p_off = (uint32_t)((p.concat ? 2 * hl + 1 : 1 + hl) * kTile) + fb_row64;
      const int i0 = 16 * m + g, i1 = i0 + 8;
      float cacc[4][4], dacc[4][4];
#pragma unroll
      for (int n = 0; n < 4; ++n)
#pragma unroll
        for (int q = 0; q < 4; ++q) cacc[n][q] = dacc[n][q] = 0.f;
      for (int cb = 0; cb < n_cb; ++cb) {
        const uint32_t sa = wait_slot();
        if (active) {
          const uint32_t da = sa + d_off, pa = sa + p_off;
          const bool tail = (cb * 32 + 32 > C);          // channels beyond C: next head's columns (concat) or padding
          uint32_t ah[2][4], al[2][4];
          if (P16) {
            // slot: [dout hi: hbd tiles][dout lo][P hi: hb tiles][P lo]; A fragments (rows = targets 16m.., k = channels)
            const uint32_t hbd = p.concat ? (uint32_t)pl.hb : 1u, planes = SINGLE ? 1u : 2u;
            const uint32_t dt = sa + (p.concat ? (uint32_t)hl * 2048u : 0u);
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
              ldsm_x4(dt + lmX[m][ks], ah[ks][0], ah[ks][1], ah[ks][2], ah[ks][3]);
              if (!SINGLE) ldsm_x4(dt + hbd * 2048u + lmX[m][ks], al[ks][0], al[ks][1], al[ks][2], al[ks][3]);
            }
            const uint32_t pt = sa + planes * hbd * 2048u + (uint32_t)hl * 2048u, plo = (uint32_t)pl.hb * 2048u;
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
#pragma unroll
              for (int np = 0; np < 2; ++np) {
                uint32_t bh[4], bl[4];
                ldsm_x4(pt + lmB[ks][np], bh[0], bh[1], bh[2], bh[3]);
                if (!SINGLE) ldsm_x4(pt + plo + lmB[ks][np], bl[0], bl[1], bl[2], bl[3]);
#pragma unroll
                for (int nn = 0; nn < 2; ++nn) {
                  const int n = 2 * np + nn;
                  if (!SINGLE) {
                    mma_f16_k16(cacc[n], al[ks], bh[2 * nn], bh[2 * nn + 1]);        // small terms first
                    mma_f16_k16(cacc[n], ah[ks], bl[2 * nn], bl[2 * nn + 1]);
                  }
                  mma_f16_k16(cacc[n], ah[ks], bh[2 * nn], bh[2 * nn + 1]);
                }
              }
            }
          } else {
#pragma unroll
          for (int ks = 0; ks < 2; ++ks) {
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
              const uint32_t ad = da ^ ((4 * ks + 2 * hf) << 4);
              float2 x0 = lds64a(ad), x1 = lds64a(ad + 1024);
              if (tail) {
                const int c = cb * 32 + 16 * ks + 8 * hf + 2 * t;
                if (c >= C) x0.x = x1.x = 0.f;
                if (c + 1 >= C) x0.y = x1.y = 0.f;
              }
              cvt_pair(x0.x, x0.y, s_dO, ah[ks][2 * hf], al[ks][2 * hf]);
              cvt_pair(x1.x, x1.y, s_dO, ah[ks][2 * hf + 1], al[ks][2 * hf + 1]);
            }
          }
#pragma unroll
          for (int ks = 0; ks < 2; ++ks) {
#pragma unroll
            for (int n = 0; n < 4; ++n) {
              uint32_t bh[2], bl[2];
#pragma unroll
              for (int hf = 0; hf < 2; ++hf) {
                float2 y = lds64a((pa ^ ((4 * ks + 2 * hf) << 4)) + n * 1024);
                if (tail) {                                // never let padding bits (possibly NaN) meet the zeros above
                  const int c = cb * 32 + 16 * ks + 8 * hf + 2 * t;
                  if (c >= C) y.x = 0.f;
                  if (c + 1 >= C) y.y = 0.f;
                }
                cvt_pair(y.x, y.y, s_P, bh[hf], bl[hf]);
              }
              mma_f16_k16(cacc[n], al[ks], bh[0], bh[1]);  // small terms first
              mma_f16_k16(cacc[n], ah[ks], bl[0], bl[1]);
              mma_f16_k16(cacc[n], ah[ks], bh[0], bh[1]);
            }
          }
          }
        }
        release_slot();
        if (active && ((cb & 3) == 3 || cb == n_cb - 1)) {  // keep tensor-core accumulation chains short: fold in fp32 RN
#pragma unroll
          for (int n = 0; n < 4; ++n)
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              dacc[n][q] += cacc[n][q];
              cacc[n][q] = 0.f;
            }
        }
      }
      if (active) {
        // softmax / LeakyReLU backward on the fragment: lane holds rows i0, i1 and columns j = 8n + 2t + {0,1}
        float al_[4][4];
        float dot0 = 0.f, dot1 = 0.f;
        // this lane's 16 entries of d_alpha (targets i0 | i1, sources 8n + 2t + {0,1}), all loads in flight at once (loaded
        // before the slot loop instead, they stay live across it and the default-geometry instantiations spill)
        float ga[4][4];
        if (GA) {
#pragma unroll
          for (int n = 0; n < 4; ++n)
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const int i = (q & 2) ? i1 : i0, j = 8 * n + 2 * t + (q & 1);
              ga[n][q] = (i < N && j < N) ? __ldg(d_alpha + (((size_t)b * H + h) * N + j) * N + i) : 0.f;
            }
        }
        uint32_t keep0 = 0xffffffffu, keep1 = 0xffffffffu;
        if (DROP) {
          // the forward used alpha * m (m = keep / (1 - p)): dalpha = m * d(alpha m); the bits also go to shared memory
          // for phase D, which needs alpha * m
          if (i0 < N) keep0 = dropout_keep_bits(p.drop, (((unsigned long long)b * H + h) * N + i0) * N, N);
          if (i1 < N) keep1 = dropout_keep_bits(p.drop, (((unsigned long long)b * H + h) * N + i1) * N, N);
          if (t == 0) {
            if (i0 < N) keep_mask[h * N + i0] = keep0;
            if (i1 < N) keep_mask[h * N + i1] = keep1;
          }
        }
#pragma unroll
        for (int n = 0; n < 4; ++n)
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int i = (q & 2) ? i1 : i0, j = 8 * n + 2 * t + (q & 1);
            const bool valid = i < N && j < N;
            // al_ keeps the coefficient with the LeakyReLU side in its sign (the record's convention: negative = z <= 0)
            const float ar = valid ? tile[(h * N + j) * NS + i] : 0.f;
            const float a = fabsf(ar);
            float da = valid ? dacc[n][q] * k_dalpha : 0.f;
            if (GA) da += ga[n][q];
            if (DROP) da = ((((q & 2) ? keep1 : keep0) >> j) & 1u) ? da * p.drop.scale : 0.f;
            al_[n][q] = ar;
            dacc[n][q] = da;
            if (q & 2) dot1 = fmaf(a, da, dot1); else dot0 = fmaf(a, da, dot0);
          }
        dot0 += __shfl_xor_sync(0xffffffffu, dot0, 1); dot0 += __shfl_xor_sync(0xffffffffu, dot0, 2);
        dot1 += __shfl_xor_sync(0xffffffffu, dot1, 1); dot1 += __shfl_xor_sync(0xffffffffu, dot1, 2);
        uint32_t mask0 = 0u, mask1 = 0u;
        if (!rec) { mask0 = i0 < N ? pos_mask[h * N + i0] : 0u; mask1 = i1 < N ? pos_mask[h * N + i1] : 0u; }
        float dd0 = 0.f, dd1 = 0.f, dii0 = 0.f, dii1 = 0.f;
        float dsc[4][2];
#pragma unroll
        for (int n = 0; n < 4; ++n) {
          dsc[n][0] = dsc[n][1] = 0.f;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int i = (q & 2) ? i1 : i0, j = 8 * n + 2 * t + (q & 1);
            const float dl = fabsf(al_[n][q]) * (dacc[n][q] - ((q & 2) ? dot1 : dot0));
            const uint32_t mk = (q & 2) ? mask1 : mask0;
            const bool pos = rec ? !(__float_as_uint(al_[n][q]) >> 31) : (((mk >> j) & 1u) != 0u);
            const float dz = pos ? dl : dl * p.slope;
            dacc[n][q] = dz;
            if (q & 2) { dd1 += dz; if (j == i) dii1 = dz; } else { dd0 += dz; if (j == i) dii0 = dz; }
            dsc[n][q & 1] += dz;
          }
        }
        dd0 += __shfl_xor_sync(0xffffffffu, dd0, 1); dd0 += __shfl_xor_sync(0xffffffffu, dd0, 2);
        dd1 += __shfl_xor_sync(0xffffffffu, dd1, 1); dd1 += __shfl_xor_sync(0xffffffffu, dd1, 2);
        dii0 += __shfl_xor_sync(0xffffffffu, dii0, 1); dii0 += __shfl_xor_sync(0xffffffffu, dii0, 2);
        dii1 += __shfl_xor_sync(0xffffffffu, dii1, 1); dii1 += __shfl_xor_sync(0xffffffffu, dii1, 2);
        if (t == 0) {
          if (i0 < N) {
            dsd_max = fmaxf(dsd_max, fabsf(dd0));
            if (args.dsd) args.dsd[((size_t)b * N + i0) * 2 * H + H + h] = dd0;
            else args.dP_aug[((size_t)b * N + i0) * p.ldp + HC + H + h] = dd0;
          }
          if (i1 < N) {
            dsd_max = fmaxf(dsd_max, fabsf(dd1));
            if (args.dsd) args.dsd[((size_t)b * N + i1) * 2 * H + H + h] = dd1;
            else args.dP_aug[((size_t)b * N + i1) * p.ldp + HC + H + h] = dd1;
          }
        }
        // ds partial over this warp's 16 targets: sum over the 8 row groups (lane bits 2..4)
#pragma unroll
        for (int n = 0; n < 4; ++n)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            float v = dsc[n][e];
            v += __shfl_xor_sync(0xffffffffu, v, 4);
            v += __shfl_xor_sync(0xffffffffu, v, 8);
            v += __shfl_xor_sync(0xffffffffu, v, 16);
            if (g == 0) ds_part[(m * H + h) * 32 + 8 * n + 2 * t + e] = v;
          }
        // dz' = dz + dz_ii / (N - 1) off the diagonal, 0 on it (gradient through the mean fill)
        const float sh0 = dii0 * inv_nm1, sh1 = dii1 * inv_nm1;
#pragma unroll
        for (int n = 0; n < 4; ++n)
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int i = (q & 2) ? i1 : i0, j = 8 * n + 2 * t + (q & 1);
            if (i < N && j < N) D[(h * N + j) * NS + i] = (j == i) ? 0.f : dacc[n][q] + ((q & 2) ? sh1 : sh0);
          }
      }
    }
    bar_sync<1, kCT>();
    lap(2);
    for (int idx = tid; idx < H * N; idx += kCT) {       // ds_j = sum over both target tiles
      const int h = idx / N, j = idx - h * N;
      const float ds = ds_part[h * 32 + j] + ds_part[(H + h) * 32 + j];
      dsd_max = fmaxf(dsd_max, fabsf(ds));
      if (args.dsd) args.dsd[((size_t)b * N + j) * 2 * H + h] = ds;
      else args.dP_aug[((size_t)b * N + j) * p.ldp + HC + h] = ds;
    }
    lap(3);
    if (p.dterms_out) {
      // edge_mode 1: the gradient w.r.t. the edge terms (dz', diagonal 0) leaves in the tile layout; dv is formed from
      // the windows by spotv2_windows_dv.  (The D tile is complete: phase A ended with a CTA barrier.)
      float4* dst = reinterpret_cast<float4*>(p.dterms_out + (size_t)b * tile_floats);
      const float4* src = reinterpret_cast<const float4*>(D);
      for (int idx = tid; idx < tile_floats / 4; idx += kCT) dst[idx] = src[idx];
    }
    // ------------------------------------------------ V: dv += dz'^T . edge rows ------------------------------------------------
    for (int c = 0; c < nchunks; ++c) {
      const uint32_t sa = wait_slot();
      const int rows = rows_in(c);
      const uint32_t trow = a_toff + (uint32_t)(c * pl.chunk_rows) * 4u;
      const uint32_t dgh = a_D + (uint32_t)g * head_bytes;                   // head g of the dz' tile (B fragment: n = g)
      static_assert(kMaxDvUnits == 2, "phase V pairs the two units of a warp");
      if (pl.dv_rpu == 16 && dv_mt[1] >= 0 && dv_rb[0] == dv_rb[1]) {
        // Both units cover the same 16 rows (feature tiles mt, mt + 1).  A = T^T: (m = feature f0 + g | + 8, k = row).
        // k index -> chunk row: k-step s takes rows 4t + 2s (k = t) and 4t + 2s + 1 (k = t + 4): rows 4 apart start 8 banks
        // apart with the 126-float pitch, so a fragment load (4 rows x 8 features) is conflict-free.  The B fragments (dz' of
        // the rows' edges, n = head g) are fetched through the row table and split once per k-step for both tiles; all
        // operand loads of the four (tile, k-step) products are issued before the first split.
        const int rbeg = dv_rb[0];
        if (rbeg < rows) {                                                    // warp-uniform
          const int rend = min(rows, rbeg + 16);
          const uint32_t rowb = (uint32_t)(Fe * 4);
          const int r4 = rbeg + 4 * t;
          int to[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) to[k] = (r4 + k < rend && g < H) ? ldsa_s32(trow + (uint32_t)(r4 + k) * 4u) : -1;
          float a[2][2][4];                                                   // [tile][k-step][fragment register]
#pragma unroll
          for (int uu = 0; uu < 2; ++uu) {
            const uint32_t ta0 = sa + (uint32_t)r4 * rowb + (uint32_t)((dv_mt[uu] * 16 + g) * 4);
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
              const uint32_t ta = ta0 + (uint32_t)(2 * ks) * rowb, tb = ta + rowb;
              a[uu][ks][0] = ldsa(ta);
              a[uu][ks][1] = ldsa(ta + 32);
              a[uu][ks][2] = ldsa(tb);
              a[uu][ks][3] = ldsa(tb + 32);
            }
          }
          float bv[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) bv[k] = to[k] >= 0 ? ldsa(dgh + (uint32_t)to[k]) : 0.f;
          if (rend < rbeg + 16) {                // rows past the chunk's end hold stale slot bytes
#pragma unroll
            for (int uu = 0; uu < 2; ++uu)
#pragma unroll
              for (int ks = 0; ks < 2; ++ks) {
                if (r4 + 2 * ks >= rend) a[uu][ks][0] = a[uu][ks][1] = 0.f;
                if (r4 + 2 * ks + 1 >= rend) a[uu][ks][2] = a[uu][ks][3] = 0.f;
              }
          }
          uint32_t bh[2][2], bl[2][2];
#pragma unroll
          for (int ks = 0; ks < 2; ++ks) {
            split_lean(bv[2 * ks], bh[ks][0], bl[ks][0]);
            split_lean(bv[2 * ks + 1], bh[ks][1], bl[ks][1]);
          }
#pragma unroll
          for (int uu = 0; uu < 2; ++uu) {
            float acc[3][4];
#pragma unroll
            for (int pr = 0; pr < 3; ++pr)
#pragma unroll
              for (int q = 0; q < 4; ++q) acc[pr][q] = 0.f;
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
              uint32_t ah[4], al[4];
#pragma unroll
              for (int q = 0; q < 4; ++q) split_lean(a[uu][ks][q], ah[q], al[q]);
              mma_tf32_16x8x8(acc[0], al, bh[ks]);
              mma_tf32_16x8x8(acc[1], ah, bl[ks]);
              mma_tf32_16x8x8(acc[2], ah, bh[ks]);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) dv_run[uu][q] += (acc[0][q] + acc[1][q]) + acc[2][q];
          }
        }
      } else {
#pragma unroll
      for (int uu = 0; uu < kMaxDvUnits; ++uu) {
        if (dv_mt[uu] < 0 || dv_rb[uu] >= rows) continue;                    // warp-uniform
        const int rbeg = dv_rb[uu], rend = min(rows, rbeg + pl.dv_rpu);
        const bool partial = rend < rbeg + pl.dv_rpu;
        // A = T^T: (m = feature f0 + g | + 8, k = row r0 + t | + 4).  Features past Fe only feed discarded
        // output rows; rows past rend are masked (they also meet zero B fragments).
        // k index -> chunk row.  16-row units (the default): k-step s takes rows 4t + 2s (k = t) and 4t + 2s + 1
        // (k = t+4): rows 4 apart start 8 banks apart with the 126-float pitch, so a fragment load (4 rows x 8
        // features) is conflict-free.  Other unit sizes: natural order (t, t+4), 8 rows per k-step.
        const bool perm = pl.dv_rpu == 16;
        const uint32_t fcol = (uint32_t)((dv_mt[uu] * 16 + g) * 4);
        const uint32_t rowb = (uint32_t)(Fe * 4);
        float acc[3][4];
#pragma unroll
        for (int pr = 0; pr < 3; ++pr)
#pragma unroll
          for (int q = 0; q < 4; ++q) acc[pr][q] = 0.f;
        auto kstep = [&](int ra, int rb, uint32_t ta, uint32_t tb) {
          const int to0 = (ra < rend && g < H) ? ldsa_s32(trow + (uint32_t)ra * 4u) : -1;
          const int to1 = (rb < rend && g < H) ? ldsa_s32(trow + (uint32_t)rb * 4u) : -1;
          const float b0 = to0 >= 0 ? ldsa(dgh + (uint32_t)to0) : 0.f;
          const float b1 = to1 >= 0 ? ldsa(dgh + (uint32_t)to1) : 0.f;
          uint32_t bh[2], bl[2];
          split_lean(b0, bh[0], bl[0]);
          split_lean(b1, bh[1], bl[1]);
          float a[4];
          a[0] = ldsa(ta);
          a[1] = ldsa(ta + 32);
          a[2] = ldsa(tb);
          a[3] = ldsa(tb + 32);
          if (partial) {                         // rows past the chunk's end hold stale slot bytes
            if (ra >= rend) a[0] = a[1] = 0.f;
            if (rb >= rend) a[2] = a[3] = 0.f;
          }
          uint32_t ah[4], al[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) split_lean(a[q], ah[q], al[q]);
          mma_tf32_16x8x8(acc[0], al, bh);
          mma_tf32_16x8x8(acc[1], ah, bl);
          mma_tf32_16x8x8(acc[2], ah, bh);
        };
        if (perm) {
          const int r4 = rbeg + 4 * t;
          const uint32_t ta0 = sa + (uint32_t)r4 * rowb + fcol;
          kstep(r4, r4 + 1, ta0, ta0 + rowb);
          kstep(r4 + 2, r4 + 3, ta0 + 2 * rowb, ta0 + 3 * rowb);
        } else {
          uint32_t ta = sa + (uint32_t)(rbeg + t) * rowb + fcol;
          for (int r0 = rbeg; r0 < rend; r0 += 8, ta += 8 * rowb) kstep(r0 + t, r0 + t + 4, ta, ta + 4 * rowb);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) dv_run[uu][q] += (acc[0][q] + acc[1][q]) + acc[2][q];
      }
      }
      release_slot();
    }
    lap(5);
    // (the dP staging tiles reuse the dz' tile: every warp must be done reading it - phase V, or the edge_mode 1 copy-out)
    if (P16 && pl.stage_ok) bar_sync<1, kCT>();
    // ------------------------------------------------ D: dP = g alpha^T dO ------------------------------------------------
    for (int r = 0; r < pl.n_rounds; ++r) {
      const int h0 = r * pl.hpr;
      const int nh = min(pl.hpr, H - h0);
      const int hl = warp >> 1, m = warp & 1;
      const bool active = (warp < 2 * nh) && (16 * m < N);
      const int h = h0 + hl;
      const int j0 = 16 * m + g, j1 = j0 + 8;
      if (P16) {
        const float sdo = active ? args.dO_scale[(size_t)b * args.units_per_graph + (p.concat ? h : 0)] : 1.f;
        k_dp = k_dp0 / sdo;
      }
      uint32_t ah[2][4], al[2][4];
      if (active) {
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
#pragma unroll
          for (int hf = 0; hf < 2; ++hf) {
            const int ia = 16 * ks + 8 * hf + 2 * t;               // k pair (ia, ia+1) = target rows of dO
            const float2 z = make_float2(0.f, 0.f);
            float2 x0 = j0 < N ? *reinterpret_cast<const float2*>(&tile[(h * N + j0) * NS + ia]) : z;
            float2 x1 = j1 < N ? *reinterpret_cast<const float2*>(&tile[(h * N + j1) * NS + ia]) : z;
            if (DROP) {            // alpha[h][source j][target ia | ia+1] * m: keep bits of the TARGET rows, bit = source
              const uint32_t ka = ia < N ? keep_mask[h * N + ia] : 0u, kb = ia + 1 < N ? keep_mask[h * N + ia + 1] : 0u;
              // the 1/(1-p) factor rides in k_dp (fp32 post-scale), never in the fp16 operand: alpha/(1-p) * 2^14
              // would leave the fp16 range from p = 0.75 on
              x0.x = ((ka >> j0) & 1u) ? x0.x : 0.f;
              x0.y = ((kb >> j0) & 1u) ? x0.y : 0.f;
              x1.x = ((ka >> j1) & 1u) ? x1.x : 0.f;
              x1.y = ((kb >> j1) & 1u) ? x1.y : 0.f;
            }
            cvt_pair(fabsf(x0.x), fabsf(x0.y), s_al, ah[ks][2 * hf], al[ks][2 * hf]);         // (record: sign = LeakyReLU side)
            cvt_pair(fabsf(x1.x), fabsf(x1.y), s_al, ah[ks][2 * hf + 1], al[ks][2 * hf + 1]);
          }
      }
      uint32_t carry_h[2] = {0u, 0u}, carry_l[2] = {0u, 0u};     // last 8-column chunk of the previous dP tile (shifted stores)
      const int n_grp = (n_cb + pl.cbs_per_grp_d - 1) / pl.cbs_per_grp_d;
      for (int gi = 0; gi < n_grp; ++gi) {
        const uint32_t sa = wait_slot();
        const int cb0 = gi * pl.cbs_per_grp_d;
        const int ncb = min(pl.cbs_per_grp_d, n_cb - cb0);
        // dbias: column sums of the staged dO tiles, one tile per warp, one column per lane (tiles of the shared
        // dO in head-mean mode are summed in round 0 only)
        if (!P16 && (p.concat || r == 0)) {
          const int n_t = p.concat ? ncb * nh : ncb;
          for (int k = warp; k < n_t; k += kW) {
            const int kc = p.concat ? k / nh : k, khl = p.concat ? k - kc * nh : 0;
            const uint32_t ta = sa + (uint32_t)k * kTile;
            float sum = 0.f;
            for (int rr = 0; rr < N; ++rr)
              sum += ldsa(ta + rr * 128 + ((((lane >> 2) ^ (rr & 7)) << 4) | ((lane & 3) << 2)));
            const int c = (cb0 + kc) * 32 + lane;
            if (c < C) dbias_s[(p.concat ? (h0 + khl) * C : 0) + c] += sum;       // one owner lane per column
          }
        }
        if (active) {
          for (int k = 0; k < ncb; ++k) {
            const int cb = cb0 + k;
            const uint32_t ta = sa + (uint32_t)(p.concat ? k * nh + hl : k) * kTile;
            const uint32_t tb0 = ta + fb_k0, tb1 = ta + fb_k1;
            float cacc[4][4];
#pragma unroll
            for (int n = 0; n < 4; ++n)
#pragma unroll
              for (int q = 0; q < 4; ++q) cacc[n][q] = 0.f;
            if (P16) {
              // B fragments (k = target rows of dO, n = channels) of the [i][c] fp16 tile by ldmatrix.trans: hi at ta, lo + 2 KB
#pragma unroll
              for (int ks = 0; ks < 2; ++ks) {
#pragma unroll
                for (int np = 0; np < 2; ++np) {
                  uint32_t bh[4], bl[4];
                  ldsm_x4_t(ta + lmX[ks][np], bh[0], bh[1], bh[2], bh[3]);
                  if (!SINGLE) ldsm_x4_t(ta + 2048 + lmX[ks][np], bl[0], bl[1], bl[2], bl[3]);
#pragma unroll
                  for (int nn = 0; nn < 2; ++nn) {
                    const int n = 2 * np + nn;
                    if (!SINGLE) {
                      mma_f16_k16(cacc[n], al[ks], bh[2 * nn], bh[2 * nn + 1]);      // small terms first
                      mma_f16_k16(cacc[n], ah[ks], bl[2 * nn], bl[2 * nn + 1]);
                    }
                    mma_f16_k16(cacc[n], ah[ks], bh[2 * nn], bh[2 * nn + 1]);
                  }
                }
              }
            } else
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
#pragma unroll
              for (int n = 0; n < 4; ++n) {
                // k pairs (2t, 2t+1) and (2t+8, 2t+9) of this k16 step = dO rows 16ks + ...; column 8n + g
                const uint32_t a0 = (tb0 ^ (n << 5)) + ks * 2048, a1 = (tb1 ^ (n << 5)) + ks * 2048;
                const float x0 = ldsa(a0), x1 = ldsa(a1), x2 = ldsa(a0 + 1024), x3 = ldsa(a1 + 1024);
                uint32_t bh[2], bl[2];
                cvt_pair(x0, x1, s_dO, bh[0], bl[0]);
                cvt_pair(x2, x3, s_dO, bh[1], bl[1]);
                if (!(P16 && SINGLE)) {
                  mma_f16_k16(cacc[n], al[ks], bh[0], bh[1]);    // small terms first
                  mma_f16_k16(cacc[n], ah[ks], bl[0], bl[1]);
                }
                mma_f16_k16(cacc[n], ah[ks], bh[0], bh[1]);
              }
            }
            if (P16 && pl.stage_ok) {
              // dP leaves through the TMA engine: the warp parks its 16-source x 32-channel tile (hi plane, then lo plane:
              // one box of rows x 64 B each, 64B swizzle, conflict-free 4-byte stores) in its 2 KB piece of the idle dz'
              // tile and one lane stores both planes with one instruction.  Pad columns [C, Cp) are exact zeros (the dout
              // box zero-fills past C), columns past Cp and rows past N are outside the box.  (The per-row st.global stream
              // this replaces bounded the phase: 38 K cycles per graph with the MMA loop at a third of that.)
              const int rows_m = m == 0 ? min(16, N) : N - 16;
              const uint32_t stg = a_D + (uint32_t)warp * 2048u;
              // A head whose first column sits 16 bytes into a 32-byte sector (odd heads when Cp % 16 == 8) would write every
              // 64-byte row piece over three sectors, two of them partially - and the L2 fills a partially written sector from
              // DRAM (measured: 0.8 GB of extra reads per launch).  Such a head stores its tiles shifted left by one 8-column
              // chunk: box k covers [32k - 8, 32k + 24) = the last chunk of tile k - 1 (kept in registers) and the first three
              // of tile k; columns past Cp are outside the tensor map's head and are not written.
              // (tile 0 goes out unshifted: a negative box coordinate faults on a store; its last chunk is then written twice,
              // with the same values)
              const bool shift = ((h * Cp) & 15) != 0 && cb > 0;
              uint32_t cur_h[2][4], cur_l[2][4];
#pragma unroll
              for (int hf = 0; hf < 2; ++hf)
#pragma unroll
                for (int n = 0; n < 4; ++n) {
                  const float w0 = cacc[n][2 * hf] * k_dp, w1 = cacc[n][2 * hf + 1] * k_dp;
                  const __half2 hh = __floats2half2_rn(w0, w1);
                  const float2 back = __half22float2(hh);
                  const __half2 ll = __floats2half2_rn(w0 - back.x, w1 - back.y);
                  cur_h[hf][n] = *reinterpret_cast<const uint32_t*>(&hh);
                  cur_l[hf][n] = *reinterpret_cast<const uint32_t*>(&ll);
                }
              if (lane == 0) bulk_wait_read();                      // the previous tile's store has read the staging
              __syncwarp();
#pragma unroll
              for (int hf = 0; hf < 2; ++hf) {
                const int rr = g + 8 * hf;                          // row inside the tile; tall-tile row of the lo plane: rows_m + rr
                if (rr < rows_m) {
#pragma unroll
                  for (int q = 0; q < 4; ++q) {                     // staging chunk q <- tile chunk q (or q - 1, chunk 0 <- the carried one)
                    const uint32_t vh = !shift ? cur_h[hf][q] : (q == 0 ? carry_h[hf] : cur_h[hf][q - 1]);
                    const uint32_t vl = !shift ? cur_l[hf][q] : (q == 0 ? carry_l[hf] : cur_l[hf][q - 1]);
                    stsa_b32(stg + sw64(rr, q) + 4u * t, vh);
                    if (!SINGLE) stsa_b32(stg + sw64(rows_m + rr, q) + 4u * t, vl);
                  }
                }
                carry_h[hf] = cur_h[hf][3];
                carry_l[hf] = cur_l[hf][3];
              }
              fence_proxy_async();
              __syncwarp();
              if (lane == 0) tma_store_4d(m == 0 ? &tmD0 : &tmD1, stg, cb * 32 - (shift ? 8 : 0), b * N + 16 * m, h, 0);
              if (((h * Cp) & 15) != 0 && cb == n_cb - 1 && n_cb > 1 && 32 * n_cb - 8 < Cp) {
                // the carried last chunk still holds columns the head owns: one more box, only its first chunk inside Cp
                if (lane == 0) bulk_wait_read();
                __syncwarp();
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                  const int rr = g + 8 * hf;
                  if (rr < rows_m) {
                    stsa_b32(stg + sw64(rr, 0) + 4u * t, carry_h[hf]);
                    if (!SINGLE) stsa_b32(stg + sw64(rows_m + rr, 0) + 4u * t, carry_l[hf]);
                  }
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) tma_store_4d(m == 0 ? &tmD0 : &tmD1, stg, n_cb * 32 - 8, b * N + 16 * m, h, 0);
              }
            } else if (args.dP_hi16 && vec4_out) {
              // fp16 pairs, coalesced: a quad exchange gives every lane 4 consecutive columns, so one 8-byte
              // store per lane writes 32 contiguous bytes per row (the fragment's native 4-byte pieces cost
              // one partial sector each and bounded this phase)
#pragma unroll
              for (int hf = 0; hf < 2; ++hf) {
                const int j = hf ? j1 : j0;
                uint32_t hi32[4], lo32[4];
#pragma unroll
                for (int n = 0; n < 4; ++n) {
                  const float w0 = cacc[n][2 * hf] * k_dp, w1 = cacc[n][2 * hf + 1] * k_dp;
                  const __half2 hh = __floats2half2_rn(w0, w1);
                  const float2 back = __half22float2(hh);
                  const __half2 ll = __floats2half2_rn(w0 - back.x, w1 - back.y);
                  hi32[n] = *reinterpret_cast<const uint32_t*>(&hh);
                  lo32[n] = *reinterpret_cast<const uint32_t*>(&ll);
                }
#pragma unroll
                for (int pr = 0; pr < 2; ++pr) {           // n-tile pairs (0,1) and (2,3): 16 columns each
                  const int src = (lane & ~3) + 2 * (t & 1);
                  const uint32_t ha0 = __shfl_sync(0xffffffffu, hi32[2 * pr], src), ha1 = __shfl_sync(0xffffffffu, hi32[2 * pr + 1], src);
                  const uint32_t hb0 = __shfl_sync(0xffffffffu, hi32[2 * pr], src + 1), hb1 = __shfl_sync(0xffffffffu, hi32[2 * pr + 1], src + 1);
                  const uint32_t la0 = __shfl_sync(0xffffffffu, lo32[2 * pr], src), la1 = __shfl_sync(0xffffffffu, lo32[2 * pr + 1], src);
                  const uint32_t lb0 = __shfl_sync(0xffffffffu, lo32[2 * pr], src + 1), lb1 = __shfl_sync(0xffffffffu, lo32[2 * pr + 1], src + 1);
                  const bool up = (t >> 1) != 0;           // lanes 2,3 of the quad take the second n-tile of the pair
                  const int c = cb * 32 + 16 * pr + 8 * (t >> 1) + 4 * (t & 1);
                  if (j < N && c < Cp) {                   // columns [C, Cp): the padded head pitch's zero columns
                    const size_t off = ((size_t)b * N + j) * args.ldp16 + (size_t)h * Cp + c;
                    const bool pad = c >= C;
                    *reinterpret_cast<uint2*>(args.dP_hi16 + off) = pad ? make_uint2(0u, 0u) : make_uint2(up ? ha1 : ha0, up ? hb1 : hb0);
                    if (!(P16 && SINGLE))
                      *reinterpret_cast<uint2*>(args.dP_lo16 + off) = pad ? make_uint2(0u, 0u) : make_uint2(up ? la1 : la0, up ? lb1 : lb0);
                  }
                }
              }
            } else {
#pragma unroll
              for (int n = 0; n < 4; ++n)
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                  const int j = hf ? j1 : j0;
                  const int c = cb * 32 + 8 * n + 2 * t;
                  if (j < N && c < Cp) {
                    // k_dp carries dp_scale (1 in fp32 mode); columns [C, Cp) are the padded head pitch's zero columns
                    const float v0 = c < C ? cacc[n][2 * hf] * k_dp : 0.f, v1 = c + 1 < C ? cacc[n][2 * hf + 1] * k_dp : 0.f;
                    const bool has1 = c + 1 < Cp;
                    if (args.dP_hi16) {
                      const size_t off = ((size_t)b * N + j) * args.ldp16 + (size_t)h * Cp + c;
                      const float w0 = v0, w1 = v1;
                      const __half h0_ = __float2half_rn(w0), h1_ = __float2half_rn(w1);
                      const __half l0_ = __float2half_rn(w0 - __half2float(h0_)), l1_ = __float2half_rn(w1 - __half2float(h1_));
                      if (P16) {           // h * Cp + c is even and c + 1 < Cp: aligned pairs
                        *reinterpret_cast<__half2*>(args.dP_hi16 + off) = __halves2half2(h0_, h1_);
                        if (!SINGLE) *reinterpret_cast<__half2*>(args.dP_lo16 + off) = __halves2half2(l0_, l1_);
                      } else if (p.vec2_ok) {
                        *reinterpret_cast<__half2*>(args.dP_hi16 + off) = __halves2half2(h0_, h1_);
                        *reinterpret_cast<__half2*>(args.dP_lo16 + off) = __halves2half2(l0_, l1_);
                      } else {
                        args.dP_hi16[off] = h0_; args.dP_lo16[off] = l0_;
                        if (has1) { args.dP_hi16[off + 1] = h1_; args.dP_lo16[off + 1] = l1_; }
                      }
                    } else {
                      const size_t off = ((size_t)b * N + j) * p.ldp + (size_t)h * C + c;
                      if (p.vec2_ok) {
                        *reinterpret_cast<float2*>(args.dP_aug + off) = make_float2(v0, v1);
                      } else {
                        args.dP_aug[off] = v0;
                        if (has1) args.dP_aug[off + 1] = v1;
                      }
                    }
                  }
                }
            }
          }
        }
        release_slot();
      }
    }
    if (P16 && pl.stage_ok && lane == 0) bulk_wait_read();        // the engine has read this warp's last dP staging tile
    bar_sync<1, kCT>();                                   // every warp is done with alpha and with the dz' tile
    if (!use_terms) {                                     // (a kept tile is copied over the whole of it)
      for (int idx = tid; idx < tile_floats; idx += kCT) tile[idx] = 0.f;      // next graph's logits accumulate into zeros
      bar_sync<1, kCT>();
    }
    lap(4);
  }
  if (P16 && pl.stage_ok && lane == 0) bulk_wait();                                                // this lane's dP stores have landed
#ifdef SPOTV2_BRINGUP
  if (tid == 0)
    for (int k = 0; k < 6; ++k) atomicAdd(&g_bwd2_counters[k], (unsigned long long)ph[k]);
#endif
  if (args.dsd_amax) {
    for (int o = 16; o > 0; o >>= 1) dsd_max = fmaxf(dsd_max, __shfl_xor_sync(0xffffffffu, dsd_max, o));
    if (lane == 0 && dsd_max > 0.f) atomicMax(args.dsd_amax, __float_as_uint(dsd_max));
  }

  // ---- per-CTA partials: dv_part[(cta * dv_rg + rg)][h][f], dbias_part[cta][col] ----
  if (Fe > 0) {
#pragma unroll
    for (int uu = 0; uu < kMaxDvUnits; ++uu) {
      if (dv_mt[uu] >= 0) {
        const int mt = dv_mt[uu], rg = dv_rb[uu] / pl.dv_rpu;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int f = mt * 16 + g + ((q & 2) ? 8 : 0), h = 2 * t + (q & 1);
          if (f < Fe && h < H)
            args.dv_part[((size_t)blockIdx.x * pl.dv_rg + rg) * H * Fe + (size_t)h * Fe + f] = dv_run[uu][q];
        }
      }
    }
  }
  if (!P16)
    for (int idx = tid; idx < p.ldo; idx += kCT) args.dbias_part[(size_t)blockIdx.x * p.ldo + idx] = dbias_s[idx];
}
