// Body of the phase-serial attention backward (attn_bwd.cu), included there twice: SPOTV2_KERNEL_NAME names the kernel and
// SPOTV2_GA = 1 makes the variant that takes d_alpha [B, H, N(j), N(i)], the gradient through the coefficients the forward
// returned (after dropout), which joins dalpha before the dropout factor (B2b).  Two kernels under their own names keep the
// machine code of the one without it exactly what it was.  No include guard: meant to be included more than once.
template <int NPAIRS>
__global__ void __launch_bounds__(kAttnThreads, 2)
SPOTV2_KERNEL_NAME(const AttnBwdArgs args, const BwdSmem sm
#if SPOTV2_GA
            , const float* __restrict__ d_alpha
#endif
) {
  constexpr bool GA = SPOTV2_GA != 0;
#if !SPOTV2_GA
  const float* const d_alpha = nullptr;
#endif
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const AttnParams& p = args.p;
  const int tid = threadIdx.x;
  const int N = p.N, H = p.H, C = p.C, NS = sm.a.NS, Fe = p.Fe;
  const int HC = H * C;
  const float inv_nm1 = 1.f / (float)(N > 1 ? N - 1 : 1);

  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + sm.a.off_bar);
  int32_t* table_s = reinterpret_cast<int32_t*>(smem_raw + sm.a.off_table);
  float4* vfrag = reinterpret_cast<float4*>(smem_raw + sm.a.off_vfrag);
  float* sd = reinterpret_cast<float*>(smem_raw + sm.a.off_sd);
  float* tile = reinterpret_cast<float*>(smem_raw + sm.a.off_tile);     // alpha[h][j][i]
  float* D = reinterpret_cast<float*>(smem_raw + sm.off_D);             // dalpha -> dz -> dz'
  uint32_t* pos_mask = reinterpret_cast<uint32_t*>(smem_raw + sm.off_mask);
  uint32_t* keep_mask = pos_mask + ((H * N + 3) / 4) * 4;
  float* dbias_s = reinterpret_cast<float*>(smem_raw + sm.off_dbias);
  unsigned char* uni = smem_raw + sm.off_union;
  float* const stage_base = reinterpret_cast<float*>(uni);             // [buf][P rows | G rows]
  // keep the address space visible to the compiler even where these pointers travel through lambdas /
  // structs (generic LD/ST to shared memory is several times slower than LDS/STS - measured)
  __builtin_assume(__isShared(table_s)); __builtin_assume(__isShared(vfrag)); __builtin_assume(__isShared(sd));
  __builtin_assume(__isShared(tile)); __builtin_assume(__isShared(D)); __builtin_assume(__isShared(pos_mask));
  __builtin_assume(__isShared(dbias_s)); __builtin_assume(__isShared(stage_base)); __builtin_assume(__isShared(uni));
  const int stage_floats = (int)((sm.stage_P_bytes + sm.stage_G_bytes) / 4);
  const int stage_g_off = (int)(sm.stage_P_bytes / 4);

  EdgeRing ring;
  ring.stage[0] = reinterpret_cast<float*>(uni);
  ring.stage[1] = reinterpret_cast<float*>(uni + sm.a.ring_stage_bytes);
  ring.full = bars;
  ring.uses[0] = ring.uses[1] = 0;
  ring.chunk_rows = sm.a.chunk_rows;
  ring.nchunks = Fe > 0 ? (p.R + sm.a.chunk_rows - 1) / sm.a.chunk_rows : 0;
  ring.p = &p;

  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    fence_mbar_init();
  }
  for (int r = tid; r < p.R; r += kAttnThreads) table_s[r] = Fe > 0 ? p.table[r] : -1;
  if (Fe > 0) build_vfrag(vfrag, p.v, H, Fe, sm.a.KS, sm.a.NT, tid, kAttnThreads);
  for (int idx = tid; idx < H * N * NS; idx += kAttnThreads) { tile[idx] = 0.f; D[idx] = 0.f; }
  for (int idx = tid; idx < p.ldo; idx += kAttnThreads) dbias_s[idx] = 0.f;
  __syncthreads();

  int b = blockIdx.x;
  // the forward kept the edge terms (p.edge_terms): B1 copies them instead of streaming the edge rows a first time
  const bool use_terms = p.edge_terms != nullptr && ring.nchunks > 0;
  if (p.bulk_ok && tid == 0 && b < p.B && ring.nchunks > 0 && !use_terms) ring.prefetch_first(b);

  const float g_scale = p.concat ? 1.f : 1.f / (float)H;
  float dp_scale = 1.f;
  if (args.dP_hi16) {
    dp_scale = dp_scale_from_amax(__uint_as_float(*reinterpret_cast<const unsigned*>(args.dout_blk)) * args.bound);
    if (blockIdx.x == 0 && tid == 0) { args.dp_blk[2] = 1.f / dp_scale; args.dp_blk[4] = dp_scale; }
  }
  const bool vec4 = (C % 4 == 0) && (p.ldo % 4 == 0);
  const int NIG = sm.NP5 / kTI;                       // tile groups along targets and sources
  const int n_tiles = H * NIG * NIG;
  const int nchan_chunks = (C + kCK - 1) / kCK;
  const int CP = (C + 1) / 2;
  const int n_items = p.concat ? H * CP : CP;

  // dv^T[f][h] = sum_e T[e][f] * dz'[e][h] on mma.sync m16n8k8 (3xTF32): warp w owns the 16-feature
  // m-tiles w, w+8, ...; heads are the n dimension.  Each staged chunk is accumulated in a fresh fragment
  // and folded into dv_run with round-to-nearest adds (tensor-core accumulation truncates).
  constexpr int kMT = kMaxFe / 16 / (kAttnThreads / 32);     // m-tiles per warp (4)
  const int warp_id = tid >> 5, lane_id = tid & 31;
  const int n_mtiles = (Fe + 15) / 16;
  float dv_run[kMT][4];
#pragma unroll
  for (int m = 0; m < kMT; ++m)
#pragma unroll
    for (int q = 0; q < 4; ++q) dv_run[m][q] = 0.f;

  long long ph[6] = {0, 0, 0, 0, 0, 0};
  long long t_ph = clock64();
  auto lap = [&](int k) { const long long now = clock64(); ph[k] += now - t_ph; t_ph = now; };
  for (; b < p.B; b += gridDim.x) {
    // ---- B1: recompute alpha --------------------------------------------------------------
    for (int idx = tid; idx < N * 2 * H; idx += kAttnThreads) {
      const int j = idx / (2 * H), k = idx - j * 2 * H;
      sd[idx] = p.P_aug[((size_t)b * N + j) * p.ldp + HC + k];
    }
    if (use_terms) {
      const float* src = p.edge_terms + (size_t)b * H * N * kEdgeTermNS;
      for (int idx = tid; idx < H * N * N; idx += kAttnThreads) {
        const int hj = idx / N, i = idx - hj * N;
        tile[hj * NS + i] = src[hj * kEdgeTermNS + i];
      }
      __syncthreads();
    } else if (ring.nchunks > 0) {
      edge_logit_phase(ring, p, sm.a, tile, table_s, vfrag, b, tid);
    } else {
      for (int idx = tid; idx < H * N * NS; idx += kAttnThreads) tile[idx] = 0.f;
      __syncthreads();
    }
    lap(0);
    softmax_phase(p, sm.a, tile, sd, 1.f, nullptr, pos_mask, tid);
    lap(1);
    // (no barrier needed before B2's loads: they write the union region, idle since B1's last barrier;
    //  D is written only after the chunk loop's barriers)

    // ---- B2: dalpha = dO . P^T -------------------------------------------------------------
    // Per-thread staging descriptors (the float4 a thread copies has the same row and column quarter in
    // every channel chunk): source pointer at channel 0 (null = zero-fill row) and shared-memory offset.
    constexpr int kFastIt = 4;
    const int stage_items = (H * sm.NP5 + (p.concat ? H : 1) * sm.NP5) * (kCK / 4);
    const bool stage_fast = vec4 && stage_items <= kFastIt * kAttnThreads;
    const float* st_src[kFastIt];
    int st_dst[kFastIt];
    if (stage_fast) {
      const int rowsP = H * sm.NP5;
#pragma unroll
      for (int itn = 0; itn < kFastIt; ++itn) {
        const int idx = tid + itn * kAttnThreads;
        const int row = idx >> 2, q = idx & 3;
        st_src[itn] = nullptr;
        st_dst[itn] = -1;
        if (idx < stage_items) {
          if (row < rowsP) {
            const int h = row / sm.NP5, j = row - h * sm.NP5;
            st_dst[itn] = row * kCKP + 4 * q;
            if (j < N) st_src[itn] = p.P_aug + ((size_t)b * N + j) * p.ldp + (size_t)h * C + 4 * q;
          } else {
            const int r2 = row - rowsP;
            const int h = r2 / sm.NP5, i = r2 - h * sm.NP5;
            st_dst[itn] = stage_g_off + r2 * kCKP + 4 * q;
            if (i < N) st_src[itn] = args.dout + ((size_t)b * N + i) * p.ldo + (size_t)h * C + 4 * q;
          }
        }
      }
    }
    auto stage = [&](int bufsel, int c_base) {
      float* base = stage_base + bufsel * stage_floats;
      if (stage_fast) {
        const bool col_ok = c_base + 4 * (tid & 3) < C;
#pragma unroll
        for (int itn = 0; itn < kFastIt; ++itn) {
          if (st_dst[itn] >= 0) {
            const bool ok = col_ok && st_src[itn] != nullptr;
            cp_async16(base + st_dst[itn], ok ? st_src[itn] + c_base : p.P_aug, ok);
          }
        }
      } else {
        stage_chunk(args, sm, base, base + stage_g_off, b, c_base, vec4, tid);
      }
    };
    for (int t0 = 0; t0 < n_tiles; t0 += kAttnThreads) {
      const int t = t0 + tid;
      const bool active = t < n_tiles;
      const int ig = t % NIG, cg = (t / NIG) % NIG, h = active ? t / (NIG * NIG) : 0;
      float2 acc[kTI][kTJ];
#pragma unroll
      for (int ii = 0; ii < kTI; ++ii)
#pragma unroll
        for (int jj = 0; jj < kTJ; ++jj) acc[ii][jj] = make_float2(0.f, 0.f);
      stage(0, 0);
      cp_async_commit();
      for (int ch = 0; ch < nchan_chunks; ++ch) {
        const int buf = ch & 1;
        if (ch + 1 < nchan_chunks) stage(buf ^ 1, (ch + 1) * kCK);
        cp_async_commit();
        cp_async_wait<1>();
        __syncthreads();
        if (active) {
          const float* Gb = stage_base + buf * stage_floats + stage_g_off + ((p.concat ? h * sm.NP5 : 0) + ig * kTI) * kCKP;
          const float* Pb = stage_base + buf * stage_floats + (h * sm.NP5 + cg * kTJ) * kCKP;
#pragma unroll
          for (int s4 = 0; s4 < kCK / 4; ++s4) {
            float4 pv[kTJ];
#pragma unroll
            for (int jj = 0; jj < kTJ; ++jj) pv[jj] = *reinterpret_cast<const float4*>(Pb + jj * kCKP + 4 * s4);
#pragma unroll
            for (int ii = 0; ii < kTI; ++ii) {
              const float4 g4 = *reinterpret_cast<const float4*>(Gb + ii * kCKP + 4 * s4);
              const float2 g0 = make_float2(g4.x, g4.y), g1 = make_float2(g4.z, g4.w);
#pragma unroll
              for (int jj = 0; jj < kTJ; ++jj) {
                acc[ii][jj] = ffma2(g0, make_float2(pv[jj].x, pv[jj].y), acc[ii][jj]);
                acc[ii][jj] = ffma2(g1, make_float2(pv[jj].z, pv[jj].w), acc[ii][jj]);
              }
            }
          }
        }
        __syncthreads();
      }
      if (active) {
#pragma unroll
        for (int ii = 0; ii < kTI; ++ii) {
          const int i = ig * kTI + ii;
#pragma unroll
          for (int jj = 0; jj < kTJ; ++jj) {
            const int j = cg * kTJ + jj;
            if (i < N && j < N) D[(h * N + j) * NS + i] = (acc[ii][jj].x + acc[ii][jj].y) * g_scale;
          }
        }
      }
    }
    __syncthreads();
    lap(2);
    // staging is idle from here: start the second pass over the edge rows under B2b/B3
    if (p.bulk_ok && tid == 0 && ring.nchunks > 0) ring.prefetch_first(b);

    // ---- B2b: softmax / LeakyReLU backward ---------------------------------------------------
    // With attention dropout the forward used alpha * m (m = keep / (1 - p)): dalpha = m * d(alpha m), the softmax
    // backward runs on the un-dropped alpha, and B3 below needs alpha * m (applied in the third loop).
    const bool drop = p.drop.p > 0.f;
    for (int idx = tid; idx < H * N; idx += kAttnThreads) {
      const int h = idx / N, i = idx - h * N;
      const float* acol = tile + (size_t)h * N * NS + i;
      float* dcol = D + (size_t)h * N * NS + i;
      uint32_t keep = 0xffffffffu;
      if (GA)
        for (int j = 0; j < N; ++j) dcol[j * NS] += __ldg(d_alpha + (((size_t)b * H + h) * N + j) * N + i);
      if (drop) {
        keep = dropout_keep_bits(p.drop, (((unsigned long long)b * H + h) * N + i) * N, N);
        keep_mask[idx] = keep;
        for (int j = 0; j < N; ++j) dcol[j * NS] = ((keep >> j) & 1u) ? dcol[j * NS] * p.drop.scale : 0.f;
      }
      float dot = 0.f;
      for (int j = 0; j < N; ++j) dot = fmaf(acol[j * NS], dcol[j * NS], dot);
      const uint32_t mask = pos_mask[idx];
      float dd = 0.f;
      for (int j = 0; j < N; ++j) {
        const float dl = acol[j * NS] * (dcol[j * NS] - dot);
        const float dz = ((mask >> j) & 1u) ? dl : dl * p.slope;
        dd += dz;
        dcol[j * NS] = dz;
      }
      if (args.dsd) args.dsd[((size_t)b * N + i) * 2 * H + H + h] = dd;
      else args.dP_aug[((size_t)b * N + i) * p.ldp + HC + H + h] = dd;
    }
    __syncthreads();
    for (int idx = tid; idx < H * N; idx += kAttnThreads) {     // ds_j = sum_i dz_ij
      const int h = idx / N, j = idx - h * N;
      const float* drow = D + (size_t)(h * N + j) * NS;
      float ds = 0.f;
      for (int k = 0; k < N; ++k) {
        int i = j + k;                                          // rotated start: conflict-free banks
        if (i >= N) i -= N;
        ds += drow[i];
      }
      if (args.dsd) args.dsd[((size_t)b * N + j) * 2 * H + h] = ds;
      else args.dP_aug[((size_t)b * N + j) * p.ldp + HC + h] = ds;
    }
    __syncthreads();
    for (int idx = tid; idx < H * N; idx += kAttnThreads) {     // dz' : gradient through the mean fill
      const int h = idx / N, i = idx - h * N;
      float* dcol = D + (size_t)h * N * NS + i;
      const float share = dcol[i * NS] * inv_nm1;
      for (int j = 0; j < N; ++j) dcol[j * NS] = (j == i) ? 0.f : dcol[j * NS] + share;
      if (drop) {
        float* acol = tile + (size_t)h * N * NS + i;
        const uint32_t keep = keep_mask[idx];
        for (int j = 0; j < N; ++j) acol[j * NS] = ((keep >> j) & 1u) ? acol[j * NS] * p.drop.scale : 0.f;
      }
    }
    // (D is next read in B4, after B3's trailing barrier)

    lap(3);
    // ---- B3: dP = alpha^T dO ------------------------------------------------------------------
    for (int item = tid; item < n_items; item += kAttnThreads) {
      const int h0 = p.concat ? item / CP : 0;
      const int cp = p.concat ? item - h0 * CP : item;
      const int c0 = 2 * cp;
      const bool has1 = c0 + 1 < C;
      const int gcol = h0 * C + c0;                       // column of dout this item reads
      float2 G[NPAIRS][2];                                // (dO[2ip][c], dO[2ip+1][c]) for c0, c0+1
      float bsum0 = 0.f, bsum1 = 0.f;
#pragma unroll
      for (int ip = 0; ip < NPAIRS; ++ip) {
        float v[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int i = 2 * ip + half;
          if (i < N) {
            const float* src = args.dout + ((size_t)b * N + i) * p.ldo + gcol;
            if (p.vec2_ok) {
              const float2 t2 = *reinterpret_cast<const float2*>(src);
              v[half][0] = t2.x; v[half][1] = t2.y;
            } else {
              v[half][0] = __ldg(src);
              if (has1) v[half][1] = __ldg(src + 1);
            }
          }
        }
        bsum0 += v[0][0] + v[1][0];
        bsum1 += v[0][1] + v[1][1];
        G[ip][0] = make_float2(v[0][0] * g_scale, v[1][0] * g_scale);
        G[ip][1] = make_float2(v[0][1] * g_scale, v[1][1] * g_scale);
      }
      dbias_s[gcol] += bsum0;                              // each column has exactly one owner thread
      if (has1) dbias_s[gcol + 1] += bsum1;

      const int h_begin = p.concat ? h0 : 0, h_end = p.concat ? h0 + 1 : H;
      for (int h = h_begin; h < h_end; ++h) {
        for (int j = 0; j < N; ++j) {
          const float* ar = tile + (size_t)(h * N + j) * NS;
          float2 s0 = make_float2(0.f, 0.f), s1 = make_float2(0.f, 0.f);
#pragma unroll
          for (int q = 0; q < NPAIRS / 2; ++q) {
            const float4 a4 = *reinterpret_cast<const float4*>(ar + 4 * q);
            const float2 a0 = make_float2(a4.x, a4.y), a1 = make_float2(a4.z, a4.w);
            s0 = ffma2(a0, G[2 * q][0], s0);
            s1 = ffma2(a0, G[2 * q][1], s1);
            s0 = ffma2(a1, G[2 * q + 1][0], s0);
            s1 = ffma2(a1, G[2 * q + 1][1], s1);
          }
          if (NPAIRS & 1) {
            const float2 a0 = *reinterpret_cast<const float2*>(ar + 2 * (NPAIRS - 1));
            s0 = ffma2(a0, G[NPAIRS - 1][0], s0);
            s1 = ffma2(a0, G[NPAIRS - 1][1], s1);
          }
          const float v0 = s0.x + s0.y, v1 = s1.x + s1.y;
          if (args.dP_hi16) {
            const size_t off = ((size_t)b * N + j) * args.ldp16 + (size_t)h * C + c0;
            const float w0 = v0 * dp_scale, w1 = v1 * dp_scale;
            const __half h0_ = __float2half_rn(w0), h1_ = __float2half_rn(w1);
            const __half l0_ = __float2half_rn(w0 - __half2float(h0_)), l1_ = __float2half_rn(w1 - __half2float(h1_));
            if (p.vec2_ok) {
              *reinterpret_cast<__half2*>(args.dP_hi16 + off) = __halves2half2(h0_, h1_);
              *reinterpret_cast<__half2*>(args.dP_lo16 + off) = __halves2half2(l0_, l1_);
            } else {
              args.dP_hi16[off] = h0_; args.dP_lo16[off] = l0_;
              if (has1) { args.dP_hi16[off + 1] = h1_; args.dP_lo16[off + 1] = l1_; }
            }
          } else {
            const size_t off = ((size_t)b * N + j) * p.ldp + (size_t)h * C + c0;
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
    __syncthreads();
    if (p.dterms_out) {
      // d(edge terms) out (the caller's d_edge_terms): dz' in the forward's edge-term layout [H][N][kEdgeTermNS]
      float* dst = p.dterms_out + (size_t)b * H * N * kEdgeTermNS;
      for (int idx = tid; idx < H * N * N; idx += kAttnThreads) {
        const int hj = idx / N, i = idx - hj * N;
        dst[hj * kEdgeTermNS + i] = D[hj * NS + i];
      }
    }

    lap(4);
    // ---- B4: dv += dz'^T . edge rows -------------------------------------------------------------
    for (int c = 0; c < ring.nchunks; ++c) {
      const int s = c & 1;
      const int rows = ring.rows_in(c);
      if (p.bulk_ok) {
        mbar_wait(&ring.full[s], ring.uses[s] & 1);
        ring.uses[s]++;
      } else {
        const float* src = p.edge_rows + ((size_t)b * p.R + (size_t)c * ring.chunk_rows) * Fe;
        for (int idx = tid; idx < rows * Fe; idx += kAttnThreads) ring.stage[s][idx] = src[idx];
        __syncthreads();
      }
      {
        const float* Ts = ring.stage[s];
        const int row_base = c * ring.chunk_rows;
        const int g8 = lane_id >> 2, t4 = lane_id & 3;
        // mma.sync latency on sm_100 is ~300 cycles: give every k-step slot and product its own
        // accumulator (kDvSlots x 3 independent chains per m-tile) and sum them after the chunk.
        constexpr int kDvSlots = 3;
#pragma unroll
        for (int m = 0; m < kMT; ++m) {
          const int mt = warp_id + m * (kAttnThreads / 32);
          if (mt >= n_mtiles) continue;                    // warp-uniform
          const int f0 = mt * 16 + g8, f1 = f0 + 8;
          float acc[kDvSlots][3][4];
#pragma unroll
          for (int sl = 0; sl < kDvSlots; ++sl)
#pragma unroll
            for (int pr = 0; pr < 3; ++pr)
#pragma unroll
              for (int q = 0; q < 4; ++q) acc[sl][pr][q] = 0.f;
          for (int rb = 0; rb < rows; rb += 8 * kDvSlots) {
#pragma unroll
            for (int sl = 0; sl < kDvSlots; ++sl) {
              const int r0 = rb + 8 * sl;
              if (r0 < rows) {
                // B fragment (k = edge row, n = head): b0 = dz'[r0+t][g], b1 = dz'[r0+t+4][g]
                float bv[2];
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                  const int r = r0 + t4 + 4 * half;
                  float val = 0.f;
                  if (r < rows && g8 < H) {
                    const int code = table_s[row_base + r];
                    if (code >= 0) val = D[(g8 * N + (code & 0xffff)) * NS + (code >> 16)];
                  }
                  bv[half] = val;
                }
                uint32_t bh[2], bl[2];
                split_tf32_trunc(bv[0], bh[0], bl[0]);
                split_tf32_trunc(bv[1], bh[1], bl[1]);
                const bool k0_ok = r0 + t4 < rows, k1_ok = r0 + t4 + 4 < rows;
                const float* t0p = Ts + (size_t)(r0 + t4) * Fe;
                const float* t1p = t0p + (size_t)4 * Fe;
                float a[4];
                a[0] = (k0_ok && f0 < Fe) ? lds_f32(t0p + f0) : 0.f;     // (m = g,   k = t)
                a[1] = (k0_ok && f1 < Fe) ? lds_f32(t0p + f1) : 0.f;     // (m = g+8, k = t)
                a[2] = (k1_ok && f0 < Fe) ? lds_f32(t1p + f0) : 0.f;     // (m = g,   k = t+4)
                a[3] = (k1_ok && f1 < Fe) ? lds_f32(t1p + f1) : 0.f;     // (m = g+8, k = t+4)
                uint32_t ah[4], al[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) split_tf32_trunc(a[q], ah[q], al[q]);
                mma_tf32_16x8x8(acc[sl][0], al, bh);
                mma_tf32_16x8x8(acc[sl][1], ah, bl);
                mma_tf32_16x8x8(acc[sl][2], ah, bh);
              }
            }
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            float corr = 0.f, mainp = 0.f;
#pragma unroll
            for (int sl = 0; sl < kDvSlots; ++sl) {
              corr += acc[sl][0][q] + acc[sl][1][q];
              mainp += acc[sl][2][q];
            }
            dv_run[m][q] += corr + mainp;
          }
        }
      }
      __syncthreads();
      if (p.bulk_ok && tid == 0 && c + 2 < ring.nchunks) ring.issue(b, c + 2);
    }
    if (p.bulk_ok && tid == 0 && b + (int)gridDim.x < p.B && ring.nchunks > 0 && !use_terms)
      ring.prefetch_first(b + gridDim.x);
    lap(5);
  }
  if (tid == 0)
    for (int k = 0; k < 6; ++k) atomicAdd(&g_bwd_counters[k], (unsigned long long)ph[k]);

  // ---- per-CTA partials ---------------------------------------------------------------------------
  // A CTA that issued a prefetch always consumes it (the prefetch is only issued for graphs it owns),
  // so no bulk copy is in flight here and the union region can be reused.
  __syncthreads();
  if (Fe > 0) {
    // C fragment of dv^T: c0 = (f = g, h = 2t), c1 = (g, 2t+1), c2 = (g+8, 2t), c3 = (g+8, 2t+1)
    const int g8 = lane_id >> 2, t4 = lane_id & 3;
#pragma unroll
    for (int m = 0; m < kMT; ++m) {
      const int mt = warp_id + m * (kAttnThreads / 32);
      if (mt < n_mtiles) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int f = mt * 16 + g8 + ((q & 2) ? 8 : 0), h = 2 * t4 + (q & 1);
          if (f < Fe && h < H) args.dv_part[(size_t)blockIdx.x * H * Fe + (size_t)h * Fe + f] = dv_run[m][q];
        }
      }
    }
  }
  for (int idx = tid; idx < p.ldo; idx += kAttnThreads)
    args.dbias_part[(size_t)blockIdx.x * p.ldo + idx] = dbias_s[idx];
}
