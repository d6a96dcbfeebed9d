// Fused GAT attention backward with the attention coefficients RECOMPUTED from the inputs
// (nothing but P_aug is kept from the forward).  Closed form of SURVEY.md Appendix A.3 in the
// augmented layout: dP_aug = [dP | ds | dd].  Replaces the autograd graph PyG records for
// edge_update / softmax / propagate ([PyG] nn/conv/gat_conv.py; /root/reference/5_train_SpotV2Net.py:157).
//
// Per graph (one CTA iteration, N <= 32):
//   B1  recompute: edge rows -> g (3xTF32 mma.sync) -> alpha tile, z>0 masks            [ring]
//   B2  dalpha[h][i][j] = <dO_i,h , P_j,h>: 5x5 register tiles, FFMA2 paired over channels,
//       operands staged 16 channels at a time with cp.async double buffering            [staging]
//   B2b thread (h,i): softmax + LeakyReLU backward -> dz ; dd_i ; then ds_j ; then the
//       self-loop mean-fill redistribution dz'
//   B3  dP[j,h,c] = sum_i alpha_h[i,j] dO_i,h[c]: thread owns a channel pair, dO in registers
//   B4  dv[h,:] += sum_e dz'[e,h] * edge_attr[e,:]: second pass over the edge rows         [ring]
// The ring and the B2 staging alias the same shared memory.  dv and dbias are accumulated per
// CTA and reduced in a fixed order by a second kernel (deterministic).
#include <algorithm>

#include "attn_bwd.cuh"

namespace spotv2 {

constexpr int kCK = 16;        // channels per B2 staging chunk
constexpr int kCKP = 20;       // padded row stride (floats): 80 B, conflict-free for the 5x5 tiles
constexpr int kTI = 5;         // register tile: targets
constexpr int kTJ = 5;         // register tile: sources

// phase-time diagnostics (thread 0 of every CTA; see spotv2_diag_counters, entries 16..31)
__device__ unsigned long long g_bwd_counters[kNumCounters];

struct BwdSmem {
  AttnSmem a;
  int NP5;                  // rows per head in the staging buffers (N rounded up to kTI)
  size_t off_D, off_mask, off_dbias, off_union, union_bytes, stage_P_bytes, stage_G_bytes, total;
};

inline BwdSmem bwd_smem_plan(int N, int Fe, int H, int C, int R, int npairs, int concat, int chunk_rows) {
  BwdSmem s;
  s.a = attn_smem_plan(N, Fe, H, R, npairs, chunk_rows);
  s.NP5 = (N + kTI - 1) / kTI * kTI;
  const int ldo = concat ? H * C : C;
  size_t o = s.a.base_total;
  s.off_D = o;     o += round_up((size_t)H * N * s.a.NS * 4, 16);
  s.off_mask = o;  o += 2 * round_up((size_t)H * N * 4, 16);      // z > 0 bits | dropout keep bits
  s.off_dbias = o; o += round_up((size_t)ldo * 4, 16);
  s.off_union = round_up(o, 128);
  s.stage_P_bytes = (size_t)H * s.NP5 * kCKP * 4;
  s.stage_G_bytes = (size_t)(concat ? H : 1) * s.NP5 * kCKP * 4;
  const size_t staging = 2 * (s.stage_P_bytes + s.stage_G_bytes);
  const size_t ring = 2 * s.a.ring_stage_bytes;
  s.union_bytes = staging > ring ? staging : ring;
  s.total = s.off_union + s.union_bytes;
  return s;
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, bool valid) {
  const uint32_t n = valid ? 16u : 0u;   // src-size 0 => zero fill
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(n)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N_>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N_) : "memory"); }

// Stage channels [c_base, c_base + kCK) of this graph's P (all heads) and dO rows.
__device__ __forceinline__ void stage_chunk(const AttnBwdArgs& a, const BwdSmem& sm, float* Ps,
                                            float* Gs, int b, int c_base, bool vec4, int tid) {
  const AttnParams& p = a.p;
  const int N = p.N, H = p.H, C = p.C, NP5 = sm.NP5;
  const int g_heads = p.concat ? H : 1;
  const int rowsP = H * NP5, rowsG = g_heads * NP5;
  for (int idx = tid; idx < (rowsP + rowsG) * (kCK / 4); idx += kAttnThreads) {
    const int row = idx >> 2, q = idx & 3;
    const int c = c_base + 4 * q;
    float* dst;
    const float* src;
    bool row_ok;
    if (row < rowsP) {
      const int h = row / NP5, j = row - h * NP5;
      row_ok = j < N;
      dst = Ps + (size_t)row * kCKP + 4 * q;
      src = p.P_aug + ((size_t)b * N + (row_ok ? j : 0)) * p.ldp + (size_t)h * C + c;
    } else {
      const int r2 = row - rowsP;
      const int h = r2 / NP5, i = r2 - h * NP5;
      row_ok = i < N;
      dst = Gs + (size_t)r2 * kCKP + 4 * q;
      src = a.dout + ((size_t)b * N + (row_ok ? i : 0)) * p.ldo + (size_t)h * C + c;
    }
    if (vec4) {
      const bool ok = row_ok && c < C;        // C % 4 == 0 on this path: whole float4 in or out
      cp_async16(dst, ok ? src : p.P_aug, ok);
    } else {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row_ok) {
        if (c + 0 < C) v.x = __ldg(src + 0);
        if (c + 1 < C) v.y = __ldg(src + 1);
        if (c + 2 < C) v.z = __ldg(src + 2);
        if (c + 3 < C) v.w = __ldg(src + 3);
      }
      *reinterpret_cast<float4*>(dst) = v;
    }
  }
}

template <int NPAIRS>
__global__ void __launch_bounds__(kAttnThreads, 2)
gat_attn_bwd_kernel(const AttnBwdArgs args, const BwdSmem sm) {
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

// out[k] = sum_c part[c][k].  Block = 32 outputs x 8 partial groups (group g takes c = g, g + 8, ...: eight independent
// load streams per output, coalesced along k), combined through shared memory in a fixed order: deterministic.
__global__ void __launch_bounds__(256)
partial_reduce_kernel(const float* __restrict__ part, int nparts, int len, float* __restrict__ out) {
  __shared__ float red[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int k = blockIdx.x * 32 + tx;
  float s = 0.f;
  if (k < len)
    for (int c = ty; c < nparts; c += 8) s += part[(size_t)c * len + k];
  red[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && k < len) {
    float t = 0.f;
#pragma unroll
    for (int g = 0; g < 8; ++g) t += red[g][tx];
    out[k] = t;
  }
}

// two reductions behind one launch: blocks [0, blocks_a) serve the first, the rest the second.  32 x 32 threads: a column of
// partials is summed by 32 threads with two independent chains each (the loads of a chain were the kernel's whole latency:
// 444 partials over 8 threads took 30 us), then across the 32 in a fixed order - deterministic.
__global__ void __launch_bounds__(1024)
partial_reduce2_kernel(const float* __restrict__ pa, int na, int la, float* __restrict__ oa, int blocks_a,
                       const float* __restrict__ pb, int nb, int lb, float* __restrict__ ob) {
  __shared__ float red[32][33];
  const bool first = (int)blockIdx.x < blocks_a;
  const float* part = first ? pa : pb;
  const int nparts = first ? na : nb, len = first ? la : lb;
  float* out = first ? oa : ob;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int k = ((int)blockIdx.x - (first ? 0 : blocks_a)) * 32 + tx;
  float s0 = 0.f, s1 = 0.f;
  if (k < len) {
    int c = ty;
    for (; c + 32 < nparts; c += 64) {
      s0 += part[(size_t)c * len + k];
      s1 += part[(size_t)(c + 32) * len + k];
    }
    if (c < nparts) s0 += part[(size_t)c * len + k];
  }
  red[ty][tx] = s0 + s1;
  __syncthreads();
  if (ty == 0 && k < len) {
    float t = 0.f;
#pragma unroll
    for (int g = 0; g < 32; ++g) t += red[g][tx];
    out[k] = t;
  }
}

int reduce_partials2(const float* part_a, int nparts_a, int len_a, float* out_a, const float* part_b, int nparts_b, int len_b,
                     float* out_b, cudaStream_t st) {
  if (!out_a) len_a = 0;
  if (!out_b) len_b = 0;
  const int ba = (len_a + 31) / 32, bb = (len_b + 31) / 32;
  if (ba + bb == 0) return SPOTV2_OK;
  partial_reduce2_kernel<<<ba + bb, 1024, 0, st>>>(part_a, nparts_a, len_a, out_a, ba, part_b, nparts_b, len_b, out_b);
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

// ds | dd [rows, 2H] fp32 -> columns [HC, HC + 2H) of the dP operand pair; the group maximum was collected by the attention
// kernel itself (dp_blk[1], atomicMax of bit patterns), so this is the only pass: scale, split, publish the scale.
__global__ void __launch_bounds__(256)
split_dsd_kernel(const float* __restrict__ dsd, size_t total, int cols, __half* __restrict__ hi, __half* __restrict__ lo, int ld16,
                 float* __restrict__ dp_blk) {
  const float s = dp_scale_from_amax(__uint_as_float(reinterpret_cast<const unsigned*>(dp_blk)[1]));
  if (blockIdx.x == 0 && threadIdx.x == 0) { dp_blk[3] = 1.f / s; dp_blk[5] = s; }
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const size_t r = idx / cols;
    const int c = (int)(idx - r * cols);
    const float w = dsd[idx] * s;
    const __half h = __float2half_rn(w);
    hi[r * ld16 + c] = h;
    if (lo) lo[r * ld16 + c] = __float2half_rn(w - __half2float(h));
  }
}

int reduce_partials(const float* part, int nparts, int len, float* out, cudaStream_t st) {
  partial_reduce_kernel<<<(len + 31) / 32, 256, 0, st>>>(part, nparts, len, out);
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

// Workspace of the N <= 32 backward (byte offsets): per-CTA partials of dv and dbias (the most any kernel needs) | ds,dd fp32
// [B*N, 2H] | scale blocks max|dout|, ds|dd, max|P| (256 B) | p_format 1: dout's pair (two planes [B*N, ld16(ldo)]) | its unit
// scales [B * upg] | the prepass's dbias partials
struct BwdWorkspace { size_t dsd, blocks, dout_pair, plane, unit_scales, dbias_part, total; };

static BwdWorkspace bwd_workspace_of(const spotv2_gat_desc* d) {
  const size_t rows = (size_t)d->B * d->N, ldo = d->concat ? (size_t)d->H * d->C : (size_t)d->C;
  BwdWorkspace w{};
  const size_t serial_partials = round_up(2 * (size_t)sm_count() * ((size_t)d->H * d->Fe + ldo) * sizeof(float), 256);
  w.dsd = std::max({serial_partials, attn_bwd2_partials_bytes(d), attn_bwd3_partials_bytes(d)});
  w.blocks = w.dsd + round_up(rows * 2 * d->H * sizeof(float), 256);
  w.total = w.blocks + 256;
  if (d->p_format == 1) {
    const int upg = d->concat ? d->H : 1;
    w.plane = round_up(rows * ld16_of((int)ldo) * 2, 256);
    w.dout_pair = w.total;
    w.unit_scales = w.dout_pair + 2 * w.plane;
    w.dbias_part = w.unit_scales + round_up((size_t)d->B * upg * sizeof(float), 256);
    w.total = w.dbias_part + round_up((size_t)dout_pair_grid(d->B * upg, upg) * ldo * sizeof(float), 256);
  }
  return w;
}

size_t attn_bwd_ws_bytes(const spotv2_gat_desc* d) {
  return attn_large_applies(d) ? attn_large_bwd_ws_bytes(d) : bwd_workspace_of(d).total;
}

int check_attn_inputs(const char* who, const spotv2_gat_desc* d, std::initializer_list<ArgCheck> own_args,
                      std::initializer_list<ArgCheck> own_layout, const AttnEdgeArgs& e) {
  for (const ArgCheck& c : own_args)
    if (!c.ok) return fail(c.st, "%s", c.msg);
  const bool structured = d->edge_mode == 1 && d->Fe > 0;
  if (d->Fe > 0 && !structured && !(e.rows && e.table && e.v))
    return fail(SPOTV2_ERR_INVALID_ARG, "%s: edge_rows, table and v are required when Fe > 0", who);
  if (structured && !e.backward && !e.terms)
    return fail(SPOTV2_ERR_INVALID_ARG, "%s: edge_mode 1 needs edge_terms (spotv2_edge_terms_from_windows)", who);
  if (structured && e.backward && !(e.terms && e.dterms && aligned16(e.dterms)))
    return fail(SPOTV2_ERR_INVALID_ARG, "%s: edge_mode 1 needs edge_terms and a 16-byte aligned d_edge_terms buffer", who);
  for (const ArgCheck& c : own_layout)
    if (!c.ok) return fail(c.st, "%s", c.msg);
  if (d->H > kMaxHeads) return fail(SPOTV2_ERR_UNSUPPORTED, "H=%d > %d", d->H, kMaxHeads);
  if (d->Fe > kMaxFe) return fail(SPOTV2_ERR_UNSUPPORTED, "Fe=%d > %d", d->Fe, kMaxFe);
  if (!aligned16(e.terms)) return fail(SPOTV2_ERR_INVALID_ARG, "%s: edge_terms must be 16-byte aligned", who);
  if (!aligned16(e.dterms)) return fail(SPOTV2_ERR_INVALID_ARG, "%s: d_edge_terms must be 16-byte aligned", who);
  return SPOTV2_OK;
}

AttnParams attn_params_of(const spotv2_gat_desc* d, const AttnEdgeArgs& e) {
  AttnParams p{};
  p.B = d->B; p.N = d->N; p.F = d->F; p.Fe = d->Fe; p.H = d->H; p.C = d->C;
  p.R = d->R; p.concat = d->concat; p.ldp = d->ldp;
  p.ldo = d->concat ? d->H * d->C : d->C;
  p.slope = d->negative_slope;
  p.drop = dropout_params(d);
  p.lg_tensor_cores = d->gemm_algo != 1;
  p.edge_rows = e.rows; p.table = e.table; p.v = e.v;
  p.bulk_ok = d->Fe > 0 && aligned16(e.rows) && ((size_t)d->R * d->Fe) % 4 == 0;
  p.vec2_ok = (d->C % 2 == 0);
  p.edge_terms = d->Fe > 0 ? const_cast<float*>(e.terms) : nullptr;
  p.terms_in = (d->edge_mode == 1 && d->Fe > 0) ? 1 : 0;
  p.dterms_out = d->Fe > 0 ? e.dterms : nullptr;      // both edge modes (edge_mode 0: spotv2_gat_edge_rows_grad)
  if (d->p_format == 1) {
    p.hp = head_pitch_of(d);
    p.ldp16 = ld16_of(n_aug_of(d));
    p.alpha_rec = attn_record_of(d);
  }
  return p;
}

enum class BwdKernel { kLarge, kTcgen05, kPipelined, kPhaseSerial };

// N > 32: the large-universe path.  Else attn_bwd_algo 0 = the pipelined kernel (attn_bwd2.cu) when its shared-memory plan
// fits, else the phase-serial one of this file; 1 = phase-serial; 2 = pipelined or error; 3 = tcgen05 (attn_bwd3.cu) or error,
// opt-in because on a B200 the shared-memory port bounds it below the pipelined kernel (DESIGN.md section 6).
static int choose_bwd_kernel(const spotv2_gat_desc* d, const AttnParams& p, BwdKernel* k) {
  *k = attn_large_applies(d) ? BwdKernel::kLarge : d->attn_bwd_algo == 3 ? BwdKernel::kTcgen05 : BwdKernel::kPipelined;
  if (*k == BwdKernel::kTcgen05 && !attn_bwd3_applies(p))
    return fail(SPOTV2_ERR_UNSUPPORTED, "attn_bwd: the tcgen05 kernel covers head-mean layers with N <= 31, C %% 4 == 0, even Fe <= 128 "
                                        "and the forward's edge terms");
  if (*k != BwdKernel::kPipelined) return SPOTV2_OK;
  if (p.terms_in && !attn_bwd2_fits(p))
    return fail(SPOTV2_ERR_UNSUPPORTED, "attn_bwd: edge_mode 1 needs the pipelined kernel, whose shared-memory plan does not fit this shape");
  if (d->attn_bwd_algo == 1 || (d->attn_bwd_algo != 2 && !attn_bwd2_fits(p))) *k = BwdKernel::kPhaseSerial;
  return SPOTV2_OK;
}

// |dP_h[j,c]| = |g sum_i alpha_h[i,j] dO[i,c]| <= g N max|dout|  (g = 1/H for the head mean); attention dropout scales the
// kept coefficients by 1/(1-p), and the bound grows with it
static float dp_bound(const AttnParams& p) { return (float)p.N * (p.concat ? 1.f : 1.f / (float)p.H) * p.drop.scale; }

// ds | dd (a.dsd) -> columns [hc, hc + 2H) of the dP operand pair (hc: first s|d column of the pair's layout)
static int split_dsd(const AttnBwdArgs& a, int hc, cudaStream_t st) {
  const size_t total = (size_t)a.p.B * a.p.N * 2 * a.p.H;
  split_dsd_kernel<<<(unsigned)std::min<size_t>((total + 255) / 256, (size_t)8 * 148), 256, 0, st>>>(
      a.dsd, total, 2 * a.p.H, a.dP_hi16 + hc, a.dP_lo16 ? a.dP_lo16 + hc : nullptr, a.ldp16, a.dp_blk);
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

template <int NPAIRS>
static int launch_bwd(AttnBwdArgs& a, float* dv, float* dbias, void* ws, size_t ws_bytes, cudaStream_t st) {
  const AttnParams& p = a.p;
  // largest ring stage (multiple of 16 rows) that keeps two CTAs per SM, else one
  BwdSmem sm = bwd_smem_plan(p.N, p.Fe, p.H, p.C, p.R, NPAIRS, p.concat, kBwdChunkRows);
  for (int rows = kBwdChunkRows - 16; rows >= 16 && sm.total > 113 * 1024; rows -= 16)
    sm = bwd_smem_plan(p.N, p.Fe, p.H, p.C, p.R, NPAIRS, p.concat, rows);
  if (sm.total > 227 * 1024)
    return fail(SPOTV2_ERR_UNSUPPORTED, "attn_bwd needs %zu B shared memory (> 227 KB)", sm.total);
  auto kern = gat_attn_bwd_kernel<NPAIRS>;
  SPOTV2_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm.total));
  int grid = 2 * sm_count();
  if (grid > p.B) grid = p.B;
  const size_t need = ((size_t)grid * ((size_t)p.H * p.Fe + p.ldo)) * sizeof(float);
  if (!ws || ws_bytes < need)
    return fail(SPOTV2_ERR_WORKSPACE, "attn_bwd needs %zu B of workspace, got %zu", need, ws_bytes);
  a.dv_part = static_cast<float*>(ws);
  a.dbias_part = a.dv_part + (size_t)grid * p.H * p.Fe;
  kern<<<grid, kAttnThreads, sm.total, st>>>(a, sm);
  SPOTV2_CUDA_OK(cudaGetLastError());
  if (dv && p.Fe > 0) {
    const int len = p.H * p.Fe;
    partial_reduce_kernel<<<(len + 31) / 32, 256, 0, st>>>(a.dv_part, grid, len, dv);
  }
  if (dbias) partial_reduce_kernel<<<(p.ldo + 31) / 32, 256, 0, st>>>(a.dbias_part, grid, p.ldo, dbias);
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

}  // namespace spotv2

namespace spotv2 {
int bwd_diag_add(unsigned long long* host_out, int reset) {
  if (int rc = diag_add(host_out, g_bwd_counters, reset)) return rc;
  if (int rc = bwd2_diag_add(host_out, reset)) return rc;       // whichever kernel ran contributes; the others add zeros
  return bwd3_diag_add(host_out, reset);
}
}  // namespace spotv2

using namespace spotv2;

extern "C" int spotv2_gat_attn_bwd(const spotv2_gat_desc* d, const float* P_aug, const float* p_amax_or_null,
                                   const float* edge_rows, const float* edge_terms_or_null, const int32_t* table,
                                   const float* v,
                                   const float* dout, float* dP_aug_or_null, void* dP_hi_or_null, void* dP_lo_or_null,
                                   float* dp_scale_or_null, float* dv_or_null, float* d_edge_terms_or_null,
                                   float* dbias_or_null, void* ws, size_t ws_bytes, void* stream) {
  if (int rc = check_desc(d)) return rc;
  const bool f16 = dP_hi_or_null != nullptr, structured = d->edge_mode == 1 && d->Fe > 0;
  const AttnEdgeArgs e{edge_rows, table, v, edge_terms_or_null, d_edge_terms_or_null, true};
  if (int rc = check_attn_inputs(
          "attn_bwd", d,
          {{P_aug && dout, "attn_bwd: P_aug and dout must be non-null"},
           {f16 || dP_aug_or_null, "attn_bwd: give dP_aug (fp32) or dP_hi/dP_lo/dp_scale (fp16 pairs)"},
           {!f16 || (dP_lo_or_null && dp_scale_or_null), "attn_bwd: dP_hi needs dP_lo and dp_scale"}},
          {{!(structured && d->N <= 32 && d->attn_bwd_algo == 1), "attn_bwd: for N <= 32, edge_mode 1 runs on the pipelined kernel only",
            SPOTV2_ERR_UNSUPPORTED},
           {aligned16(P_aug) && aligned16(dout) && (f16 || aligned16(dP_aug_or_null)) &&
                (!f16 || (aligned16(dP_hi_or_null) && aligned16(dP_lo_or_null))),
            "attn_bwd: P_aug/dout/dP must be 16-byte aligned"}},
          e))
    return rc;
  AttnBwdArgs a{};
  a.p = attn_params_of(d, e);
  a.p.P_aug = P_aug;
  a.dout = dout; a.dP_aug = f16 ? nullptr : dP_aug_or_null;
  a.dP_hi16 = static_cast<__half*>(dP_hi_or_null); a.dP_lo16 = static_cast<__half*>(dP_lo_or_null);
  const int HC = d->H * d->C;
  a.ldp16 = ld16_of(HC + 2 * d->H);
  a.bound = 1.f; a.dp_blk = dp_scale_or_null;
  cudaStream_t st = as_stream(stream);
  BwdKernel kern;
  if (int rc = choose_bwd_kernel(d, a.p, &kern)) return rc;
  if (kern == BwdKernel::kLarge)       // several CTAs per graph (attn_large.cu); emits the pair through a split pass
    return attn_large_bwd(d, a, dv_or_null, dbias_or_null, ws, ws_bytes, st);
  const BwdWorkspace w = bwd_workspace_of(d);
  if (!ws || ws_bytes < w.total)
    return fail(SPOTV2_ERR_WORKSPACE, "attn_bwd needs %zu B of workspace, got %zu", w.total, ws_bytes);
  unsigned char* base = static_cast<unsigned char*>(ws);
  float* blk_dout = reinterpret_cast<float*>(base + w.blocks);
  float* blk_tmp = blk_dout + kScaleBlockFloats;
  float* blk_p = blk_tmp + kScaleBlockFloats;
  const size_t rows = (size_t)d->B * d->N;
  // the two big products run on fp16 operand pairs scaled by their tensors' maxima
  a.dout_blk = blk_dout;
  if (int rc = amax_flat(dout, rows * (size_t)a.p.ldo, blk_dout, st)) return rc;
  a.p_amax = p_amax_or_null;
  if (!a.p_amax) {            // P_aug did not come from spotv2_proj_fwd: one extra pass over it
    if (int rc = amax_2d(P_aug, (int)rows, HC, (size_t)d->ldp, blk_p, st)) return rc;
    a.p_amax = blk_p;
  }
  // the pipelined and the tcgen05 kernels collect max |ds|, |dd| themselves (dp_scale block entry 1, zeroed here)
  const bool dsd_fused = f16 && kern != BwdKernel::kPhaseSerial;
  if (f16) {
    a.dsd = reinterpret_cast<float*>(base + w.dsd);
    a.bound = dp_bound(a.p);
    SPOTV2_CUDA_OK(cudaMemsetAsync(dp_scale_or_null, 0, kScaleBlockFloats * sizeof(float), st));
  }
  if (dsd_fused) a.dsd_amax = reinterpret_cast<unsigned*>(dp_scale_or_null) + 1;
  float* dv = structured ? nullptr : dv_or_null;      // edge_mode 1: spotv2_windows_dv forms dv
  const int np = (d->N + 1) / 2;
  int rc;
  if (kern == BwdKernel::kTcgen05) rc = launch_attn_bwd3(a, dv, dbias_or_null, ws, ws_bytes, st);
  else if (kern == BwdKernel::kPipelined) rc = launch_attn_bwd2(a, dv, dbias_or_null, ws, ws_bytes, st);
  else if (np <= 4) rc = launch_bwd<4>(a, dv_or_null, dbias_or_null, ws, ws_bytes, st);
  else if (np <= 8) rc = launch_bwd<8>(a, dv_or_null, dbias_or_null, ws, ws_bytes, st);
  else if (np <= 15) rc = launch_bwd<15>(a, dv_or_null, dbias_or_null, ws, ws_bytes, st);
  else if (np <= 16) rc = launch_bwd<16>(a, dv_or_null, dbias_or_null, ws, ws_bytes, st);
  else return fail(SPOTV2_ERR_UNSUPPORTED, "N=%d > 32: the one-CTA-per-graph kernel covers N <= 32", d->N);
  if (rc) return rc;
  if (dsd_fused) return split_dsd(a, HC, st);
  if (f16) {
    // ds | dd: own scale group (columns [HC, HC + 2H) of the fp16 pair arrays)
    const int none = 0x7fffffff;
    if ((rc = split_f16(a.dsd, (int)rows, 2 * d->H, 2 * d->H, 0, none, nullptr, 0, a.dP_hi16 + HC, a.dP_lo16 + HC,
                        a.ldp16, blk_tmp, st)))
      return rc;
    SPOTV2_CUDA_OK(cudaMemcpyAsync(dp_scale_or_null + 3, blk_tmp + 2, sizeof(float), cudaMemcpyDeviceToDevice, st));
    SPOTV2_CUDA_OK(cudaMemcpyAsync(dp_scale_or_null + 5, blk_tmp + 4, sizeof(float), cudaMemcpyDeviceToDevice, st));
  }
  return SPOTV2_OK;
}


// p_format 1: same operator, P as the fp16 operand pair, dP emitted in the padded head pitch (attn_bwd2.cu, P16 instantiations)
extern "C" int spotv2_gat_attn_bwd_pair(const spotv2_gat_desc* d, const void* P_hi, const void* P_lo_or_null, const float* p_scale,
                                        const float* sd, const float* edge_rows, const float* edge_terms_or_null, const int32_t* table,
                                        const float* v, const float* dout, void* dP_hi, void* dP_lo_or_null, float* dp_scale,
                                        float* dv_or_null, float* d_edge_terms_or_null, float* dbias_or_null, void* ws,
                                        size_t ws_bytes, void* stream) {
  if (int rc = check_desc(d)) return rc;
  const bool single = d->gemm_algo == 3;
  const AttnEdgeArgs e{edge_rows, table, v, edge_terms_or_null, d_edge_terms_or_null, true};
  if (int rc = check_attn_inputs(
          "attn_bwd_pair", d,
          {{d->p_format == 1, "attn_bwd_pair: the descriptor must say p_format 1"},
           {P_hi && p_scale && sd && dout && dP_hi && dp_scale, "attn_bwd_pair: P_hi, p_scale, sd, dout, dP_hi and dp_scale must be non-null"},
           {single || (P_lo_or_null && dP_lo_or_null), "attn_bwd_pair: the lo planes may be omitted with gemm_algo 3 only"}},
          {{aligned16(P_hi) && aligned16(dout) && aligned16(dP_hi) && (single || (aligned16(P_lo_or_null) && aligned16(dP_lo_or_null))),
            "attn_bwd_pair: P / dout / dP must be 16-byte aligned"}},
          e))
    return rc;
  AttnBwdArgs a{};
  a.p = attn_params_of(d, e);
  a.p.P_hi = static_cast<const __half*>(P_hi);
  a.p.P_lo = single ? nullptr : static_cast<const __half*>(P_lo_or_null);
  a.p.p_blk = p_scale;
  a.p.sd32 = sd;
  a.dout = dout;
  a.dP_hi16 = static_cast<__half*>(dP_hi);
  a.dP_lo16 = single ? nullptr : static_cast<__half*>(dP_lo_or_null);
  a.ldp16 = a.p.ldp16;
  a.dp_blk = dp_scale;
  cudaStream_t st = as_stream(stream);
  if (!attn_bwd2_fits(a.p))
    return fail(SPOTV2_ERR_UNSUPPORTED, "attn_bwd_pair: the pipelined kernel's shared-memory plan does not fit this shape");
  const BwdWorkspace w = bwd_workspace_of(d);
  if (!ws || ws_bytes < w.total)
    return fail(SPOTV2_ERR_WORKSPACE, "attn_bwd_pair needs %zu B of workspace, got %zu", w.total, ws_bytes);
  unsigned char* base = static_cast<unsigned char*>(ws);
  // dout -> operand pair, unit scales, max|dout|, dbias: one pass (attn_prep.cu)
  {
    const int upg = d->concat ? d->H : 1;
    const int ldo16 = ld16_of(a.p.ldo);
    float* blk_dout = reinterpret_cast<float*>(base + w.blocks);
    __half* dhi = reinterpret_cast<__half*>(base + w.dout_pair);
    __half* dlo = single ? nullptr : reinterpret_cast<__half*>(base + w.dout_pair + w.plane);
    float* scales = reinterpret_cast<float*>(base + w.unit_scales);
    // (the bias gradient's per-CTA partials are reduced together with the dv partials, behind the attention kernel)
    float* bpart = dbias_or_null ? reinterpret_cast<float*>(base + w.dbias_part) : nullptr;
    int n_parts = 0;
    if (int rc = dout_pair_prepass(dout, d->B, d->N, d->C, upg, dhi, dlo, ldo16, scales, blk_dout, nullptr, bpart, st, &n_parts))
      return rc;
    a.dout_blk = blk_dout;
    a.dO_hi = dhi; a.dO_lo = dlo; a.dO_scale = scales; a.ldo16 = ldo16; a.units_per_graph = upg;
    a.prep_dbias_part = bpart; a.prep_dbias_n = n_parts;
  }
  a.dsd = reinterpret_cast<float*>(base + w.dsd);
  a.bound = dp_bound(a.p);
  SPOTV2_CUDA_OK(cudaMemsetAsync(dp_scale, 0, kScaleBlockFloats * sizeof(float), st));
  a.dsd_amax = reinterpret_cast<unsigned*>(dp_scale) + 1;
  if (int rc = launch_attn_bwd2(a, a.p.terms_in ? nullptr : dv_or_null, dbias_or_null, ws, ws_bytes, st)) return rc;
  return split_dsd(a, d->H * a.p.hp, st);
}


// 1 when every p_format 1 kernel covers this problem (shapes, alignment rules and the shared-memory plans of the forward
// and of the pipelined backward); callers fall back to p_format 0 otherwise.  Host-side only: no device work.
extern "C" int spotv2_gat_pair_format_supported(const spotv2_gat_desc* d) {
  if (!d || d->B <= 0 || d->N <= 0 || d->N > 32 || d->H <= 0 || d->H > kMaxHeads || d->C <= 0 || d->Fe < 0 || d->Fe > kMaxFe) return 0;
  if (d->gemm_algo == 1 || d->attn_bwd_algo == 1 || d->attn_bwd_algo == 3) return 0;
  if (d->C % 4 != 0 || d->C > 1024 || (d->concat && d->C % 8 != 0)) return 0;
  spotv2_gat_desc pair = *d;
  pair.p_format = 1;
  const AttnParams p = attn_params_of(&pair, AttnEdgeArgs{});
  return (attn_fwd16_fits(p) && attn_bwd2_fits(p)) ? 1 : 0;
}
