// Large-universe attention (N > 32 nodes per graph, BASELINE config D: the 500-node S&P-style complete
// graph): the multi-CTA-per-graph form of edge_update + softmax + propagate ([PyG] gat_conv.py
// edge_update/message, utils/softmax.py, aggr='add'; reached from /root/reference/utils/models.py:146)
// and of its autograd.
//
// One graph no longer fits a CTA (the attention tile alone is H*N*N*4 = 6 MB at N = 500), so the work of a
// graph is spread over many CTAs and the attention tile lives in HBM/L2 as Z[b][h][j (source)][i (target)]
// — 5 % of the edge rows' bytes, the same layout spotv2_gat_attn_fwd hands out for return_attention_weights.
//   L  edge logits   g_ij,h = <e_ij, v_h>: the edge rows stream once through a 2-stage shared-memory ring
//                    (1-D bulk async copies), 3xTF32 mma.sync per 16-row tile, scattered by the row table;
//   S  softmax       one thread per (graph, head, target) column: mean fill of the self loop, LeakyReLU,
//                    max-subtracted softmax over the N sources (online max/sum, 3 passes over the column);
//   G  aggregation   out_i = mean_h | concat_h  sum_j alpha_h[j][i] P[j,h,:]  as a batched exact-fp32 GEMM
//                    (128x128 tiles: ceil(N/128)^2 CTAs per (graph, head)).
// Backward (attention coefficients recomputed from the edge rows, nothing kept from the forward but P_aug):
//   L, S again;  dalpha_h = g dO_h P_h^T (batched GEMM);  softmax + LeakyReLU backward per column (writes dz in
//   place, dd, and the share of the self-loop gradient that the mean fill hands back to every incoming edge);
//   ds = row sums;  dv = sum_r (dz + fill)_r e_r over a second pass of the edge rows;  dP_h = g alpha_h dO_h
//   (batched GEMM);  dbias = column sums of dout.
// Every reduction has a fixed order (per-CTA partials summed by index), so results are reproducible.
#include <algorithm>

#include "attn_bwd.cuh"

namespace spotv2 {

namespace {

constexpr int kLgThreads = 128;

struct LgRing {               // work item q = graph * chunks_per_graph + chunk; a CTA walks q = cta, cta + grid, ...
  const float* edge_rows;
  int R, Fe, CR, cpg;         // rows per graph, features, rows per chunk, chunks per graph
  long long items;
  int bulk_ok;
  __device__ __forceinline__ int rows_of(long long q) const {
    const int c = (int)(q % cpg);
    const int r = R - c * CR;
    return r < CR ? r : CR;
  }
  __device__ __forceinline__ const float* src_of(long long q) const {
    const long long b = q / cpg, c = q - b * cpg;
    return edge_rows + ((size_t)b * R + (size_t)c * CR) * Fe;
  }
};

// Brings item q into `stage`: thread 0 issues a bulk copy (completion on `bar`) or, for unaligned edge
// blocks, the whole CTA copies cooperatively (caller syncs).
__device__ __forceinline__ void lg_issue(const LgRing& rg, long long q, float* stage, uint64_t* bar) {
  const uint32_t bytes = (uint32_t)rg.rows_of(q) * rg.Fe * 4u;
  mbar_expect_tx(bar, bytes);
  bulk_g2s(stage, rg.src_of(q), bytes, bar);
}
__device__ __forceinline__ void lg_copy(const LgRing& rg, long long q, float* stage, int tid) {
  const float* src = rg.src_of(q);
  const int n = rg.rows_of(q) * rg.Fe;
  for (int idx = tid; idx < n; idx += kLgThreads) stage[idx] = src[idx];
}

struct LgLogitArgs {
  LgRing rg;
  const int32_t* table;
  const float* v;
  float* Z;                   // [B][H][N][N]
  int N, H, KS, NT;
  uint32_t off_vfrag, off_stage, stage_bytes;
};

// L: Z[b][h][j][i] = <edge row (j -> i), v_h>.  4 warps, one 16-row MMA tile each per 64-row chunk.
__global__ void __launch_bounds__(kLgThreads) lg_edge_logit_kernel(const LgLogitArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);
  float4* vfrag = reinterpret_cast<float4*>(smem + a.off_vfrag);
  float* stage[2] = {reinterpret_cast<float*>(smem + a.off_stage),
                     reinterpret_cast<float*>(smem + a.off_stage + a.stage_bytes)};
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const LgRing& rg = a.rg;
  if (tid == 0) {
    mbar_init(&full[0], 1);
    mbar_init(&full[1], 1);
    fence_mbar_init();
  }
  build_vfrag(vfrag, a.v, a.H, rg.Fe, a.KS, a.NT, tid, kLgThreads);
  __syncthreads();
  const long long q0 = blockIdx.x, step = gridDim.x;
  if (rg.bulk_ok && tid == 0) {
    if (q0 < rg.items) lg_issue(rg, q0, stage[0], &full[0]);
    if (q0 + step < rg.items) lg_issue(rg, q0 + step, stage[1], &full[1]);
  }
  uint32_t it = 0;
  for (long long q = q0; q < rg.items; q += step, ++it) {
    const int s = it & 1;
    const int rows = rg.rows_of(q);
    if (rg.bulk_ok) {
      mbar_wait(&full[s], (it >> 1) & 1);
    } else {
      lg_copy(rg, q, stage[s], tid);
      __syncthreads();
    }
    if (warp * 16 < rows) {
      const long long b = q / rg.cpg;
      const int row_base = (int)(q - b * rg.cpg) * rg.CR;
      float* Zb = a.Z + (size_t)b * a.H * a.N * a.N;
      const int N = a.N, H = a.H;
      const int32_t* table = a.table;
      warp_edge_logits<1, 4>(stage[s], vfrag, rg.Fe, a.KS, a.NT, warp * 16, lane, [&](int r, int h, float val) {
        if (r < rows && h < H) {
          const int code = __ldg(table + row_base + r);
          if (code >= 0) Zb[((size_t)h * N + (code & 0xffff)) * N + (code >> 16)] = val;
        }
      });
    }
    __syncthreads();
    if (rg.bulk_ok && tid == 0 && q + 2 * step < rg.items) lg_issue(rg, q + 2 * step, stage[s], &full[s]);
  }
}

// S: a block owns 32 target columns i of one (b, h) tile; its 8 thread rows split the N sources (j = ty, ty + 8,
// ...), so a warp reads 128 contiguous bytes per source row and every column has 8 independent load streams.
// Partial results meet in shared memory in a fixed order.  Zraw may be null (layer called without edge_attr: all
// edge terms 0) and may alias A.  gii_out (optional) receives the self-loop fill for the backward.
constexpr int kSmX = 32, kSmY = 8;

__device__ __forceinline__ float lg_logit(const float* zc, int j, int i, int N, float gii, float sj, float di, float slope) {
  const float g = (j == i) ? gii : (zc ? zc[(size_t)j * N] : 0.f);
  const float z = g + sj + di;
  return z > 0.f ? z : z * slope;
}

__global__ void __launch_bounds__(kSmX * kSmY)
lg_softmax_kernel(const float* __restrict__ P_aug, const float* Zraw, float* A, float* __restrict__ gii_out,
                  int N, int H, int HC, int ldp, float slope, const DropoutParams drop) {
  extern __shared__ float s_src[];             // s_j of this (b, h)
  __shared__ float red[2][kSmY][kSmX];
  const int b = blockIdx.z, h = blockIdx.y, tx = threadIdx.x, ty = threadIdx.y;
  const float* Pb = P_aug + (size_t)b * N * ldp;
  for (int j = ty * kSmX + tx; j < N; j += kSmX * kSmY) s_src[j] = Pb[(size_t)j * ldp + HC + h];
  __syncthreads();
  const int i = blockIdx.x * kSmX + tx;
  const bool live = i < N;
  const int ic = live ? i : N - 1;             // dead lanes shadow the last column and never store
  const size_t base = ((size_t)b * H + h) * N * N + ic;
  const float* zc = Zraw ? Zraw + base : nullptr;
  float* ac = A + base;
  const float di = Pb[(size_t)ic * ldp + HC + H + h];
  float gsum = 0.f;
  if (zc) {
#pragma unroll 8
    for (int j = ty; j < N; j += kSmY) gsum += (j != ic) ? zc[(size_t)j * N] : 0.f;
  }
  red[0][ty][tx] = gsum;
  __syncthreads();
  gsum = 0.f;
#pragma unroll
  for (int k = 0; k < kSmY; ++k) gsum += red[0][k][tx];
  const float gii = gsum / (float)(N > 1 ? N - 1 : 1);
  if (gii_out && live && ty == 0) gii_out[((size_t)b * H + h) * N + i] = gii;
  float mx = -INFINITY, sum = 0.f;
#pragma unroll 8
  for (int j = ty; j < N; j += kSmY) {
    const float l = lg_logit(zc, j, ic, N, gii, s_src[j], di, slope);
    if (l > mx) {
      sum *= expf(mx - l);
      mx = l;
    }
    sum += expf(l - mx);
  }
  __syncthreads();
  red[0][ty][tx] = mx;
  red[1][ty][tx] = sum;
  __syncthreads();
  float M = -INFINITY;
#pragma unroll
  for (int k = 0; k < kSmY; ++k) M = fmaxf(M, red[0][k][tx]);
  float S = 0.f;
#pragma unroll
  for (int k = 0; k < kSmY; ++k) S += red[0][k][tx] == -INFINITY ? 0.f : red[1][k][tx] * expf(red[0][k][tx] - M);
  const float inv = 1.f / (S + 1e-16f);
  if (!live) return;
#pragma unroll 8
  for (int j = ty; j < N; j += kSmY) {
    const float l = lg_logit(zc, j, ic, N, gii, s_src[j], di, slope);
    float a = expf(l - M) * inv;
    if (drop.p > 0.f)        // forward only: the backward recomputes with drop.p = 0 and applies the mask itself
      a = dropout_keep(drop, (((unsigned long long)b * H + h) * N + i) * N + j) ? a * drop.scale : 0.f;
    ac[(size_t)j * N] = a;
  }
}

// Softmax + LeakyReLU backward, same thread layout.  dA holds dalpha on entry and dz on exit (diagonal included:
// it is the self loop's dz); fill[b,h,i] = dz_ii / (N - 1), the gradient every incoming edge term of i receives
// through the mean fill; dd_i goes to column HC + H + h of dP_aug.
// The kernel without and with the gradient through the returned coefficients (spotv2_gat_attn_bwd_dalpha)
#define SPOTV2_KERNEL_NAME lg_softmax_bwd_kernel
#define SPOTV2_GA 0
#include "attn_large_softmax_bwd.cuh"
#undef SPOTV2_KERNEL_NAME
#undef SPOTV2_GA
#define SPOTV2_KERNEL_NAME lg_softmax_bwd_dalpha_kernel
#define SPOTV2_GA 1
#include "attn_large_softmax_bwd.cuh"
#undef SPOTV2_KERNEL_NAME
#undef SPOTV2_GA

// ds_j = sum_i dz[j][i] -> column HC + h of dP_aug.  One warp per (b, h, j) row, fixed lane-strided order.
__global__ void __launch_bounds__(256)
lg_rowsum_kernel(const float* __restrict__ dZ, float* dP_aug, int B, int N, int H, int HC, int ldp) {
  const long long w = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= (long long)B * H * N) return;
  const int j = (int)(w % N);
  const long long bh = w / N;
  const int h = (int)(bh % H);
  const long long b = bh / H;
  const float* row = dZ + (size_t)w * N;
  float s = 0.f;
  for (int i = lane; i < N; i += 32) s += row[i];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) dP_aug[((size_t)b * N + j) * ldp + HC + h] = s;
}

// d(edge terms) for the structured source: w[b][h][j][i] = dz[b][h][j][i] + fill[b][h][i] off the diagonal, 0 on it.
// One block per row (b*H + h)*N + j, threads along i: no index divisions in the hot path.
__global__ void __launch_bounds__(128)
lg_dterms_kernel(const float* __restrict__ dZ, const float* __restrict__ fill, float* __restrict__ out, int N) {
  const size_t row = blockIdx.x;
  const int j = (int)(row % N);
  const float* fl = fill + (row / N) * N;
  const float* src = dZ + row * N;
  float* dst = out + row * N;
  for (int i = threadIdx.x; i < N; i += blockDim.x) dst[i] = (i != j) ? src[i] + fl[i] : 0.f;
}

struct LgDvArgs {
  LgRing rg;
  const int32_t* table;
  const float* dZ;            // [B][H][N][N] dz
  const float* fill;          // [B][H][N]
  double* part;               // [grid][H*Fe]
  int N, H;
  uint32_t off_w, off_stage, stage_bytes;
};

// dv[h][k] = sum over edge rows r = (j -> i) of (dz[h][j][i] + fill[h][i]) * e_r[k].  Thread = (feature k [+128, ...],
// row group rg): the RG row groups take alternate rows of a chunk, so a CTA carries 4*RG warps of independent
// LDS -> FFMA2 chains (one group alone left the SM at 12 warps and 23 % issue utilisation - ncu).  Per-chunk sums
// in fp32, each thread's running total in fp64; every (CTA, row group) writes its own partial.
template <int KPT, int RG>
__global__ void __launch_bounds__(kLgThreads * RG, RG >= 4 ? 2 : 3) lg_dv_kernel(const LgDvArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  constexpr int NT = kLgThreads * RG;
  constexpr int GIT = (64 * 8 + NT - 1) / NT;                    // (row, head) weights each thread gathers per chunk
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);
  float* wrow = reinterpret_cast<float*>(smem + a.off_w);       // [2][CR][8]
  float* stage[2] = {reinterpret_cast<float*>(smem + a.off_stage),
                     reinterpret_cast<float*>(smem + a.off_stage + a.stage_bytes)};
  const int tid = threadIdx.x, kt = tid & (kLgThreads - 1), rgp = tid / kLgThreads;
  const LgRing& rg = a.rg;
  const int Fe = rg.Fe, N = a.N, H = a.H;
  if (tid == 0) {
    mbar_init(&full[0], 1);
    mbar_init(&full[1], 1);
    fence_mbar_init();
  }
  __syncthreads();
  const long long q0 = blockIdx.x, step = gridDim.x;
  if (rg.bulk_ok && tid == 0) {
    if (q0 < rg.items) lg_issue(rg, q0, stage[0], &full[0]);
    if (q0 + step < rg.items) lg_issue(rg, q0 + step, stage[1], &full[1]);
  }
  double tot[KPT][8];
#pragma unroll
  for (int kk = 0; kk < KPT; ++kk)
#pragma unroll
    for (int h = 0; h < 8; ++h) tot[kk][h] = 0.0;
  // Row weights w_r[h] = dz[h][j][i] + fill[h][i] of a chunk, one (row, head) per thread slot, gathered through the
  // row table one chunk AHEAD so the two dependent scattered loads hide behind the current chunk's wait and FMAs.
  auto gather = [&](long long q, float (&w)[GIT]) {
    const int rows = rg.rows_of(q);
    const long long b = q / rg.cpg;
    const int row_base = (int)(q - b * rg.cpg) * rg.CR;
#pragma unroll
    for (int g = 0; g < GIT; ++g) {
      const int idx = tid + g * NT, r = idx >> 3, h = idx & 7;
      w[g] = 0.f;
      if (r < rows && h < H) {
        const int code = __ldg(a.table + row_base + r);
        if (code >= 0) {
          const int i = code >> 16, j = code & 0xffff;
          w[g] = __ldg(a.dZ + (((size_t)b * H + h) * N + j) * N + i) + __ldg(a.fill + ((size_t)b * H + h) * N + i);
        }
      }
    }
  };
  auto put = [&](int buf, const float (&w)[GIT]) {
#pragma unroll
    for (int g = 0; g < GIT; ++g) {
      const int idx = tid + g * NT;
      if (idx < rg.CR * 8) wrow[(size_t)buf * rg.CR * 8 + idx] = w[g];
    }
  };
  float wnext[GIT];
  if (q0 < rg.items) {
    gather(q0, wnext);
    put(0, wnext);
  }
  uint32_t it = 0;
  for (long long q = q0; q < rg.items; q += step, ++it) {
    const int s = it & 1;
    const int rows = rg.rows_of(q);
    const bool more = q + step < rg.items;
    if (more) gather(q + step, wnext);
    if (rg.bulk_ok) {
      mbar_wait(&full[s], (it >> 1) & 1);
    } else {
      const float* src = rg.src_of(q);
      for (int idx = tid; idx < rows * Fe; idx += NT) stage[s][idx] = src[idx];
    }
    __syncthreads();
    float2 acc[KPT][4];
#pragma unroll
    for (int kk = 0; kk < KPT; ++kk)
#pragma unroll
      for (int p = 0; p < 4; ++p) acc[kk][p] = make_float2(0.f, 0.f);
    const float* T = stage[s];
    const float* wr = wrow + (size_t)s * rg.CR * 8;
#pragma unroll 4
    for (int r = rgp; r < rows; r += RG) {
      const float4 w0 = *reinterpret_cast<const float4*>(wr + r * 8);
      const float4 w1 = *reinterpret_cast<const float4*>(wr + r * 8 + 4);
      const float2 wp[4] = {make_float2(w0.x, w0.y), make_float2(w0.z, w0.w), make_float2(w1.x, w1.y),
                            make_float2(w1.z, w1.w)};
#pragma unroll
      for (int kk = 0; kk < KPT; ++kk) {
        const int k = kt + kk * kLgThreads;
        const float e = k < Fe ? T[r * Fe + k] : 0.f;
        const float2 ed = make_float2(e, e);
#pragma unroll
        for (int p = 0; p < 4; ++p) acc[kk][p] = ffma2(ed, wp[p], acc[kk][p]);
      }
    }
#pragma unroll
    for (int kk = 0; kk < KPT; ++kk)
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        tot[kk][2 * p] += (double)acc[kk][p].x;
        tot[kk][2 * p + 1] += (double)acc[kk][p].y;
      }
    if (more) put(s ^ 1, wnext);
    __syncthreads();
    if (rg.bulk_ok && tid == 0 && q + 2 * step < rg.items) lg_issue(rg, q + 2 * step, stage[s], &full[s]);
  }
  double* out = a.part + ((size_t)blockIdx.x * RG + rgp) * H * Fe;
#pragma unroll
  for (int kk = 0; kk < KPT; ++kk) {
    const int k = kt + kk * kLgThreads;
    if (k < Fe)
#pragma unroll
      for (int h = 0; h < 8; ++h)
        if (h < H) out[(size_t)h * Fe + k] = tot[kk][h];
  }
}

// out[k] = sum_c part[c][k], fixed order; a warp per output element strides over the partials (lane l takes c = l,
// l + 32, ...) and combines its 32 lane sums by a butterfly.
__global__ void lg_reduce_f64_kernel(const double* __restrict__ part, int nparts, int len, float* __restrict__ out) {
  const int k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (k >= len) return;
  double s = 0.0;
  for (int c = lane; c < nparts; c += 32) s += part[(size_t)c * len + k];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) out[k] = (float)s;
}

// dbias partials: part[chunk][c] = sum of dout[r][c] over the chunk's rows.
__global__ void __launch_bounds__(128)
lg_colsum_kernel(const float* __restrict__ src, long long rows, int cols, int rows_per_chunk, float* __restrict__ part) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  const long long r0 = (long long)blockIdx.y * rows_per_chunk;
  const long long r1 = r0 + rows_per_chunk < rows ? r0 + rows_per_chunk : rows;
  float s = 0.f;
  for (long long r = r0; r < r1; ++r) s += src[(size_t)r * cols + c];
  part[(size_t)blockIdx.y * cols + c] = s;
}

struct LgPlan {
  int CR, cpg, KS, NT, grid;
  uint32_t off_vfrag, off_w, off_stage, stage_bytes;
  size_t smem_logit, smem_dv;
};

LgPlan lg_plan(const AttnParams& p) {
  LgPlan pl{};
  if (p.Fe <= 0) return pl;
  pl.KS = ((p.Fe + 7) / 8 + 7) / 8 * 8;
  pl.NT = (p.H + 7) / 8;
  const size_t vfrag = (size_t)pl.NT * pl.KS * 32 * 16;
  pl.off_vfrag = 128;
  pl.off_stage = (uint32_t)round_up(128 + vfrag, 128);       // the dv kernel keeps its row weights where vfrag sits
  pl.off_w = 128;
  pl.CR = 64;
  while (pl.CR > 16 && pl.off_stage + 2 * round_up((size_t)pl.CR * p.Fe * 4, 128) > 110 * 1024) pl.CR -= 16;
  pl.stage_bytes = (uint32_t)round_up((size_t)pl.CR * p.Fe * 4, 128);
  pl.smem_logit = pl.smem_dv = (size_t)pl.off_stage + 2 * (size_t)pl.stage_bytes;
  pl.cpg = (p.R + pl.CR - 1) / pl.CR;
  const long long items = (long long)p.B * pl.cpg;
  const int per_sm = (int)(220 * 1024 / (pl.smem_logit + 1024));
  long long grid = (long long)sm_count() * (per_sm < 1 ? 1 : per_sm > 4 ? 4 : per_sm);
  pl.grid = (int)(grid < items ? grid : items);
  return pl;
}

LgRing lg_ring(const AttnParams& p, const LgPlan& pl) {
  LgRing rg;
  rg.edge_rows = p.edge_rows;
  rg.R = p.R; rg.Fe = p.Fe; rg.CR = pl.CR; rg.cpg = pl.cpg;
  rg.items = (long long)p.B * pl.cpg;
  rg.bulk_ok = p.bulk_ok;
  return rg;
}

int lg_logits(const AttnParams& p, const LgPlan& pl, float* Z, cudaStream_t st) {
  // diagonal entries are never written by L; S ignores them, but keep the tile free of stale NaNs for consumers
  // that read whole rows
  LgLogitArgs a;
  a.rg = lg_ring(p, pl);
  a.table = p.table; a.v = p.v; a.Z = Z; a.N = p.N; a.H = p.H; a.KS = pl.KS; a.NT = pl.NT;
  a.off_vfrag = pl.off_vfrag; a.off_stage = pl.off_stage; a.stage_bytes = pl.stage_bytes;
  SPOTV2_CUDA_OK(cudaFuncSetAttribute(lg_edge_logit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem_logit));
  lg_edge_logit_kernel<<<pl.grid, kLgThreads, pl.smem_logit, st>>>(a);
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

int lg_softmax(const AttnParams& p, const float* Zraw, float* A, float* gii, bool apply_dropout, cudaStream_t st) {
  DropoutParams drop = p.drop;
  if (!apply_dropout) drop.p = 0.f;
  dim3 grid((p.N + kSmX - 1) / kSmX, p.H, p.B);
  lg_softmax_kernel<<<grid, dim3(kSmX, kSmY), (size_t)p.N * sizeof(float), st>>>(p.P_aug, Zraw, A, gii, p.N, p.H, p.H * p.C, p.ldp, p.slope, drop);
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

size_t tile_bytes(const spotv2_gat_desc* d) { return round_up((size_t)d->B * d->H * d->N * d->N * sizeof(float), 256); }
size_t vec_bytes(const spotv2_gat_desc* d) { return round_up((size_t)d->B * d->H * d->N * sizeof(float), 256); }
constexpr int kColsumRows = 256;

}  // namespace

bool attn_large_applies(const spotv2_gat_desc* d) { return d->N > 32; }

size_t attn_large_fwd_ws_bytes(const spotv2_gat_desc* d) { return attn_large_applies(d) ? tile_bytes(d) : 0; }

size_t attn_large_bwd_ws_bytes(const spotv2_gat_desc* d) {
  if (!attn_large_applies(d)) return 0;
  const size_t rows = (size_t)d->B * d->N;
  const size_t ldo = d->concat ? (size_t)d->H * d->C : (size_t)d->C;
  const size_t dv_part = round_up((size_t)16 * sm_count() * d->H * (d->Fe > 0 ? d->Fe : 1) * sizeof(double), 256);
  const size_t db_part = round_up(((rows + kColsumRows - 1) / kColsumRows) * ldo * sizeof(float), 256);
  // Zraw | A | dA | gii | fill | dv partials | dbias partials | fp32 dP_aug scratch (fp16-pair output only)
  return 3 * tile_bytes(d) + 2 * vec_bytes(d) + dv_part + db_part + round_up(rows * d->ldp * sizeof(float), 256) + 256;
}

int attn_large_fwd(const AttnParams& p, const float* bias, float* out, float* alpha_out, void* ws, size_t ws_bytes,
                   cudaStream_t st) {
  const size_t tile = round_up((size_t)p.B * p.H * p.N * p.N * sizeof(float), 256);
  float* A = alpha_out;
  if (!A) {
    if (!ws || ws_bytes < tile)
      return fail(SPOTV2_ERR_WORKSPACE, "attn_fwd (N=%d > 32) needs %zu B of workspace for the attention tile, got %zu",
                  p.N, tile, ws_bytes);
    A = static_cast<float*>(ws);
  }
  const LgPlan pl = lg_plan(p);
  float* Zraw = p.edge_terms ? p.edge_terms : A;       // kept for the backward when the caller provides the buffer
  if (p.Fe > 0 && !p.terms_in) {          // terms_in: the caller computed the edge terms (structured source)
    if (pl.smem_logit > 227 * 1024) return fail(SPOTV2_ERR_UNSUPPORTED, "attn_fwd (large N): Fe=%d needs %zu B shared memory", p.Fe, pl.smem_logit);
    if (int rc = lg_logits(p, pl, Zraw, st)) return rc;
  }
  if (int rc = lg_softmax(p, p.Fe > 0 ? Zraw : nullptr, A, nullptr, true, st)) return rc;
  const long long NN = (long long)p.N * p.N;
  BGemm g{};
  g.tensor_cores = p.lg_tensor_cores;
  g.M = p.N; g.N = p.C; g.K = p.N;
  g.A = A; g.lda = p.N;                   // alpha_h stored [j][i]: [K, rows]
  g.B = p.P_aug; g.ldb = p.ldp;           // P_h stored [j][c]:     [K, rows]
  g.C = out; g.ldc = p.ldo;
  g.a_o = (long long)p.H * NN; g.b_o = (long long)p.N * p.ldp; g.c_o = (long long)p.N * p.ldo;
  g.bias = bias;
  if (p.concat) {
    g.inner = p.H; g.a_i = NN; g.b_i = p.C; g.c_i = p.C; g.segs = 1; g.scale = 1.f; g.bias_i = p.C;
    return bgemm_simt(false, false, g, p.B * p.H, st);
  }
  g.inner = 1; g.segs = p.H; g.a_s = NN; g.b_s = p.C; g.scale = 1.f / (float)p.H; g.bias_i = 0;
  return bgemm_simt(false, false, g, p.B, st);
}

int attn_large_bwd(const spotv2_gat_desc* d, AttnBwdArgs& a, float* dv, float* dbias, void* ws, size_t ws_bytes,
                   cudaStream_t st, const float* d_alpha) {
  const AttnParams& p = a.p;
  if (!ws || ws_bytes < attn_large_bwd_ws_bytes(d))
    return fail(SPOTV2_ERR_WORKSPACE, "attn_bwd (N=%d > 32) needs %zu B of workspace, got %zu", p.N,
                attn_large_bwd_ws_bytes(d), ws_bytes);
  const size_t rows = (size_t)p.B * p.N;
  const int HC = p.H * p.C;
  unsigned char* w = static_cast<unsigned char*>(ws);
  float* Zraw = reinterpret_cast<float*>(w); w += tile_bytes(d);
  float* A = reinterpret_cast<float*>(w);    w += tile_bytes(d);
  float* dA = reinterpret_cast<float*>(w);   w += tile_bytes(d);
  float* gii = reinterpret_cast<float*>(w);  w += vec_bytes(d);
  float* fill = reinterpret_cast<float*>(w); w += vec_bytes(d);
  double* dv_part = reinterpret_cast<double*>(w);
  w += round_up((size_t)16 * sm_count() * p.H * (p.Fe > 0 ? p.Fe : 1) * sizeof(double), 256);
  float* db_part = reinterpret_cast<float*>(w);
  const int db_chunks = (int)((rows + kColsumRows - 1) / kColsumRows);
  w += round_up((size_t)db_chunks * p.ldo * sizeof(float), 256);
  float* dP = a.dP_aug ? a.dP_aug : reinterpret_cast<float*>(w);

  const LgPlan pl = lg_plan(p);
  if (p.Fe > 0) {
    if (pl.smem_logit > 227 * 1024) return fail(SPOTV2_ERR_UNSUPPORTED, "attn_bwd (large N): Fe=%d needs %zu B shared memory", p.Fe, pl.smem_logit);
    if (p.edge_terms) Zraw = p.edge_terms;            // the forward kept them: no first pass over the edge rows
    else if (int rc = lg_logits(p, pl, Zraw, st)) return rc;
  }
  const float* Zr = p.Fe > 0 ? Zraw : nullptr;
  if (int rc = lg_softmax(p, Zr, A, gii, false, st)) return rc;

  const long long NN = (long long)p.N * p.N;
  const float gsc = p.concat ? 1.f : 1.f / (float)p.H;
  {   // dalpha_h[j][i] = g sum_c P[j,h,c] dO[i,(h)c]
    BGemm g{};
    g.tensor_cores = p.lg_tensor_cores;
    g.M = p.N; g.N = p.N; g.K = p.C;
    g.A = p.P_aug; g.lda = p.ldp; g.B = a.dout; g.ldb = p.ldo; g.C = dA; g.ldc = p.N;
    g.inner = p.H; g.segs = 1; g.scale = gsc;
    g.a_o = (long long)p.N * p.ldp; g.a_i = p.C;
    g.b_o = (long long)p.N * p.ldo; g.b_i = p.concat ? p.C : 0;
    g.c_o = (long long)p.H * NN; g.c_i = NN;
    if (int rc = bgemm_simt(true, true, g, p.B * p.H, st)) return rc;
  }
  {
    dim3 grid((p.N + kSmX - 1) / kSmX, p.H, p.B);
    if (d_alpha)
      lg_softmax_bwd_dalpha_kernel<<<grid, dim3(kSmX, kSmY), (size_t)p.N * sizeof(float), st>>>(p.P_aug, Zr, A, dA, gii, fill, dP, p.N,
                                                                                   p.H, HC, p.ldp, p.slope, p.drop, d_alpha);
    else
      lg_softmax_bwd_kernel<<<grid, dim3(kSmX, kSmY), (size_t)p.N * sizeof(float), st>>>(p.P_aug, Zr, A, dA, gii, fill, dP, p.N, p.H, HC,
                                                                            p.ldp, p.slope, p.drop);
    SPOTV2_CUDA_OK(cudaGetLastError());
    const long long warps = (long long)p.B * p.H * p.N;
    lg_rowsum_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, st>>>(dA, dP, p.B, p.N, p.H, HC, p.ldp);
    SPOTV2_CUDA_OK(cudaGetLastError());
  }
  if (p.Fe > 0 && p.dterms_out) {
    // the gradient w.r.t. the edge terms leaves as w[b][h][j][i] = dz + fill[b][h][i] (0 on the diagonal).  Structured
    // source: dv is formed from the windows by spotv2_windows_dv; edge rows: dv below, and the caller expands w into
    // the edge rows' gradient (spotv2_gat_edge_rows_grad)
    lg_dterms_kernel<<<(unsigned)((size_t)p.B * p.H * p.N), 128, 0, st>>>(dA, fill, p.dterms_out, p.N);
    SPOTV2_CUDA_OK(cudaGetLastError());
  }
  if (p.Fe > 0 && dv && !p.terms_in) {
    LgDvArgs v;
    v.rg = lg_ring(p, pl);
    v.table = p.table; v.dZ = dA; v.fill = fill; v.part = dv_part; v.N = p.N; v.H = p.H;
    v.off_w = pl.off_w; v.off_stage = pl.off_stage; v.stage_bytes = pl.stage_bytes;
    if ((size_t)2 * pl.CR * 8 * sizeof(float) > pl.off_stage - pl.off_w || pl.CR > 64)
      return fail(SPOTV2_ERR_UNSUPPORTED, "attn_bwd (large N): row-weight block does not fit its slot");
    const int kpt = (p.Fe + kLgThreads - 1) / kLgThreads;
    int nparts = 0;
    auto launch = [&](auto kern, int rgs) -> int {
      SPOTV2_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem_dv));
      // one wave of resident CTAs (2 per SM with 4 row groups, else what shared memory allows, at most 3)
      const long long per_sm = rgs >= 4 ? 2 : 3;
      long long grid = (long long)sm_count() * per_sm;
      if (grid > pl.grid) grid = pl.grid;
      kern<<<(unsigned)grid, kLgThreads * rgs, pl.smem_dv, st>>>(v);
      SPOTV2_CUDA_OK(cudaGetLastError());
      nparts = (int)grid * rgs;
      return SPOTV2_OK;
    };
    int rc;
    if (kpt <= 1) rc = launch(lg_dv_kernel<1, 4>, 4);
    else if (kpt <= 2) rc = launch(lg_dv_kernel<2, 2>, 2);
    else rc = launch(lg_dv_kernel<4, 1>, 1);
    if (rc) return rc;
    const int len = p.H * p.Fe;
    lg_reduce_f64_kernel<<<(len * 32 + 255) / 256, 256, 0, st>>>(dv_part, nparts, len, dv);
    SPOTV2_CUDA_OK(cudaGetLastError());
  }
  {   // dP_h[j][c] = g sum_i alpha_h[j][i] dO[i,(h)c]
    BGemm g{};
    g.tensor_cores = p.lg_tensor_cores;
    g.M = p.N; g.N = p.C; g.K = p.N;
    g.A = A; g.lda = p.N; g.B = a.dout; g.ldb = p.ldo; g.C = dP; g.ldc = p.ldp;
    g.inner = p.H; g.segs = 1; g.scale = gsc;
    g.a_o = (long long)p.H * NN; g.a_i = NN;
    g.b_o = (long long)p.N * p.ldo; g.b_i = p.concat ? p.C : 0;
    g.c_o = (long long)p.N * p.ldp; g.c_i = p.C;
    if (int rc = bgemm_simt(true, false, g, p.B * p.H, st)) return rc;
  }
  if (dbias) {
    dim3 grid((p.ldo + 127) / 128, db_chunks);
    lg_colsum_kernel<<<grid, 128, 0, st>>>(a.dout, (long long)rows, p.ldo, kColsumRows, db_part);
    SPOTV2_CUDA_OK(cudaGetLastError());
    if (int rc = reduce_partials(db_part, db_chunks, p.ldo, dbias, st)) return rc;
  }
  if (a.dP_hi16) {
    // the tensor-core GEMMs take dP_aug as an fp16 pair with two scale groups (P columns | ds,dd columns)
    if (int rc = split_f16(dP, (int)rows, HC + 2 * p.H, (size_t)p.ldp, 1, HC, nullptr, 0, a.dP_hi16, a.dP_lo16,
                           (size_t)a.ldp16, a.dp_blk, st))
      return rc;
  }
  return SPOTV2_OK;
}

}  // namespace spotv2
