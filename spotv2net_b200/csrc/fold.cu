// Parameter folding / gradient unfolding, the edge-row table, the PyG-order view of the attention
// tile and the device-side window collation.  All small, bandwidth-trivial kernels.
#include <cuda_fp16.h>

#include "common.cuh"
#include "gemm.cuh"

namespace spotv2 {

__device__ __forceinline__ float block_sum_128(float x, float* red) {
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  const int w = threadIdx.x >> 5;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[w] = x;
  __syncthreads();
  return red[0] + red[1] + red[2] + red[3];
}

// One block (128 threads) per output row hc = h*C + c.
__global__ void __launch_bounds__(128)
unfold_kernel(const float* __restrict__ W, const float* __restrict__ a_src,
              const float* __restrict__ a_dst, const float* __restrict__ We,
              const float* __restrict__ a_edge, const float* __restrict__ dW_aug,
              const float* __restrict__ dv, float* __restrict__ dW, float* __restrict__ da_src,
              float* __restrict__ da_dst, float* __restrict__ dWe, float* __restrict__ da_edge,
              int H, int C, int Cp, int F, int Fe) {
  __shared__ float red[4];
  const int hc = blockIdx.x, h = hc / C;
  const int HC = H * Cp;                               // dW_aug rows: head pitch Cp (>= C; pad rows ignored)
  const size_t row = (size_t)h * Cp + (hc - h * C);
  const float as = a_src[hc], ad = a_dst[hc];
  const float* dUs = dW_aug + (size_t)(HC + h) * F;
  const float* dUd = dW_aug + (size_t)(HC + H + h) * F;
  float ps = 0.f, pd = 0.f;
  for (int f = threadIdx.x; f < F; f += 128) {
    const float w = W[(size_t)hc * F + f];
    const float us = dUs[f], ud = dUd[f];
    dW[(size_t)hc * F + f] = dW_aug[row * F + f] + as * us + ad * ud;
    ps = fmaf(w, us, ps);
    pd = fmaf(w, ud, pd);
  }
  ps = block_sum_128(ps, red);
  pd = block_sum_128(pd, red);
  if (threadIdx.x == 0) { da_src[hc] = ps; da_dst[hc] = pd; }
  if (Fe > 0) {
    const float ae = a_edge[hc];
    float pe = 0.f;
    for (int f = threadIdx.x; f < Fe; f += 128) {
      const float g = dv[(size_t)h * Fe + f];
      dWe[(size_t)hc * Fe + f] = ae * g;
      pe = fmaf(We[(size_t)hc * Fe + f], g, pe);
    }
    pe = block_sum_128(pe, red);
    if (threadIdx.x == 0) da_edge[hc] = pe;
  }
}

// The whole fold in one launch (256 threads = 32 features x 8 channel slices), three kinds of blocks:
//   ceil(F/32) * H blocks         u_src | u_dst rows of W_aug: u_k[h][f] = sum_c W[(h*C + c)*F + f] * a_k[h][c]
//   then ceil(Fe/32) * H blocks   v[h][f] = sum_c W_e[(h*C + c)*Fe + f] * a_edge[h][c]
//   then H*Cp blocks              copy: W_aug row r <- head h's row of W, or zeros for the Cp - C pad rows (p_format 1)
// Fixed-order shared-memory reductions (deterministic).
__global__ void __launch_bounds__(256)
fold_all_kernel(const float* __restrict__ W, const float* __restrict__ a_src, const float* __restrict__ a_dst,
                const float* __restrict__ We, const float* __restrict__ a_edge, float* __restrict__ W_aug, float* __restrict__ v,
                int H, int C, int Cp, int F, int Fe) {
  __shared__ float red[2][32][33];
  const int fb = (F + 31) / 32;
  const int n_red = fb * H + (We ? ((Fe + 31) / 32) * H : 0);
  int blk = blockIdx.x;
  // the reduction blocks come FIRST in the grid: each thread walks C / 8 (or C / 32) rows in a dependent chain, and with
  // the thousands of short copy blocks scheduled ahead of them they were the kernel's tail
  if (blk >= n_red) {
    blk -= n_red;
    const int h = blk / Cp, c = blk - h * Cp;
    float* dst = W_aug + (size_t)blk * F;
    if (c < C) {
      const float* src = W + ((size_t)h * C + c) * F;
      for (int f = threadIdx.x; f < F; f += 256) dst[f] = src[f];
    } else {
      for (int f = threadIdx.x; f < F; f += 256) dst[f] = 0.f;
    }
    return;
  }
  const bool edge = blk >= fb * H;
  if (edge) blk -= fb * H;
  const int nb = edge ? (Fe + 31) / 32 : fb, Fd = edge ? Fe : F;
  const int h = blk / nb, tx = threadIdx.x & 31, y = threadIdx.x >> 5;
  const int f = (blk - h * nb) * 32 + tx;
  // channel slices: 8 for the u rows, 32 for v (four per thread) - the partial sums and their order are those of the
  // two kernels this one replaced, so every folded value keeps its bits
  const int NY = edge ? 32 : 8, NQ = edge ? 4 : 1;
  const float* M = edge ? We : W;
  const float* a0 = edge ? a_edge : a_src;
  const float* a1 = edge ? nullptr : a_dst;
  for (int q = 0; q < NQ; ++q) {
    const int sl = y + 8 * q;
    float s0 = 0.f, s1 = 0.f;
    if (f < Fd) {
      const float* Mh = M + (size_t)h * C * Fd + f;
#pragma unroll 8
      for (int c = sl; c < C; c += NY) {
        const float w = Mh[(size_t)c * Fd];
        s0 = fmaf(w, a0[h * C + c], s0);
        if (a1) s1 = fmaf(w, a1[h * C + c], s1);
      }
    }
    red[0][sl][tx] = s0;
    red[1][sl][tx] = s1;
  }
  __syncthreads();
  if (y == 0 && f < Fd) {
    float t0 = 0.f, t1 = 0.f;
    for (int k = 0; k < NY; ++k) { t0 += red[0][k][tx]; t1 += red[1][k][tx]; }
    if (edge) {
      v[(size_t)h * Fe + f] = t0;
    } else {
      W_aug[((size_t)H * Cp + h) * F + f] = t0;
      W_aug[((size_t)H * Cp + H + h) * F + f] = t1;
    }
  }
}

// ---- edge-row table ---------------------------------------------------------------------
// status[0]=ok, [1]=first offending edge, [2]=reason (1 id out of range, 2 pattern differs between
// graphs, 3 pair missing or duplicated), [3] unused; status[4 .. 4+N*N) = pair counts.
__device__ __forceinline__ void table_fail(int32_t* status, int64_t where, int reason) {
  atomicExch(&status[0], 0);
  atomicMin(&status[1], (int)(where > 0x7fffffff ? 0x7fffffff : where));
  atomicMax(&status[2], reason);
}

__global__ void table_init_kernel(int32_t* status, int NN) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx == 0) { status[0] = 1; status[1] = 0x7fffffff; status[2] = 0; status[3] = 0; }
  if (idx < NN) status[4 + idx] = 0;
}

__global__ void table_local_kernel(const int64_t* __restrict__ ei, int64_t E_total, int N, int R,
                                   int32_t* __restrict__ table, int32_t* status) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  const int64_t src = ei[r], dst = ei[E_total + r];
  if (src < 0 || src >= N || dst < 0 || dst >= N) {
    table[r] = SPOTV2_ROW_SKIP;
    table_fail(status, r, 1);
    return;
  }
  if (src == dst) { table[r] = SPOTV2_ROW_SKIP; return; }
  table[r] = (int32_t)((dst << 16) | src);
  atomicAdd(&status[4 + dst * N + src], 1);
}

__global__ void table_repeat_kernel(const int64_t* __restrict__ ei, int64_t E_total, int N, int R,
                                    int32_t* status) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E_total) return;
  const int64_t b = e / R, r = e - b * R;
  if (ei[e] - b * N != ei[r] || ei[E_total + e] - b * N != ei[E_total + r]) table_fail(status, e, 2);
}

__global__ void table_complete_kernel(int N, int32_t* status) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * N) return;
  const int i = idx / N, j = idx - i * N;
  if (i != j && status[4 + idx] != 1) table_fail(status, idx, 3);
}

__global__ void table_dense_kernel(int N, int32_t* table) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * N) return;
  const int i = idx / N, j = idx - i * N;
  table[idx] = i == j ? SPOTV2_ROW_SKIP : ((i << 16) | j);
}

// alpha tile [B, H, N(j), N(i)] -> [B*R rows in input order | B*N loops] x H
__global__ void alpha_to_pyg_kernel(const float* __restrict__ tile, const int32_t* __restrict__ table,
                                    float* __restrict__ out, int B, int N, int H, int R) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n_real = (int64_t)B * R * H, n_all = n_real + (int64_t)B * N * H;
  if (idx >= n_all) return;
  if (idx < n_real) {
    const int h = idx % H;
    const int64_t e = idx / H;
    const int64_t b = e / R;
    const int r = (int)(e - b * R);
    const int code = table[r];
    float a = 0.f;
    if (code >= 0) a = tile[(((size_t)b * H + h) * N + (code & 0xffff)) * N + (code >> 16)];
    out[idx] = a;
  } else {
    const int64_t k = idx - n_real;
    const int h = k % H;
    const int64_t node = k / H;
    const int64_t b = node / N;
    const int i = (int)(node - b * N);
    out[idx] = tile[(((size_t)b * H + h) * N + i) * N + i];
  }
}

// Inverse of alpha_to_pyg_kernel for gradients: [B*R rows | B*N loops] x H -> tile [B, H, N(j), N(i)].  The table of a
// complete graph names every ordered pair i != j exactly once and the loop rows give the diagonal, so every tile entry is
// written exactly once (no atomics, no clearing pass); SPOTV2_ROW_SKIP rows (input self loops) are not read.  Threads run
// over (graph, head, row) with the row fastest: a warp's stores follow the table (source-major in PyG's order, so mostly
// consecutive), its loads are H floats apart inside the graph's block of rows, which the other heads' warps read as well.
__global__ void alpha_to_pyg_grad_kernel(const float* __restrict__ d_pyg, const int32_t* __restrict__ table,
                                         float* __restrict__ d_tile, int B, int N, int H, int R) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n_real = (int64_t)B * R * H, n_all = n_real + (int64_t)B * N * H;
  if (idx >= n_all) return;
  if (idx < n_real) {
    const int64_t bh = idx / R;
    const int r = (int)(idx - bh * R);
    const int64_t b = bh / H;
    const int h = (int)(bh - b * H);
    const int code = table[r];
    if (code >= 0) d_tile[((size_t)bh * N + (code & 0xffff)) * N + (code >> 16)] = d_pyg[((size_t)b * R + r) * H + h];
  } else {
    const int64_t k = idx - n_real;
    const int64_t bh = k / N;
    const int i = (int)(k - bh * N);
    const int64_t b = bh / H;
    const int h = (int)(bh - b * H);
    d_tile[((size_t)bh * N + i) * N + i] = d_pyg[(size_t)B * R * H + ((size_t)b * N + i) * H + h];
  }
}

// The same for graphs whose tile fits in shared memory (H*N*N floats <= 48 KB; every N <= 32 with H <= 8): one block per graph
// reads its rows coalesced, scatters them into the tile in shared memory and writes the tile out in order, so that neither
// the loads nor the stores of a warp are strided.  Every entry is written by the scatter (complete table), none is cleared.
__global__ void __launch_bounds__(256)
alpha_to_pyg_grad_graph_kernel(const float* __restrict__ d_pyg, const int32_t* __restrict__ table, float* __restrict__ d_tile,
                               int B, int N, int H, int R) {
  extern __shared__ float t_s[];                 // [H][N(j)][N(i)]
  const int b = blockIdx.x, NN = N * N;
  const float* rows = d_pyg + (size_t)b * R * H;
  for (int idx = threadIdx.x; idx < R * H; idx += blockDim.x) {
    const int r = idx / H, h = idx - r * H;
    const int code = table[r];
    if (code >= 0) t_s[h * NN + (code & 0xffff) * N + (code >> 16)] = rows[idx];
  }
  const float* loops = d_pyg + (size_t)B * R * H + (size_t)b * N * H;
  for (int idx = threadIdx.x; idx < N * H; idx += blockDim.x) {
    const int i = idx / H, h = idx - i * H;
    t_s[h * NN + i * N + i] = loops[idx];
  }
  __syncthreads();
  float* dst = d_tile + (size_t)b * H * NN;
  for (int idx = threadIdx.x; idx < H * NN; idx += blockDim.x) dst[idx] = t_s[idx];
}

// ---- window collation (utils/dataset.py:182-289 layouts, SURVEY.md Appendix B) -------------
__global__ void collate_x_kernel(const float* __restrict__ M_vol, const int32_t* __restrict__ t0,
                                 int N, int L, float* __restrict__ x, float* __restrict__ y) {
  const int node = blockIdx.x;            // b*N + i
  const int b = node / N, i = node - b * N;
  const int start = t0[b];
  const int NL = N * L;
  for (int k = threadIdx.x; k < NL; k += blockDim.x) {
    const int c = k / L, t = k - c * L;
    x[(size_t)node * NL + k] = M_vol[((size_t)(start + t) * N + i) * N + c];
  }
  if (threadIdx.x == 0) y[node] = M_vol[((size_t)(start + L) * N + i) * N + i];
}

// Same gather, and the row also leaves as the projection GEMMs' fp16 operand pair: x values are entries of the
// [T, N, N] stack, so the pair's power-of-two scale comes from the stack-wide maximum (spotv2_stack_scale, once per
// dataset) and neither an amax pass nor a split pass over x is left in the training step.
__global__ void collate_x_pair_kernel(const float* __restrict__ M_vol, const int32_t* __restrict__ t0, int N, int L,
                                      float* __restrict__ x, __half* __restrict__ hi, __half* __restrict__ lo, int ld16,
                                      const float* __restrict__ blk, float* __restrict__ y) {
  const int node = blockIdx.x;            // b*N + i
  const int b = node / N, i = node - b * N;
  const int start = t0[b];
  const int NL = N * L;
  const float s = blk[4];
  for (int k = threadIdx.x; k < NL; k += blockDim.x) {
    const int c = k / L, t = k - c * L;
    const float v = M_vol[((size_t)(start + t) * N + i) * N + c];
    if (x) x[(size_t)node * NL + k] = v;
    const float w = v * s;
    const __half h = __float2half_rn(w);
    hi[(size_t)node * ld16 + k] = h;
    lo[(size_t)node * ld16 + k] = __float2half_rn(w - __half2float(h));
  }
  for (int k = NL + threadIdx.x; k < ld16; k += blockDim.x) {          // row padding: finite zeros
    hi[(size_t)node * ld16 + k] = __float2half_rn(0.f);
    lo[(size_t)node * ld16 + k] = __float2half_rn(0.f);
  }
  if (threadIdx.x == 0) y[node] = M_vol[((size_t)(start + L) * N + i) * N + i];
}

// blk[0] holds the bit pattern of max |.|: fill in the inverse scale [2] and the scale [4] (same rule as gemm_f16.cu)
__global__ void finish_scale_block_kernel(float* blk) {
  const float amax = __uint_as_float(reinterpret_cast<const unsigned*>(blk)[0]);
  float s = 1.f;
  if (amax > 0.f && amax < INFINITY) {
    int ex;
    frexpf(amax, &ex);
    s = exp2f((float)(15 - ex));
  }
  blk[1] = 0.f; blk[2] = 1.f / s; blk[3] = 1.f / s; blk[4] = s; blk[5] = s; blk[6] = 0.f; blk[7] = 0.f;
}

__device__ __forceinline__ void tri_decode(int idx, int N, int& r, int& c) {
  // idx = r*(2N-r-1)/2 + (c-r-1), r < c
  const float fn = (float)(2 * N - 1);
  r = (int)((fn - sqrtf(fn * fn - 8.f * (float)idx)) * 0.5f);
  if (r < 0) r = 0;
  while (r > 0 && r * (2 * N - r - 1) / 2 > idx) --r;
  while ((r + 1) * (2 * N - r - 2) / 2 <= idx) ++r;
  c = idx - r * (2 * N - r - 1) / 2 + r + 1;
}

// One block per (graph b, 8 consecutive edge rows): 3L floats per row, rows written contiguously.
__global__ void __launch_bounds__(256)
collate_edge_kernel(const float* __restrict__ M_vv, const int32_t* __restrict__ t0, int N, int L,
                    float* __restrict__ ea) {
  const int E = N * (N - 1), half = E / 2;
  const int b = blockIdx.y;
  const int e_base = blockIdx.x * 8;
  const int start = t0[b];
  const int row_len = 3 * L;
  __shared__ int s_r[8], s_c[8], s_src[8], s_dst[8];
  if (threadIdx.x < 8) {
    const int e = e_base + threadIdx.x;
    if (e < E) {
      int r, c;
      tri_decode(e < half ? e : e - half, N, r, c);
      s_r[threadIdx.x] = r; s_c[threadIdx.x] = c;
      s_src[threadIdx.x] = e < half ? r : c;
      s_dst[threadIdx.x] = e < half ? c : r;
    }
  }
  __syncthreads();
  const int rows = min(8, E - e_base);
  float* out = ea + ((size_t)b * E + e_base) * row_len;
  for (int idx = threadIdx.x; idx < rows * row_len; idx += blockDim.x) {
    const int er = idx / row_len, k = idx - er * row_len;
    const int which = k / L, t = k - which * L;
    const float* M = M_vv + (size_t)(start + t) * N * N;
    const int r = s_r[er], c = s_c[er], src = s_src[er], dst = s_dst[er];
    out[idx] = which == 0 ? M[r * N + c] : (which == 1 ? M[src * N + src] : M[dst * N + dst]);
  }
}

}  // namespace spotv2

using namespace spotv2;

extern "C" int spotv2_gat_fold(const spotv2_gat_desc* d, const float* W, const float* a_src,
                               const float* a_dst, const float* W_e, const float* a_edge,
                               float* W_aug, float* v, void* stream) {
  if (int rc = check_desc(d)) return rc;
  SPOTV2_REQUIRE(W && a_src && a_dst && W_aug, "fold: W, a_src, a_dst, W_aug must be non-null");
  SPOTV2_REQUIRE(d->Fe == 0 || (W_e && a_edge && v), "fold: W_e, a_edge, v required when Fe > 0");
  cudaStream_t st = as_stream(stream);
  const int Cp = head_pitch_of(d);
  const int blocks = d->H * Cp + ((d->F + 31) / 32) * d->H + (d->Fe > 0 ? ((d->Fe + 31) / 32) * d->H : 0);
  fold_all_kernel<<<blocks, 256, 0, st>>>(W, a_src, a_dst, d->Fe > 0 ? W_e : nullptr, d->Fe > 0 ? a_edge : nullptr, W_aug, v, d->H, d->C, Cp,
                                          d->F, d->Fe);
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

extern "C" int spotv2_gat_unfold(const spotv2_gat_desc* d, const float* W, const float* a_src,
                                 const float* a_dst, const float* W_e, const float* a_edge,
                                 const float* dW_aug, const float* dv, float* dW, float* da_src,
                                 float* da_dst, float* dW_e, float* da_edge, void* stream) {
  if (int rc = check_desc(d)) return rc;
  SPOTV2_REQUIRE(W && a_src && a_dst && dW_aug && dW && da_src && da_dst, "unfold: null pointer");
  SPOTV2_REQUIRE(d->Fe == 0 || (W_e && a_edge && dv && dW_e && da_edge),
                 "unfold: edge pointers required when Fe > 0");
  unfold_kernel<<<d->H * d->C, 128, 0, as_stream(stream)>>>(W, a_src, a_dst, W_e, a_edge, dW_aug, dv,
                                                            dW, da_src, da_dst, dW_e, da_edge, d->H,
                                                            d->C, head_pitch_of(d), d->F, d->Fe);
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

extern "C" int spotv2_edge_table_build(const int64_t* edge_index, int64_t num_edges, int32_t B,
                                       int32_t N, int32_t R, int32_t* table, int32_t* status,
                                       void* stream) {
  SPOTV2_REQUIRE(edge_index && table && status, "edge_table_build: null pointer");
  SPOTV2_REQUIRE(B > 0 && N > 0 && R > 0 && N <= 0xffff, "edge_table_build: bad B/N/R");
  SPOTV2_REQUIRE(num_edges == (int64_t)B * R, "edge_table_build: num_edges=%lld != B*R=%lld",
                 (long long)num_edges, (long long)B * R);
  cudaStream_t st = as_stream(stream);
  const int NN = N * N;
  table_init_kernel<<<(NN + 255) / 256 + 1, 256, 0, st>>>(status, NN);
  table_local_kernel<<<(R + 255) / 256, 256, 0, st>>>(edge_index, num_edges, N, R, table, status);
  table_repeat_kernel<<<(unsigned)((num_edges + 255) / 256), 256, 0, st>>>(edge_index, num_edges, N, R, status);
  table_complete_kernel<<<(NN + 255) / 256, 256, 0, st>>>(N, status);
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

extern "C" int spotv2_edge_table_dense(int32_t N, int32_t* table, void* stream) {
  SPOTV2_REQUIRE(table && N > 0 && N <= 0xffff, "edge_table_dense: bad arguments");
  table_dense_kernel<<<(N * N + 255) / 256, 256, 0, as_stream(stream)>>>(N, table);
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

extern "C" int spotv2_alpha_to_pyg(const spotv2_gat_desc* d, const float* alpha_tile,
                                   const int32_t* table, float* alpha_pyg, void* stream) {
  if (int rc = check_desc(d)) return rc;
  SPOTV2_REQUIRE(alpha_tile && table && alpha_pyg, "alpha_to_pyg: null pointer");
  const int64_t total = ((int64_t)d->B * d->R + (int64_t)d->B * d->N) * d->H;
  alpha_to_pyg_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(
      alpha_tile, table, alpha_pyg, d->B, d->N, d->H, d->R);
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

extern "C" int spotv2_alpha_to_pyg_grad(const spotv2_gat_desc* d, const float* d_alpha_pyg, const int32_t* table,
                                        float* d_alpha_tile, void* stream) {
  if (int rc = check_desc(d)) return rc;
  SPOTV2_REQUIRE(d_alpha_pyg && table && d_alpha_tile, "alpha_to_pyg_grad: d_alpha_pyg, table and d_alpha_tile must be non-null");
  const size_t tile_bytes = (size_t)d->H * d->N * d->N * sizeof(float);
  if (tile_bytes <= 48 * 1024) {
    alpha_to_pyg_grad_graph_kernel<<<(unsigned)d->B, 256, tile_bytes, as_stream(stream)>>>(
        d_alpha_pyg, table, d_alpha_tile, d->B, d->N, d->H, d->R);
  } else {
    const int64_t total = ((int64_t)d->B * d->R + (int64_t)d->B * d->N) * d->H;
    alpha_to_pyg_grad_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(
        d_alpha_pyg, table, d_alpha_tile, d->B, d->N, d->H, d->R);
  }
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

extern "C" int spotv2_collate_windows(const float* M_vol, const float* M_vv, int32_t T, int32_t N,
                                      int32_t L, const int32_t* t0, int32_t B, float* x,
                                      float* edge_attr, float* y, void* stream) {
  SPOTV2_REQUIRE(M_vol && M_vv && t0 && x && y, "collate_windows: null pointer");
  SPOTV2_REQUIRE(T > L && N > 1 && L > 0 && B > 0, "collate_windows: need T > L, N > 1, L > 0, B > 0");
  cudaStream_t st = as_stream(stream);
  collate_x_kernel<<<B * N, 256, 0, st>>>(M_vol, t0, N, L, x, y);
  if (edge_attr) {            // null: the caller keeps the edges structured (window references, csrc/windows.cu)
    dim3 ge((N * (N - 1) + 7) / 8, B);
    collate_edge_kernel<<<ge, 256, 0, st>>>(M_vv, t0, N, L, edge_attr);
  }
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

extern "C" int spotv2_stack_scale(const float* M, int64_t count, float* scale_block, void* stream) {
  SPOTV2_REQUIRE(M && scale_block && count > 0, "stack_scale: null pointer or empty stack");
  cudaStream_t st = as_stream(stream);
  if (int rc = amax_flat(M, (size_t)count, scale_block, st)) return rc;
  finish_scale_block_kernel<<<1, 1, 0, st>>>(scale_block);
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

extern "C" int spotv2_collate_windows_pair(const float* M_vol, const float* M_vv, int32_t T, int32_t N, int32_t L,
                                           const int32_t* t0, int32_t B, float* x_or_null, void* x_hi, void* x_lo,
                                           int32_t ld16, const float* x_scale, float* edge_attr, float* y, void* stream) {
  SPOTV2_REQUIRE(M_vol && M_vv && t0 && x_hi && x_lo && x_scale && y, "collate_windows_pair: null pointer");
  SPOTV2_REQUIRE(T > L && N > 1 && L > 0 && B > 0, "collate_windows_pair: need T > L, N > 1, L > 0, B > 0");
  SPOTV2_REQUIRE(ld16 >= N * L && ld16 % 8 == 0, "collate_windows_pair: ld16 must be >= N*L and a multiple of 8");
  cudaStream_t st = as_stream(stream);
  collate_x_pair_kernel<<<B * N, 256, 0, st>>>(M_vol, t0, N, L, x_or_null, static_cast<__half*>(x_hi), static_cast<__half*>(x_lo),
                                               ld16, x_scale, y);
  if (edge_attr) {
    dim3 ge((N * (N - 1) + 7) / 8, B);
    collate_edge_kernel<<<ge, 256, 0, st>>>(M_vv, t0, N, L, edge_attr);
  }
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}
