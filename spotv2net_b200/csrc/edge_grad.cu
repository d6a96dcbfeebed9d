// Gradient of the layer with respect to the materialised edge rows (PyG's edge_attr.grad):
//   d edge_rows[b*R + r, :] = sum_h dz'[b][h][j][i] * v'_h      for table[r] = (i << 16) | j
//   d edge_rows[b*R + r, :] = 0                                  for SPOTV2_ROW_SKIP rows
// dz' is the attention backward's gradient w.r.t. the edge terms <e_ij, v'_h> (d_edge_terms_or_null of
// spotv2_gat_attn_bwd: the mean self-loop fill already folded in, 0 on the diagonal), v' the folded edge vector the
// forward used.  A rank-H expansion whose output is Fe / H times larger than its input: a pure store stream
// (4096 graphs x 870 rows x 126 features = 1.80 GB written, 107 MB read at the default geometry).
//
// Layout of the work.  The output is one flat fp32 array of B*R rows.  Rows are taken in groups of g = 4 / gcd(Fe, 4)
// (g * Fe floats, a multiple of 16 bytes: every group starts 16-byte aligned whatever the row pitch - Fe = 126 gives
// 504-byte rows, g = 2).  Thread q of a group owns the group's float4 number q at every group it visits, so the four
// (row offset, feature) positions it writes are fixed for the whole kernel and their v' columns live in registers.
// A persistent grid walks chunks of up to kEgChunkRows consecutive rows (chunks may straddle graphs): the chunk's
// per-row coefficients dz'[b][h][j][i] are gathered once into shared memory, then every float4 of the chunk is
// H fused multiply-adds per element and one 16-byte streaming store.
#include "attn_common.cuh"

namespace spotv2 {

constexpr int kEgThreads = 512;        // >= the largest group (Fe = 511: 511 float4) so one pass covers any group
constexpr int kEgChunkRows = 1024;     // coefficient staging: 1024 rows x 8 heads x 4 B = 32 KB of shared memory

struct EgArgs {
  const float* dz;          // [B][H][N][ns] (ns = kEdgeTermNS for N <= 32, N above)
  const int32_t* table;     // [R]
  const float* v;           // [H][Fe]
  float* out;               // [B*R][Fe]
  long long total;          // B*R*Fe floats
  long long rows;           // B*R
  long long nchunks;
  int N, Fe, R, ns;
  int g;                    // rows per group
  int slots;                // float4 per group: g*Fe/4
  int gpp;                  // groups one pass of the block covers
  int chunk_rows;           // rows per chunk (multiple of g)
};

template <int H>
__global__ void __launch_bounds__(kEgThreads, 2) edge_rows_grad_kernel(const EgArgs a) {
  extern __shared__ float4 coef_s[];                   // [chunk_rows][2]: dz' of the row for heads 0..3 | 4..7
  constexpr int kV4 = H > 4 ? 2 : 1;
  const int tid = threadIdx.x;
  const int q = tid % a.slots, gi = tid / a.slots;
  const bool active = gi < a.gpp;
  // the four positions this thread writes inside every group: row offset rk (0 .. g-1) and feature column
  int rk[4];
  float vr[4][H];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int e = 4 * q + k;
    rk[k] = e / a.Fe;
    const int f = e - rk[k] * a.Fe;
#pragma unroll
    for (int h = 0; h < H; ++h) vr[k][h] = active ? __ldg(a.v + h * a.Fe + f) : 0.f;
  }
  const size_t graph_floats = (size_t)H * a.N * a.ns;
  for (long long c = blockIdx.x; c < a.nchunks; c += gridDim.x) {
    const long long row0 = c * a.chunk_rows;
    const int rows = (int)min((long long)a.chunk_rows, a.rows - row0);
    // ---- coefficients of the chunk's rows (gathered through L1: a graph's dz' tile is read from DRAM once)
    for (int r = tid; r < rows; r += kEgThreads) {
      const long long gr = row0 + r;
      const long long b = gr / a.R;
      const int code = __ldg(a.table + (int)(gr - b * a.R));
      float cv[8];
#pragma unroll
      for (int h = 0; h < 8; ++h) cv[h] = 0.f;
      if (code >= 0) {
        const float* src = a.dz + (size_t)b * graph_floats + (size_t)(code & 0xffff) * a.ns + (code >> 16);
#pragma unroll
        for (int h = 0; h < H; ++h) cv[h] = __ldg(src + (size_t)h * a.N * a.ns);
      }
      coef_s[kV4 * r] = make_float4(cv[0], cv[1], cv[2], cv[3]);
      if (kV4 == 2) coef_s[kV4 * r + 1] = make_float4(cv[4], cv[5], cv[6], cv[7]);
    }
    __syncthreads();
    // ---- the chunk's rows: H FMAs per element, one 16-byte store per thread and group
    if (active) {
      const int ngroups = (rows + a.g - 1) / a.g;
      for (int G = gi; G < ngroups; G += a.gpp) {
        const int rbase = G * a.g;
        const long long e0 = (row0 + rbase) * a.Fe + 4 * q;
        float o[4];
        float cf[8];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if (k == 0 || rk[k] != rk[k - 1]) {            // a float4 spans at most g rows: reload on a row change only
            const float4 c0 = coef_s[kV4 * (rbase + rk[k])];
            cf[0] = c0.x; cf[1] = c0.y; cf[2] = c0.z; cf[3] = c0.w;
            if (kV4 == 2) {
              const float4 c1 = coef_s[kV4 * (rbase + rk[k]) + 1];
              cf[4] = c1.x; cf[5] = c1.y; cf[6] = c1.z; cf[7] = c1.w;
            }
          }
          float s = 0.f;
#pragma unroll
          for (int h = 0; h < H; ++h) s = fmaf(cf[h], vr[k][h], s);
          o[k] = s;
        }
        if (e0 + 4 <= a.total) {
          __stcs(reinterpret_cast<float4*>(a.out + e0), make_float4(o[0], o[1], o[2], o[3]));
        } else {                                          // the array's last group when B*R is not a multiple of g
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (e0 + k < a.total) a.out[e0 + k] = o[k];
        }
      }
    }
    __syncthreads();
  }
}

template <int H>
int launch_edge_rows_grad(const EgArgs& a, cudaStream_t st) {
  const size_t smem = (size_t)a.chunk_rows * (H > 4 ? 2 : 1) * sizeof(float4);
  long long grid = 2LL * sm_count();
  if (grid > a.nchunks) grid = a.nchunks;
  edge_rows_grad_kernel<H><<<(unsigned)grid, kEgThreads, smem, st>>>(a);
  SPOTV2_CUDA_OK(cudaGetLastError());
  return SPOTV2_OK;
}

}  // namespace spotv2

using namespace spotv2;

extern "C" int spotv2_gat_edge_rows_grad(const spotv2_gat_desc* d, const float* d_edge_terms, const int32_t* table,
                                         const float* v, float* d_edge_rows, void* stream) {
  if (int rc = check_desc(d)) return rc;
  SPOTV2_REQUIRE(d_edge_terms && table && v && d_edge_rows,
                 "edge_rows_grad: d_edge_terms, table, v and d_edge_rows must be non-null");
  SPOTV2_REQUIRE(d->Fe > 0, "edge_rows_grad: the layer has no edge features (Fe = 0)");
  SPOTV2_REQUIRE(aligned16(d_edge_rows), "edge_rows_grad: d_edge_rows must be 16-byte aligned");
  if (d->H > kMaxHeads) return fail(SPOTV2_ERR_UNSUPPORTED, "H=%d > %d", d->H, kMaxHeads);
  if (d->Fe > kMaxFe) return fail(SPOTV2_ERR_UNSUPPORTED, "Fe=%d > %d", d->Fe, kMaxFe);
  EgArgs a;
  a.dz = d_edge_terms; a.table = table; a.v = v; a.out = d_edge_rows;
  a.N = d->N; a.Fe = d->Fe; a.R = d->R;
  a.ns = d->N > 32 ? d->N : kEdgeTermNS;
  a.rows = (long long)d->B * d->R;
  a.total = a.rows * d->Fe;
  a.g = (d->Fe % 4 == 0) ? 1 : (d->Fe % 2 == 0) ? 2 : 4;
  a.slots = a.g * d->Fe / 4;
  a.gpp = kEgThreads / a.slots;
  if (a.gpp > kEgChunkRows / a.g) a.gpp = kEgChunkRows / a.g;
  a.chunk_rows = (kEgChunkRows / a.g) / a.gpp * a.gpp * a.g;
  a.nchunks = (a.rows + a.chunk_rows - 1) / a.chunk_rows;
  cudaStream_t st = as_stream(stream);
  switch (d->H) {
    case 1: return launch_edge_rows_grad<1>(a, st);
    case 2: return launch_edge_rows_grad<2>(a, st);
    case 3: return launch_edge_rows_grad<3>(a, st);
    case 4: return launch_edge_rows_grad<4>(a, st);
    case 5: return launch_edge_rows_grad<5>(a, st);
    case 6: return launch_edge_rows_grad<6>(a, st);
    case 7: return launch_edge_rows_grad<7>(a, st);
    default: return launch_edge_rows_grad<8>(a, st);
  }
}
