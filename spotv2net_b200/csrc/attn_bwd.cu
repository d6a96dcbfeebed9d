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

// The kernel without and with the gradient through the returned coefficients (spotv2_gat_attn_bwd_dalpha)
#define SPOTV2_KERNEL_NAME gat_attn_bwd_kernel
#define SPOTV2_GA 0
#include "attn_bwd_kernel.cuh"
#undef SPOTV2_KERNEL_NAME
#undef SPOTV2_GA
#define SPOTV2_KERNEL_NAME gat_attn_bwd_dalpha_kernel
#define SPOTV2_GA 1
#include "attn_bwd_kernel.cuh"
#undef SPOTV2_KERNEL_NAME
#undef SPOTV2_GA

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
static int launch_bwd(AttnBwdArgs& a, float* dv, float* dbias, void* ws, size_t ws_bytes, cudaStream_t st, const float* d_alpha) {
  const AttnParams& p = a.p;
  // largest ring stage (multiple of 16 rows) that keeps two CTAs per SM, else one
  BwdSmem sm = bwd_smem_plan(p.N, p.Fe, p.H, p.C, p.R, NPAIRS, p.concat, kBwdChunkRows);
  for (int rows = kBwdChunkRows - 16; rows >= 16 && sm.total > 113 * 1024; rows -= 16)
    sm = bwd_smem_plan(p.N, p.Fe, p.H, p.C, p.R, NPAIRS, p.concat, rows);
  if (sm.total > 227 * 1024)
    return fail(SPOTV2_ERR_UNSUPPORTED, "attn_bwd needs %zu B shared memory (> 227 KB)", sm.total);
  if (d_alpha) SPOTV2_CUDA_OK(cudaFuncSetAttribute(gat_attn_bwd_dalpha_kernel<NPAIRS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm.total));
  else SPOTV2_CUDA_OK(cudaFuncSetAttribute(gat_attn_bwd_kernel<NPAIRS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm.total));
  int grid = 2 * sm_count();
  if (grid > p.B) grid = p.B;
  const size_t need = ((size_t)grid * ((size_t)p.H * p.Fe + p.ldo)) * sizeof(float);
  if (!ws || ws_bytes < need)
    return fail(SPOTV2_ERR_WORKSPACE, "attn_bwd needs %zu B of workspace, got %zu", need, ws_bytes);
  a.dv_part = static_cast<float*>(ws);
  a.dbias_part = a.dv_part + (size_t)grid * p.H * p.Fe;
  if (d_alpha) gat_attn_bwd_dalpha_kernel<NPAIRS><<<grid, kAttnThreads, sm.total, st>>>(a, sm, d_alpha);
  else gat_attn_bwd_kernel<NPAIRS><<<grid, kAttnThreads, sm.total, st>>>(a, sm);
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

// spotv2_gat_attn_bwd and, with d_alpha, spotv2_gat_attn_bwd_dalpha
static int attn_bwd(const spotv2_gat_desc* d, const float* P_aug, const float* p_amax_or_null, const float* edge_rows,
                    const float* edge_terms_or_null, const int32_t* table, const float* v, const float* dout,
                    float* dP_aug_or_null, void* dP_hi_or_null, void* dP_lo_or_null, float* dp_scale_or_null, float* dv_or_null,
                    float* d_edge_terms_or_null, float* dbias_or_null, void* ws, size_t ws_bytes, void* stream,
                    const float* d_alpha) {
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
    return attn_large_bwd(d, a, dv_or_null, dbias_or_null, ws, ws_bytes, st, d_alpha);
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
  if (kern == BwdKernel::kTcgen05) rc = launch_attn_bwd3(a, dv, dbias_or_null, ws, ws_bytes, st, d_alpha);
  else if (kern == BwdKernel::kPipelined) rc = launch_attn_bwd2(a, dv, dbias_or_null, ws, ws_bytes, st, d_alpha);
  else if (np <= 4) rc = launch_bwd<4>(a, dv_or_null, dbias_or_null, ws, ws_bytes, st, d_alpha);
  else if (np <= 8) rc = launch_bwd<8>(a, dv_or_null, dbias_or_null, ws, ws_bytes, st, d_alpha);
  else if (np <= 15) rc = launch_bwd<15>(a, dv_or_null, dbias_or_null, ws, ws_bytes, st, d_alpha);
  else if (np <= 16) rc = launch_bwd<16>(a, dv_or_null, dbias_or_null, ws, ws_bytes, st, d_alpha);
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


extern "C" int spotv2_gat_attn_bwd(const spotv2_gat_desc* d, const float* P_aug, const float* p_amax_or_null,
                                   const float* edge_rows, const float* edge_terms_or_null, const int32_t* table,
                                   const float* v,
                                   const float* dout, float* dP_aug_or_null, void* dP_hi_or_null, void* dP_lo_or_null,
                                   float* dp_scale_or_null, float* dv_or_null, float* d_edge_terms_or_null,
                                   float* dbias_or_null, void* ws, size_t ws_bytes, void* stream) {
  return attn_bwd(d, P_aug, p_amax_or_null, edge_rows, edge_terms_or_null, table, v, dout, dP_aug_or_null, dP_hi_or_null,
                  dP_lo_or_null, dp_scale_or_null, dv_or_null, d_edge_terms_or_null, dbias_or_null, ws, ws_bytes, stream, nullptr);
}

extern "C" int spotv2_gat_attn_bwd_dalpha(const spotv2_gat_desc* d, const float* P_aug, const float* p_amax_or_null,
                                          const float* edge_rows, const float* edge_terms_or_null, const int32_t* table,
                                          const float* v, const float* dout, float* dP_aug_or_null, void* dP_hi_or_null,
                                          void* dP_lo_or_null, float* dp_scale_or_null, float* dv_or_null,
                                          float* d_edge_terms_or_null, float* dbias_or_null, void* ws, size_t ws_bytes,
                                          void* stream, const float* d_alpha) {
  if (int rc = check_desc(d)) return rc;
  SPOTV2_REQUIRE(d_alpha, "attn_bwd_dalpha: d_alpha must be non-null");
  return attn_bwd(d, P_aug, p_amax_or_null, edge_rows, edge_terms_or_null, table, v, dout, dP_aug_or_null, dP_hi_or_null,
                  dP_lo_or_null, dp_scale_or_null, dv_or_null, d_edge_terms_or_null, dbias_or_null, ws, ws_bytes, stream, d_alpha);
}

// p_format 1: same operator, P as the fp16 operand pair, dP emitted in the padded head pitch (attn_bwd2.cu, P16 instantiations)
static int attn_bwd_pair(const spotv2_gat_desc* d, const void* P_hi, const void* P_lo_or_null, const float* p_scale,
                         const float* sd, const float* edge_rows, const float* edge_terms_or_null, const int32_t* table,
                         const float* v, const float* dout, void* dP_hi, void* dP_lo_or_null, float* dp_scale,
                         float* dv_or_null, float* d_edge_terms_or_null, float* dbias_or_null, void* ws,
                         size_t ws_bytes, void* stream, const float* d_alpha) {
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
  if (int rc = launch_attn_bwd2(a, a.p.terms_in ? nullptr : dv_or_null, dbias_or_null, ws, ws_bytes, st, d_alpha)) return rc;
  return split_dsd(a, d->H * a.p.hp, st);
}

extern "C" int spotv2_gat_attn_bwd_pair(const spotv2_gat_desc* d, const void* P_hi, const void* P_lo_or_null, const float* p_scale,
                                        const float* sd, const float* edge_rows, const float* edge_terms_or_null, const int32_t* table,
                                        const float* v, const float* dout, void* dP_hi, void* dP_lo_or_null, float* dp_scale,
                                        float* dv_or_null, float* d_edge_terms_or_null, float* dbias_or_null, void* ws,
                                        size_t ws_bytes, void* stream) {
  return attn_bwd_pair(d, P_hi, P_lo_or_null, p_scale, sd, edge_rows, edge_terms_or_null, table, v, dout, dP_hi, dP_lo_or_null,
                       dp_scale, dv_or_null, d_edge_terms_or_null, dbias_or_null, ws, ws_bytes, stream, nullptr);
}

extern "C" int spotv2_gat_attn_bwd_pair_dalpha(const spotv2_gat_desc* d, const void* P_hi, const void* P_lo_or_null,
                                               const float* p_scale, const float* sd, const float* edge_rows,
                                               const float* edge_terms_or_null, const int32_t* table, const float* v,
                                               const float* dout, void* dP_hi, void* dP_lo_or_null, float* dp_scale,
                                               float* dv_or_null, float* d_edge_terms_or_null, float* dbias_or_null, void* ws,
                                               size_t ws_bytes, void* stream, const float* d_alpha) {
  if (int rc = check_desc(d)) return rc;
  SPOTV2_REQUIRE(d_alpha, "attn_bwd_pair_dalpha: d_alpha must be non-null");
  return attn_bwd_pair(d, P_hi, P_lo_or_null, p_scale, sd, edge_rows, edge_terms_or_null, table, v, dout, dP_hi, dP_lo_or_null,
                       dp_scale, dv_or_null, d_edge_terms_or_null, dbias_or_null, ws, ws_bytes, stream, d_alpha);
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
