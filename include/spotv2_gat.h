/*
 * spotv2_gat.h — C ABI of libspotv2_gat.so, the B200 (sm_100a) replacement for
 * the GAT hot path of loopinf/SpotV2Net.
 *
 * What it replaces.  The reference has no native code; its hot path is the
 * third-party PyG 2.3.0 `GATConv` reached from
 *     /root/reference/utils/models.py:11      (import)
 *     /root/reference/utils/models.py:87-113  (layer construction)
 *     /root/reference/utils/models.py:146     (x = l(x, edge_index, edge_attr))
 *     /root/reference/5_train_SpotV2Net.py:150-159 (forward + autograd backward)
 * and the PyG batch collation reached from
 *     /root/reference/5_train_SpotV2Net.py:90,142-143.
 * Each entry point below names the eager op(s) it stands in for.  The binding
 * a maintainer adds on the reference side is a ctypes stub; see INTEGRATION.md.
 *
 * Conventions.
 *  - extern "C", plain pointers and sizes; no torch / ATen types.
 *  - every pointer is a DEVICE pointer owned by the caller unless it says host.
 *    The library allocates nothing persistent and keeps no global state.
 *  - every entry point enqueues work on `stream` (a cudaStream_t passed as
 *    void*) and returns without synchronising; it is safe to capture into a
 *    CUDA graph.
 *  - return value: SPOTV2_OK (0) or a spotv2_status; a human-readable message
 *    for the calling thread's last failure is at spotv2_last_error().
 *  - all inputs, outputs and parameters are IEEE fp32; row-major; leading dimensions in elements.
 *    The only other format is the tensor-core GEMM operand ("fp16 pair", see spotv2_split_f16), an
 *    internal representation that resolves 22 significand bits and never leaves the library's buffers.
 *  - batches are B identical complete directed graphs on N nodes (the only
 *    topology /root/reference/utils/dataset.py:216-226 produces).  Anything
 *    else is rejected by spotv2_edge_table_build — there is no generic or CPU
 *    fallback.
 */
#ifndef SPOTV2_GAT_H_
#define SPOTV2_GAT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPOTV2_ABI_VERSION 5

typedef enum spotv2_status {
  SPOTV2_OK = 0,
  SPOTV2_ERR_INVALID_ARG = 1,   /* null pointer, non-positive size, bad stride/alignment */
  SPOTV2_ERR_UNSUPPORTED = 2,   /* shape outside what the kernels cover (e.g. H > 8, Fe > 512) */
  SPOTV2_ERR_WORKSPACE = 3,     /* workspace too small */
  SPOTV2_ERR_CUDA = 4,          /* a CUDA runtime call failed */
  SPOTV2_ERR_NO_DEVICE = 5      /* no sm_100 device / driver */
} spotv2_status;

/* One GATConv layer applied to one batch.
 * PyG ctor kwargs used by the reference (utils/models.py:87-113):
 *   in_channels=F, out_channels=C, heads=H, concat, edge_dim=Fe, negative_slope. */
typedef struct spotv2_gat_desc {
  int32_t B;              /* graphs in the batch                                   */
  int32_t N;              /* nodes per graph (30 by default).  N <= 32: one CTA per
                             graph, everything fused in shared memory; N > 32 (the
                             500-node universe): several CTAs per graph, attention
                             tile [B,H,N,N] in the workspace                       */
  int32_t F;              /* in_channels                                           */
  int32_t Fe;             /* edge_dim; 0 = layer called with edge_attr=None        */
  int32_t H;              /* heads                                                 */
  int32_t C;              /* out_channels per head                                 */
  int32_t R;              /* edge rows per graph in the edge block (N*(N-1) for
                             PyG order, N*N for a dense target-major tile)         */
  int32_t concat;         /* 1: out is [B*N, H*C]; 0: head mean, out is [B*N, C]   */
  float   negative_slope; /* LeakyReLU slope                                       */
  int32_t ldp;            /* row stride of P_aug / dP_aug: >= H*C + 2*H, % 4 == 0  */
  int32_t gemm_algo;      /* 0 | 2 tcgen05, fp32-accurate (fp16 operand pairs, 3 products); 1 fp32 CUDA
                             cores; 3 tcgen05 half-precision class (one fp16 product, fp32
                             accumulate: BASELINE config C's "bf16" variant, error ~1e-3)       */
  int32_t attn_bwd_algo;  /* 0 auto (pipelined mma.sync kernel when its shared-memory plan fits, else phase-serial),
                             1 phase-serial kernel, 2 pipelined mma.sync or error, 3 tcgen05/TMEM kernel or error
                             (head-mean layers, N <= 31; opt-in: measured slower than 2 on B200)        */
  float   dropout_p;      /* attention dropout of this call: 0 = none (eval mode, or PyG's
                             dropout=0.0 default, config/GNN_param.yaml:36).  In (0,1): every
                             attention coefficient is zeroed with probability p and the rest
                             scaled by 1/(1-p) AFTER the softmax (F.dropout(alpha) in [PyG]
                             gat_conv.py message); attn_bwd regenerates the same mask            */
  int32_t edge_mode;      /* 0: edge features arrive as rows (edge_rows [B, R, Fe]); the default and the reference
                             contract.  1: structured source - the caller computed the edge terms itself
                             (spotv2_edge_terms_from_windows) and passes them as edge_terms; edge_rows and table are
                             ignored, and attn_bwd returns d(edge terms) instead of dv                          */
  uint32_t dropout_seed_lo, dropout_seed_hi;   /* Philox4x32-10 key of the mask; element (b,h,i,j)
                             uses counter ((((b*H+h)*N+i)*N+j) >> 2), lane (.. & 3); pass
                             the same key to attn_fwd and attn_bwd of one step              */
  int32_t p_format;       /* how the projection travels between proj_fwd and the attention kernels, and dP back:
                             0: fp32 P_aug [B*N, ldp] (the contract above; every kernel covers it).
                             1: "pair" - P never exists in fp32: the projection GEMM's epilogue emits the fp16 operand
                                pair (hi, lo planes [B*N, ld16(n_aug)], n_aug = H*Cp + 2H, head pitch Cp = C rounded up
                                to 8 so that every (head, channel block) tile starts on a 16-byte boundary for TMA) with
                                a power-of-two scale per column group taken from an a-priori bound
                                |P| <= max|x| * max_j ||W_aug[j,:]||_1, and the attention kernels feed the planes to
                                the tensor cores without converting anything.  W_aug, dW_aug and the dP pair use the
                                same padded row / column layout (pad rows of W_aug are zero).  N <= 32, tensor-core
                                GEMM only (gemm_algo 0 | 2 | 3); with gemm_algo 3 only the hi planes exist (fp16
                                storage of P and dP: BASELINE config C's reduced-precision variant).
                             Use the *_pair entry points below with p_format 1.                                  */
} spotv2_gat_desc;

/* Row table entry: (i << 16) | j  = "this edge row is j -> i" (i target, j source),
 * or SPOTV2_ROW_SKIP for rows the layer ignores (self loops in the input, which
 * PyG's remove_self_loops drops; the diagonal of a dense tile). */
#define SPOTV2_ROW_SKIP (-1)

const char* spotv2_last_error(void);
int32_t     spotv2_abi_version(void);

/* Smallest legal ldp for (H, C). */
int32_t spotv2_gat_ldp(int32_t H, int32_t C);
/* Rows of W_aug / dW_aug and columns of the P / dP pair planes for this descriptor: H*Cp + 2H with the head pitch
 * Cp = C (p_format 0) or C rounded up to 8 (p_format 1); head h's channel c sits at h*Cp + c, s_h at H*Cp + h,
 * d_h at H*Cp + H + h. */
int32_t spotv2_gat_n_aug(const spotv2_gat_desc* d);
/* 1 when the p_format 1 kernels cover this problem (N <= 32, tensor-core GEMM, pipelined backward, C % 4 == 0 - % 8 for
 * concat layers -, C <= 1024, and the shared-memory plans of both attention kernels fit), else 0: use p_format 0.
 * The descriptor's own p_format field is ignored.  Host-side, no device work. */
int spotv2_gat_pair_format_supported(const spotv2_gat_desc* d);
int32_t spotv2_gat_head_pitch(const spotv2_gat_desc* d);

/* Bytes of scratch each phase wants (device memory, 256-byte aligned). */
int spotv2_gat_workspace_bytes(const spotv2_gat_desc* d, size_t* proj_fwd, size_t* attn_bwd,
                               size_t* proj_bwd);
/* Scratch of spotv2_gat_attn_fwd: 0 for N <= 32; the [B, H, N, N] fp32 attention tile for larger graphs
 * (not needed when the caller passes alpha_or_null, which then doubles as the tile). */
int spotv2_gat_attn_fwd_workspace_bytes(const spotv2_gat_desc* d, size_t* attn_fwd);
/* Size of the optional edge-term buffer g[b][h][j][i] = <e_ij, v_h> (6 floats per edge instead of Fe): when the
 * caller hands one to spotv2_gat_attn_fwd, the forward fills it, and spotv2_gat_attn_bwd given the same buffer skips
 * its first pass over the edge rows (it still recomputes the softmax; the rows are read once, for dv).  0 when the
 * layer has no edge features.  Layout is the kernels' own ([H][N][36] floats per graph for N <= 32, [H][N][N] above). */
int spotv2_gat_edge_terms_bytes(const spotv2_gat_desc* d, size_t* bytes);

/* Replaces the per-call topology work PyG does on edge_index
 * (remove_self_loops / add_self_loops / index_select by edge_index[0|1];
 * [PyG] gat_conv.py forward, utils/loop.py).  Reads edge_index [2, B*R] int64
 * (PyG concatenated order, node ids offset by b*N), writes table[R] and
 * status[4] = {ok, first bad edge, reason, 0}.  ok==1 iff every graph repeats
 * graph 0's local pattern and that pattern holds each ordered pair i!=j once. */
int spotv2_edge_table_build(const int64_t* edge_index, int64_t num_edges, int32_t B, int32_t N,
                            int32_t R, int32_t* table, int32_t* status, void* stream);
/* Table of a dense target-major tile: row r = i*N + j, diagonal skipped. */
int spotv2_edge_table_dense(int32_t N, int32_t* table, void* stream);

/* Folds the attention vectors into the linear maps (SURVEY.md §0.6):
 *   W_aug [n_aug, F] = [ W ; u_src ; u_dst ],  u_src,h = W_h^T a_src,h   (n_aug = spotv2_gat_n_aug(d): H*C + 2H, or with
 *                        p_format 1 every head's C rows followed by Cp - C zero rows, Cp = spotv2_gat_head_pitch(d))
 *   v     [H, Fe]       = W_e,h^T a_edge,h            (skipped when Fe == 0)
 * Stands in for `(x_src * att_src).sum(-1)`, `(x_dst * att_dst).sum(-1)` and
 * `lin_edge(edge_attr)` + `(e * att_edge).sum(-1)` of [PyG] gat_conv.py. */
int spotv2_gat_fold(const spotv2_gat_desc* d, const float* W, const float* a_src,
                    const float* a_dst, const float* W_e, const float* a_edge, float* W_aug,
                    float* v, void* stream);

/* 1 when the projection GEMMs of this descriptor run on the tensor cores (tcgen05 kind::f16 on fp16
 * operand pairs), 0 when they take the exact-fp32 CUDA-core kernel (gemm_algo == 1). */
int spotv2_gat_uses_tensor_cores(const spotv2_gat_desc* d);

/* Leading dimension (elements) of an fp16-pair array holding `cols` columns: cols rounded up to 16, so that
 * every row starts on a 32-byte sector (the kernels themselves only need ld16 % 8 == 0). */
int32_t spotv2_gat_ld16(int32_t cols);

/* Tensor-core operand preparation ("fp16 pair").  src [rows, cols] fp32 (row pitch ld) becomes
 *   hi = fp16(src * s),  lo = fp16(src * s - hi)        both [rows, ld16] fp16, ld16 % 8 == 0,
 * with s a power of two per group that maps the group's largest magnitude into [2^14, 2^15)
 * (hi + lo == src * s to 2^-22; removing s is exact).  Groups: index < split_at / >= split_at along
 * split_dim (0 rows, 1 cols); split_at <= 0 means one group.  scale_block (8 floats, device) receives
 * {bits of max|.| x2, inverse scales x2, scales x2, -, -}; the GEMM entry points read the inverse scales
 * from it.  Lets the caller prepare x once per step for both proj_fwd and proj_bwd_weight. */
int spotv2_split_f16(const float* src, int32_t rows, int32_t cols, int32_t ld, int32_t split_dim,
                     int32_t split_at, void* hi, void* lo, int32_t ld16, float* scale_block, void* stream);

/* lin_src: P_aug [B*N, ldp] = x [B*N, F] . W_aug^T ; columns [0,HC) are P,
 * [HC,HC+H) are s = alpha_src, [HC+H,HC+2H) are d = alpha_dst.
 * x_hi/x_lo/x_scale: optional fp16 pair of x ([B*N, ld16(F)], all three or none); otherwise x is
 * prepared inside the workspace.  p_amax_or_null (8 floats, device): [0] receives the bit pattern of
 * max |P| over the H*C projection columns, which spotv2_gat_attn_bwd uses to scale its fp16 operands. */
int spotv2_proj_fwd(const spotv2_gat_desc* d, const float* x, const void* x_hi, const void* x_lo,
                    const float* x_scale, const float* W_aug, float* P_aug, float* p_amax_or_null,
                    void* ws, size_t ws_bytes, void* stream);

/* edge_update + softmax + propagate + head reduce + bias ([PyG] gat_conv.py
 * edge_update/message, utils/softmax.py, aggr='add').  edge_rows is [B, R, Fe]
 * (ignored when Fe == 0).  alpha_or_null, if given, receives the attention
 * tile [B, H, N(source j), N(target i)] (for return_attention_weights). */
int spotv2_gat_attn_fwd(const spotv2_gat_desc* d, const float* P_aug, const float* edge_rows,
                        const int32_t* table, const float* v, const float* bias_or_null,
                        float* out, float* alpha_or_null, float* edge_terms_or_null, void* ws, size_t ws_bytes,
                        void* stream);

/* autograd of the above with the attention coefficients recomputed, not stored (edge_terms_or_null: what the
 * forward wrote, see spotv2_gat_edge_terms_bytes; null = recompute the edge terms from edge_rows as well).
 * d_edge_terms_or_null (16-byte aligned, spotv2_gat_edge_terms_bytes, the edge-term tile layout) receives dz', the
 * gradient w.r.t. the edge terms <e_ij, v_h> with the mean self-loop fill folded in (0 on the diagonal).
 * edge_mode 1: edge_terms and d_edge_terms are required and dv is left to spotv2_windows_dv.  edge_mode 0: optional;
 * dv is formed as usual, and spotv2_gat_edge_rows_grad turns d_edge_terms into the edge rows' gradient.  Null: none of
 * that work is done.
 * dout [B*N, C or HC] -> dP_aug (dP | ds | dd), dv [H, Fe], dbias.  The gradient is emitted either as
 * fp32 dP_aug [B*N, ldp] (CUDA-core GEMM path) or, when dP_hi/dP_lo/dp_scale are given, directly as the
 * fp16 pair [B*N, ld16(HC+2H)] the tensor-core GEMMs consume (two scale groups: columns < HC from a
 * bound on max|dout|, the ds|dd columns from their own maximum); dp_scale is an 8-float scale block.
 * p_amax_or_null: what spotv2_proj_fwd wrote (saves one pass over P_aug). */
int spotv2_gat_attn_bwd(const spotv2_gat_desc* d, const float* P_aug, const float* p_amax_or_null,
                        const float* edge_rows, const float* edge_terms_or_null,
                        const int32_t* table, const float* v, const float* dout, float* dP_aug_or_null,
                        void* dP_hi_or_null, void* dP_lo_or_null, float* dp_scale_or_null,
                        float* dv_or_null, float* d_edge_terms_or_null, float* dbias_or_null, void* ws, size_t ws_bytes,
                        void* stream);

/* spotv2_gat_attn_bwd with the gradient through the attention coefficients the forward returned: d_alpha [B, H, N(source j),
 * N(target i)] fp32 (the layout of alpha_or_null; spotv2_alpha_to_pyg_grad makes it from a PyG-order gradient) is dL/d(alpha m/(1-p)),
 * the coefficients after attention dropout (m = keep mask; m = 1 without dropout).  It joins dalpha = g dO P^T (g = 1/H for the
 * head mean, 1 for concat) before the dropout factor: dalpha_ij = m_ij/(1-p) (<g dO_i, P_j> + d_alpha_ij); everything after
 * that (softmax, LeakyReLU, ds | dd, dz', dv, d_edge_terms) follows unchanged.  d_alpha is required; the preconditions and the
 * other arguments are those of spotv2_gat_attn_bwd. */
int spotv2_gat_attn_bwd_dalpha(const spotv2_gat_desc* d, const float* P_aug, const float* p_amax_or_null,
                               const float* edge_rows, const float* edge_terms_or_null,
                               const int32_t* table, const float* v, const float* dout, float* dP_aug_or_null,
                               void* dP_hi_or_null, void* dP_lo_or_null, float* dp_scale_or_null,
                               float* dv_or_null, float* d_edge_terms_or_null, float* dbias_or_null, void* ws, size_t ws_bytes,
                               void* stream, const float* d_alpha);

/* Gradient w.r.t. the edge rows (edge_mode 0): d_edge_rows [B, R, Fe] in PyG row order,
 *   d_edge_rows[b*R + r, :] = sum_h d_edge_terms[b][h][j][i] * v[h, :]   for table[r] = (i << 16) | j,
 *   d_edge_rows[b*R + r, :] = 0                                           for SPOTV2_ROW_SKIP rows,
 * from what spotv2_gat_attn_bwd / _attn_bwd_pair wrote to d_edge_terms_or_null, the row table and the folded edge
 * vector v [H, Fe] the forward used (spotv2_gat_fold's output, after any per-feature scaling the caller applied).
 * Stands in for the autograd of `lin_edge(edge_attr)` + `(e * att_edge).sum(-1)`, of the mean self-loop fill
 * (add_self_loops(fill_value='mean')) and of remove_self_loops in [PyG] gat_conv.py.  d_edge_rows is 16-byte aligned;
 * H <= 8, Fe <= 512; any N and row pitch. */
int spotv2_gat_edge_rows_grad(const spotv2_gat_desc* d, const float* d_edge_terms, const int32_t* table, const float* v,
                              float* d_edge_rows, void* stream);

/* ---- p_format 1: the projection as an fp16 operand pair end to end ---------------------------------------------
 * Same operators as spotv2_proj_fwd / spotv2_gat_attn_fwd / spotv2_gat_attn_bwd ([PyG] F.linear, edge_update,
 * softmax, propagate and their autograd), different intermediate: P_hi / P_lo are [B*N, ld16(n_aug)] fp16 planes
 * (P_lo may be null with gemm_algo 3), p_scale an 8-float scale block ({bound bits x2, inverse scales x2, scales x2}:
 * group 0 the H*Cp projection columns, group 1 the s|d columns) written by proj_fwd_pair and read by the other two;
 * sd [B*N, 2H] fp32 receives the logit terms s | d as the GEMM accumulated them (the attention kernels read these, not the
 * planes' s|d columns: the LeakyReLU kinks of the logits must not depend on the pair's 22-bit rounding).
 * x must be given as a pair (x_hi, x_lo, x_scale; spotv2_split_f16 or spotv2_collate_windows_pair): the bound needs
 * max|x|, which the scale block holds.  W_aug is spotv2_gat_fold's output for the same descriptor ([n_aug, F]).
 * attn_bwd_pair emits dP as the pair [B*N, ld16(n_aug)] in the padded layout (pad columns zero), consumed by
 * spotv2_proj_bwd_weight / spotv2_proj_bwd_input with the same descriptor.
 * edge_terms between attn_fwd_pair and attn_bwd_pair is an OPAQUE record of the forward for the backward of the same step
 * (same descriptor, same buffer, spotv2_gat_edge_terms_bytes): without attention dropout the forward leaves its attention
 * coefficients there (same tile layout; LeakyReLU side in the sign bit), so the backward redoes neither logits nor softmax;
 * with dropout_p > 0 it leaves the edge terms.  edge_mode 1: the forward overwrites the edge terms it was given. */
int spotv2_proj_fwd_pair(const spotv2_gat_desc* d, const void* x_hi, const void* x_lo, const float* x_scale,
                         const float* W_aug, void* P_hi, void* P_lo_or_null, float* p_scale, float* sd, void* ws,
                         size_t ws_bytes, void* stream);
int spotv2_gat_attn_fwd_pair(const spotv2_gat_desc* d, const void* P_hi, const void* P_lo_or_null, const float* p_scale,
                             const float* sd, const float* edge_rows, const int32_t* table, const float* v, const float* bias_or_null,
                             float* out, float* alpha_or_null, float* edge_terms_or_null, void* stream);
int spotv2_gat_attn_bwd_pair(const spotv2_gat_desc* d, const void* P_hi, const void* P_lo_or_null, const float* p_scale,
                             const float* sd, const float* edge_rows, const float* edge_terms_or_null, const int32_t* table,
                             const float* v, const float* dout, void* dP_hi, void* dP_lo_or_null, float* dp_scale,
                             float* dv_or_null, float* d_edge_terms_or_null, float* dbias_or_null, void* ws,
                             size_t ws_bytes, void* stream);
/* spotv2_gat_attn_bwd_pair with the gradient through the returned coefficients, as spotv2_gat_attn_bwd_dalpha. */
int spotv2_gat_attn_bwd_pair_dalpha(const spotv2_gat_desc* d, const void* P_hi, const void* P_lo_or_null, const float* p_scale,
                                    const float* sd, const float* edge_rows, const float* edge_terms_or_null, const int32_t* table,
                                    const float* v, const float* dout, void* dP_hi, void* dP_lo_or_null, float* dp_scale,
                                    float* dv_or_null, float* d_edge_terms_or_null, float* dbias_or_null, void* ws,
                                    size_t ws_bytes, void* stream, const float* d_alpha);

/* ---- structured edge source (SURVEY.md 8f-2; csrc/windows.cu) ---------------------------------------------------
 * In the reference's dataset (utils/dataset.py:228-242) edge_attr is a pure function of the window of co-volatility
 * matrices: edge (j -> i), feature k*L + t = vv[t0+t][min][max] | vv[t0+t][j][j] | vv[t0+t][i][i] for k = 0 | 1 | 2.
 * These two calls replace the passes over the materialised [B*N*(N-1), 3L] rows by passes over the [L, N, N] windows
 * (2.9x fewer bytes, 3x fewer multiply-adds); use them with desc.edge_mode = 1:
 *   edge_terms_from_windows -> attn_fwd(edge_terms) ... attn_bwd(edge_terms, d_edge_terms_out) -> windows_dv -> dv.
 * M_vv [T, N, N] fp32 on the device, t0 [B] int32 window starts, v [H, 3L] from spotv2_gat_fold. */
int spotv2_edge_terms_from_windows_workspace_bytes(const spotv2_gat_desc* d, size_t* bytes);   /* 0 for N <= 32 */
int spotv2_edge_terms_from_windows(const spotv2_gat_desc* d, const float* M_vv, int32_t T, int32_t L,
                                   const int32_t* t0, const float* v, float* edge_terms, void* ws, size_t ws_bytes,
                                   void* stream);
int spotv2_windows_dv_workspace_bytes(const spotv2_gat_desc* d, size_t* bytes);
int spotv2_windows_dv(const spotv2_gat_desc* d, const float* M_vv, int32_t T, int32_t L, const int32_t* t0,
                      const float* d_edge_terms, float* dv, void* ws, size_t ws_bytes, void* stream);

/* lin_src backward: dW_aug [n_aug, F] = dP_aug^T . x  and  dX [B*N, F] = dP_aug . W_aug  (p_format 1: dP as the pair in the
 * padded layout, required; x as a pair for the weight gradient).
 * x and dP_aug are taken as fp16 pairs when given (hi, lo, scale block: all three), else as fp32 and
 * prepared inside the workspace. */
int spotv2_proj_bwd_weight(const spotv2_gat_desc* d, const float* x, const void* x_hi, const void* x_lo,
                           const float* x_scale, const float* dP_aug, const void* dP_hi, const void* dP_lo,
                           const float* dp_scale, float* dW_aug, void* ws, size_t ws_bytes, void* stream);
int spotv2_proj_bwd_input(const spotv2_gat_desc* d, const float* dP_aug, const void* dP_hi, const void* dP_lo,
                          const float* dp_scale, const float* W_aug, float* dX, void* ws, size_t ws_bytes,
                          void* stream);

/* Inverse of spotv2_gat_fold for gradients: from dW_aug and dv to the gradients of
 * lin_src.weight, att_src, att_dst, lin_edge.weight, att_edge (PyG parameter names). */
int spotv2_gat_unfold(const spotv2_gat_desc* d, const float* W, const float* a_src,
                      const float* a_dst, const float* W_e, const float* a_edge,
                      const float* dW_aug, const float* dv, float* dW, float* da_src,
                      float* da_dst, float* dW_e, float* da_edge, void* stream);

/* return_attention_weights ordering (SURVEY.md App. A.4): real edges in batch
 * order, then the B*N self loops: alpha_pyg [B*R_real + B*N, H]. */
int spotv2_alpha_to_pyg(const spotv2_gat_desc* d, const float* alpha_tile, const int32_t* table,
                        float* alpha_pyg, void* stream);
/* Its inverse for gradients: d_alpha_pyg [B*R + B*N, H] (same order) -> d_alpha_tile [B, H, N(j), N(i)], the d_alpha input of
 * the _dalpha backward entry points.  Real-edge rows go through the table, loop rows give the diagonal, SPOTV2_ROW_SKIP rows
 * (input self loops, absent from what PyG returns) are ignored.  With the table of a complete graph every tile entry is
 * written exactly once: the output needs no clearing. */
int spotv2_alpha_to_pyg_grad(const spotv2_gat_desc* d, const float* d_alpha_pyg, const int32_t* table,
                             float* d_alpha_tile, void* stream);

/* Graph-batch collation on the device (replaces PyG DataLoader/Batch.from_data_list
 * over CovarianceLaggedDataset, /root/reference/utils/dataset.py:182-289 and
 * 5_train_SpotV2Net.py:90,142-143).  M_vol, M_vv: [T, N, N] fp32 resident in HBM;
 * t0[B] int32 window starts; L = seq_length.  Writes x [B*N, N*L],
 * edge_attr [B*N*(N-1), 3L] in PyG row order (null: not materialised, see the structured edge source below), y [B*N]. */
int spotv2_collate_windows(const float* M_vol, const float* M_vv, int32_t T, int32_t N, int32_t L,
                           const int32_t* t0, int32_t B, float* x, float* edge_attr, float* y,
                           void* stream);

/* Collation that also emits x as the tensor-core operand pair (see spotv2_split_f16), so that the training step holds
 * neither an amax pass nor a split pass over x (619 MB per 4096-graph batch).  x values are entries of M_vol, hence the
 * pair's power-of-two scale is a property of the dataset: spotv2_stack_scale fills an 8-float scale block from
 * max |M_vol| once (count = T*N*N), and every batch collated from that stack shares it.  x_or_null: also write the fp32
 * x [B*N, N*L] (the reference layout, utils/dataset.py:250,278); x_hi / x_lo: [B*N, ld16] fp16, ld16 = spotv2_gat_ld16(N*L).
 * Pass (x_hi, x_lo, x_scale) to spotv2_proj_fwd / spotv2_proj_bwd_weight as their x operand. */
int spotv2_stack_scale(const float* M, int64_t count, float* scale_block, void* stream);
int spotv2_collate_windows_pair(const float* M_vol, const float* M_vv, int32_t T, int32_t N, int32_t L,
                                const int32_t* t0, int32_t B, float* x_or_null, void* x_hi, void* x_lo, int32_t ld16,
                                const float* x_scale, float* edge_attr, float* y, void* stream);

/* ---- diagnostics (bring-up and parity tests of the GEMM back ends; not reference-facing) ----
 * C[M,N] (ld ldc) = sum_k A(m,k) B(n,k).  a_kc/b_kc = 1: operand stored [rows, K] (K contiguous),
 * 0: stored [K, rows].  algo 1 = exact-fp32 CUDA-core kernel, 2 = tcgen05 3xTF32 kernel (the first
 * tensor-core version, kept as a yardstick), 3 = tcgen05 fp16-pair kernel (the production path);
 * operands are split inside ws.  bn = 128|256 tile width (+16: half-depth k-blocks, deeper ring),
 * kb_per_chunk = k-blocks per TMEM accumulation chain (0 = 128 elements), splits = split-K factor. */
int spotv2_diag_gemm(int a_kc, int b_kc, int M, int N, int K, const float* A, int lda, const float* B,
                     int ldb, float* C, int ldc, int algo, int splits, int bn, int kb_per_chunk,
                     void* ws, size_t ws_bytes, void* stream);

/* The operand preparation spotv2_gat_attn_bwd_pair runs on dout (csrc/attn_prep.cu), exposed for the parity tests:
 * dout [B*N, upg*C] fp32 -> hi | lo [B*N, ld16] fp16 with one power-of-two scale per unit (upg = 1: a graph; upg = H: a
 * (graph, head) block of a concat layer), scales [B*upg], scale_block[0] = bit pattern of max|dout|, dbias [upg*C] column
 * sums (null: skipped).  ws: at least spotv2_diag_dout_pair_ws_bytes(B, C, upg) bytes. */
size_t spotv2_diag_dout_pair_ws_bytes(int32_t B, int32_t C, int32_t upg);
int spotv2_diag_dout_pair(const float* dout, int32_t B, int32_t N, int32_t C, int32_t upg, void* hi, void* lo_or_null,
                          int32_t ld16, float* scales, float* scale_block, float* dbias_or_null, void* ws, void* stream);

/* Copies (and optionally resets) 32 device-side cycle counters.  [0,16): forward kernel, cycles one
 * sampling thread per role spent parked on the edge ring, alpha-tile empty/full, P-tile full/empty, then
 * per-role loop totals.  [16,32): backward kernel, cycles per phase (logits, softmax, dalpha GEMM,
 * softmax backward, dP, dv) summed over CTAs.  host_out: 32 x uint64 on the host; synchronises the device.
 * Profiling aid only. */
int spotv2_diag_counters(unsigned long long* host_out, int reset);

/* Split-K factor spotv2_gat_proj_bwd_weight uses for dW_aug[m, n] = sum over `rows` (host-side rule, no kernel launch):
 * ceil(rows / 8192) clamped to [1, 32], then raised by up to a quarter so that (256 x 256 pair tiles) x splits fills
 * the last wave of the GEMM's resident CTA pairs (an occupancy query; 74 on a B200, sm_count / 2 without a device).
 * spotv2_gat_workspace_bytes sizes the partial buffers with the same rule. */
int32_t spotv2_diag_weight_grad_splits(int32_t rows, int32_t m, int32_t n);

#ifdef __cplusplus
}
#endif
#endif /* SPOTV2_GAT_H_ */
