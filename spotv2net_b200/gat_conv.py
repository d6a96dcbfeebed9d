"""Drop-in ``GATConv`` for batches of identical complete graphs, backed by libspotv2_gat.so.

Constructor kwargs, ``forward(x, edge_index, edge_attr=None, size=None,
return_attention_weights=None)``, parameter names and init follow PyG 2.3.0
``torch_geometric.nn.GATConv`` as the reference uses it
(/root/reference/utils/models.py:11,87-113,146; 6_results.ipynb:213), so
``state_dict`` files saved by the reference (5_train_SpotV2Net.py:195) load
unchanged.  All arithmetic runs in the hand-written sm_100a kernels; there is
no eager or CPU path.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import weakref
from dataclasses import dataclass
from typing import Optional

import torch
from torch import Tensor, nn

from . import _lib
from ._lib import GatDesc, SpotV2Error, check, ptr, stream_ptr


# --------------------------------------------------------------------------- topology
@dataclass
class WindowSource:
    """Structured edge source (SURVEY.md 8f-2): the [T, N, N] co-volatility stack the reference's dataset builds
    edge_attr from (utils/dataset.py:228-242) plus each graph's window start.  A layer given this reads the windows
    (151 KB per graph at the default geometry) instead of the materialised edge rows (438 KB)."""
    volvol: Tensor         # [T, N, N] fp32 on the device
    t0: Tensor             # [B] int32 on the device
    L: int                 # seq_length; edge_dim must be 3 * L
    checked: bool = False  # t0 + L <= T already verified (WindowDataset.collate checks on the host)
    # [T, 4] float64 per-matrix sums (upper triangle: sum, sum of squares; diagonal: sum, sum of squares), kept by the
    # dataset: the batch statistics of edge_attr (standardize=True) follow from them without touching an edge
    mat_stats: Optional[Tensor] = None

    def edge_stats(self):
        """(sum, sum of squares, count) per edge feature over the batch's B*N*(N-1) real edges, float64 [3L] each.
        Feature k*L + t (utils/dataset.py:228-242): k = 0 the pair's co-volatility - every upper-triangle entry of matrix
        t0 + t twice (once per direction); k = 1 / 2 the source / target variance - every diagonal entry N - 1 times."""
        N, L = self.volvol.shape[1], self.L
        idx = self.t0.long().view(-1, 1) + torch.arange(L, device=self.t0.device).view(1, L)
        m = self.mat_stats[idx].sum(0)                                   # [L, 4]
        se = torch.cat([2.0 * m[:, 0], (N - 1.0) * m[:, 2], (N - 1.0) * m[:, 2]])
        qe = torch.cat([2.0 * m[:, 1], (N - 1.0) * m[:, 3], (N - 1.0) * m[:, 3]])
        return se, qe, float(self.t0.numel() * N * (N - 1))


@dataclass
class Topology:
    """What the kernels need to know about ``edge_index``: B graphs of N nodes,
    R edge rows per graph, and the row table (row -> target/source)."""
    B: int
    N: int
    R: int
    table: Tensor          # int32 [R] on the device
    has_skips: bool        # some rows are self loops (dropped by PyG's remove_self_loops)


_TOPO_CACHE: dict = {}
_REASONS = {1: "node id outside [0, N) in the first graph",
            2: "a graph's edge pattern differs from the first graph's",
            3: "an ordered pair i != j is missing or duplicated (graph is not complete)"}


def _try_topology(edge_index: Tensor, n_nodes: int, N: int) -> Optional[Topology]:
    E = edge_index.shape[1]
    if N <= 0 or n_nodes % N:
        return None
    B = n_nodes // N
    if B <= 0 or E % B:
        return None
    R = E // B
    if R < N * (N - 1):
        return None
    lib = _lib.load()
    dev = edge_index.device
    table = torch.empty(R, dtype=torch.int32, device=dev)
    status = torch.empty(4 + N * N, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        check(lib.spotv2_edge_table_build(ptr(edge_index), E, B, N, R, ptr(table), ptr(status), stream_ptr(dev)),
              "spotv2_edge_table_build")
    ok, where, reason = status[:3].tolist()              # one sync per new topology
    if not ok:
        _try_topology.last_failure = f"{_REASONS.get(reason, reason)} (first offending index {where})"
        return None
    return Topology(B, N, R, table, bool((table < 0).any().item()))


_try_topology.last_failure = ""


def topology_from_edge_index(edge_index: Tensor, n_nodes: int, nodes_per_graph: Optional[int] = None) -> Topology:
    """Validate ``edge_index`` [2, E] (PyG concatenated order) as B identical
    complete graphs and build the row table.  Cached per tensor identity."""
    if edge_index.dim() != 2 or edge_index.shape[0] != 2 or edge_index.dtype != torch.int64:
        raise SpotV2Error("edge_index must be an int64 tensor of shape [2, E]")
    _lib.require_cuda(edge_index, "edge_index")
    # Cached per tensor OBJECT (weak reference), never per address: the caching allocator hands the same
    # address to unrelated tensors, and a stale hit would silently mis-route edges.
    key = id(edge_index)
    hit = _TOPO_CACHE.get(key)
    if hit is not None:
        ref, version, args, topo = hit
        if ref() is edge_index and version == edge_index._version and args == (n_nodes, nodes_per_graph):
            return topo
        del _TOPO_CACHE[key]
    owner = edge_index
    edge_index = edge_index.contiguous()
    E = edge_index.shape[1]
    cands = [nodes_per_graph] if nodes_per_graph else []
    if not cands and n_nodes > 0 and E % n_nodes == 0:
        cands = [E // n_nodes + 1, E // n_nodes]          # without / with self loops in the input
    topo = None
    for N in cands:
        topo = _try_topology(edge_index, n_nodes, int(N))
        if topo is not None:
            break
    if topo is None:
        raise SpotV2Error(
            "edge_index is not a batch of identical complete directed graphs "
            f"(n_nodes={n_nodes}, E={E}; {_try_topology.last_failure or 'sizes do not factor'}). "
            "Sparse / irregular graphs (CovarianceSparseDataset) are outside this library's scope; "
            "there is no generic fallback.")
    if len(_TOPO_CACHE) > 64:
        _TOPO_CACHE.clear()
    _TOPO_CACHE[key] = (weakref.ref(owner), owner._version, (n_nodes, nodes_per_graph), topo)
    return topo


# --------------------------------------------------------------------------- autograd
# Kernel selection knobs of spotv2_gat_desc (0 = the library's choice); tests set them to run every back end.
GEMM_ALGO = 0
ATTN_BWD_ALGO = 0
# How the projection travels between the GEMM and the attention kernels (spotv2_gat_desc.p_format): None = the library's
# choice (the fp16 operand pair whenever the shapes allow it), 0 = always fp32 P_aug, 1 = the pair or an error.
P_FORMAT = None if os.environ.get("SPOTV2_P_FORMAT") is None else int(os.environ["SPOTV2_P_FORMAT"])      # A/B switch
_KEEP = None      # tools/ set this to a dict to receive the backward's dP (bring-up aid)


PRECISIONS = {"fp32": None, "half": 3}      # "half": single fp16 tensor-core product in the projections (config C)


def pair_format_applies(N: int, Fe: int, Cc: int, gemm_algo: int, attn_bwd_algo: int, concat: bool = False) -> bool:
    """Shapes the p_format 1 kernels cover: one CTA per graph, tensor-core GEMM, the pipelined backward, head blocks of dout
    that one CTA of the prepass holds in registers and whose tiles start on 16-byte boundaries."""
    return (N <= 32 and gemm_algo != 1 and Cc % 4 == 0 and Cc <= 1024 and Fe <= 384 and attn_bwd_algo in (0, 2)
            and (not concat or Cc % 8 == 0))


def _desc(topo: Topology, F_in: int, Fe: int, H: int, Cc: int, concat: bool, slope: float,
          dropout_p: float = 0.0, seed: int = 0, gemm_algo: Optional[int] = None, edge_mode: int = 0,
          p_format: Optional[int] = None) -> GatDesc:
    lib = _lib.load()
    algo = GEMM_ALGO if gemm_algo is None else gemm_algo
    if p_format is None:
        p_format = P_FORMAT
    d = GatDesc(topo.B, topo.N, F_in, Fe, H, Cc, topo.R, int(concat), float(slope),
                lib.spotv2_gat_ldp(H, Cc), algo, ATTN_BWD_ALGO,
                float(dropout_p), int(edge_mode), seed & 0xffffffff, (seed >> 32) & 0xffffffff, 0)
    if p_format is None:      # the library's own answer (shape rules AND the kernels' shared-memory plans); else p_format 0
        p_format = 1 if (pair_format_applies(topo.N, Fe, Cc, algo, ATTN_BWD_ALGO, bool(concat))
                         and lib.spotv2_gat_pair_format_supported(C.byref(d))) else 0
    d.p_format = int(p_format)
    return d


def _workspace(desc: GatDesc):
    lib = _lib.load()
    a, b, c = C.c_size_t(), C.c_size_t(), C.c_size_t()
    check(lib.spotv2_gat_workspace_bytes(C.byref(desc), C.byref(a), C.byref(b), C.byref(c)), "workspace_bytes")
    return a.value, b.value, c.value


def _edge_terms_bytes(desc: GatDesc) -> int:
    a = C.c_size_t()
    check(_lib.load().spotv2_gat_edge_terms_bytes(C.byref(desc), C.byref(a)), "edge_terms_bytes")
    return a.value


def _attn_fwd_workspace(desc: GatDesc) -> int:
    a = C.c_size_t()
    check(_lib.load().spotv2_gat_attn_fwd_workspace_bytes(C.byref(desc), C.byref(a)), "attn_fwd_workspace_bytes")
    return a.value


class _GatLayerFn(torch.autograd.Function):
    """fold -> projection GEMM -> fused attention, and the recompute-based backward."""

    @staticmethod
    def forward(ctx, x, edge_attr, W, a_src, a_dst, W_e, a_edge, bias, topo, H, Cc, concat, slope, want_alpha,
                dropout_p=0.0, seed=0, gemm_algo=None, windows=None, x_pair=None, edge_scale=None, edge_mean=None):
        with torch.cuda.device(x.device):        # launches, attribute calls and tensor maps go to the CURRENT device
            return _GatLayerFn._forward(ctx, x, edge_attr, W, a_src, a_dst, W_e, a_edge, bias, topo, H, Cc, concat, slope,
                                        want_alpha, dropout_p, seed, gemm_algo, windows, x_pair, edge_scale, edge_mean)

    @staticmethod
    def _forward(ctx, x, edge_attr, W, a_src, a_dst, W_e, a_edge, bias, topo, H, Cc, concat, slope, want_alpha,
                 dropout_p, seed, gemm_algo, windows, x_pair, edge_scale, edge_mean):
        lib = _lib.load()
        dev = x.device
        st = stream_ptr(dev)
        Fe = 0 if edge_attr is None or W_e is None else edge_attr.shape[1]
        if windows is not None:                     # structured edge source: the edge rows are never touched
            Fe, edge_attr = 3 * windows.L, None
        # the descriptor (incl. this step's dropout key) is kept for the backward, which regenerates the same mask
        # (standardize=True shifts the d columns of an fp32 P_aug: that path keeps p_format 0)
        desc = _desc(topo, x.shape[1], Fe, H, Cc, concat, slope, dropout_p, seed, gemm_algo, 1 if windows is not None else 0,
                     0 if (edge_mean is not None and Fe) else None)
        pair = desc.p_format == 1
        n, HC = x.shape[0], H * Cc
        n_aug = lib.spotv2_gat_n_aug(C.byref(desc))
        x = x.contiguous()
        ea = edge_attr.contiguous() if (Fe and windows is None) else None
        # every tensor whose address is handed to the library is held in a local until the call returns
        W, a_src, a_dst = W.contiguous(), a_src.contiguous(), a_dst.contiguous()
        W_e = W_e.contiguous() if W_e is not None else None
        a_edge = a_edge.contiguous() if a_edge is not None else None
        bias_c = bias.contiguous() if bias is not None else None
        W_aug = torch.empty(n_aug, x.shape[1], device=dev, dtype=torch.float32)
        v = torch.empty(H, Fe, device=dev, dtype=torch.float32) if Fe else None
        check(lib.spotv2_gat_fold(C.byref(desc), ptr(W), ptr(a_src), ptr(a_dst), ptr(W_e) if Fe else None,
                                  ptr(a_edge) if Fe else None, ptr(W_aug), ptr(v), st), "spotv2_gat_fold")
        if Fe and edge_scale is not None:
            # per-feature scale of the edge features (BatchNorm1d(affine=False) of the model's standardize=True): its
            # 1/sqrt(var + eps) rides on v; its mean is a per-head constant -<mean, v'> INSIDE the LeakyReLU, added to the
            # target term d after the projection (below)
            v.mul_(edge_scale.view(1, Fe))
        ws_f, _, _ = _workspace(desc)
        ws = torch.empty(ws_f, device=dev, dtype=torch.uint8)
        p_amax = torch.empty(8, device=dev, dtype=torch.float32)      # max|P|, sizes the backward's fp16 operand scale
        if pair:     # P as the GEMM-written fp16 operand pair (hi | lo planes; hi only in the half-precision class); p_amax = its scale block
            P_aug = torch.empty(1 if desc.gemm_algo == 3 else 2, n, lib.spotv2_gat_ld16(n_aug), device=dev, dtype=torch.float16)
        else:
            P_aug = torch.empty(n, desc.ldp, device=dev, dtype=torch.float32)
        # tensor-core path: x becomes an fp16 operand pair once; the weight-gradient GEMM reuses it
        x16 = x_blk = None
        if lib.spotv2_gat_uses_tensor_cores(C.byref(desc)) and x_pair is not None:
            x16, x_blk = x_pair                    # emitted by the collation (WindowDataset): no amax / split pass over x
        elif lib.spotv2_gat_uses_tensor_cores(C.byref(desc)):
            ld16 = lib.spotv2_gat_ld16(x.shape[1])
            x16 = torch.empty(2, n, ld16, device=dev, dtype=torch.float16)
            x_blk = torch.empty(8, device=dev, dtype=torch.float32)
            check(lib.spotv2_split_f16(ptr(x), n, x.shape[1], x.shape[1], 0, 0, ptr(x16[0]), ptr(x16[1]), ld16,
                                       ptr(x_blk), st), "spotv2_split_f16")
        sd32 = torch.empty(n, 2 * H, device=dev, dtype=torch.float32) if pair else None      # the logit terms s | d in fp32
        if pair:
            check(lib.spotv2_proj_fwd_pair(C.byref(desc), ptr(x16[0]), ptr(x16[1]), ptr(x_blk), ptr(W_aug), ptr(P_aug[0]),
                                           ptr(P_aug[1]) if P_aug.shape[0] > 1 else None, ptr(p_amax), ptr(sd32), ptr(ws), ws_f, st),
                  "spotv2_proj_fwd_pair")
        else:
            check(lib.spotv2_proj_fwd(C.byref(desc), ptr(x), ptr(x16[0]) if x16 is not None else None,
                                      ptr(x16[1]) if x16 is not None else None, ptr(x_blk), ptr(W_aug), ptr(P_aug), ptr(p_amax),
                                      ptr(ws), ws_f, st), "spotv2_proj_fwd")
        if Fe and edge_scale is not None and edge_mean is not None:
            # <e_hat, v> = <e, v'> - <mean, v'>: the same shift on every logit of the head, self loop included (its fill is the
            # mean of the real edges' e_hat) - carried by the d columns of P_aug, which both attention kernels read
            P_aug[:, HC + H:HC + 2 * H].sub_((v @ edge_mean.view(Fe, 1)).view(1, H))
        out = torch.empty(n, HC if concat else Cc, device=dev, dtype=torch.float32)
        alpha = torch.empty(topo.B, H, topo.N, topo.N, device=dev, dtype=torch.float32) if want_alpha else None
        # N > 32 only: the [B,H,N,N] attention tile lives in a workspace unless the caller asked for alpha itself
        ws_t = _attn_fwd_workspace(desc) if alpha is None else 0
        ws_attn = torch.empty(ws_t, device=dev, dtype=torch.uint8) if ws_t else None
        # the forward keeps the edge terms <e_ij, v_h> (6 floats per edge) when a backward will follow: the backward
        # then reads the Fe-wide edge rows once (for dv) instead of twice
        et = None
        if Fe and (windows is not None or any(ctx.needs_input_grad)):
            et = torch.empty(_edge_terms_bytes(desc) // 4, device=dev, dtype=torch.float32)
        if windows is not None:
            wsz = C.c_size_t()
            check(lib.spotv2_edge_terms_from_windows_workspace_bytes(C.byref(desc), C.byref(wsz)), "edge_terms_from_windows ws")
            ws_w = torch.empty(wsz.value, device=dev, dtype=torch.uint8) if wsz.value else None
            check(lib.spotv2_edge_terms_from_windows(C.byref(desc), ptr(windows.volvol), windows.volvol.shape[0], windows.L,
                                                     ptr(windows.t0), ptr(v), ptr(et), ptr(ws_w), wsz.value, st),
                  "spotv2_edge_terms_from_windows")
        tbl = ptr(topo.table) if (Fe and windows is None) else None
        if pair:
            check(lib.spotv2_gat_attn_fwd_pair(C.byref(desc), ptr(P_aug[0]), ptr(P_aug[1]) if P_aug.shape[0] > 1 else None, ptr(p_amax),
                                               ptr(sd32), ptr(ea), tbl, ptr(v), ptr(bias_c), ptr(out), ptr(alpha), ptr(et), st),
                  "spotv2_gat_attn_fwd_pair")
        else:
            check(lib.spotv2_gat_attn_fwd(C.byref(desc), ptr(P_aug), ptr(ea), tbl, ptr(v),
                                          ptr(bias_c), ptr(out), ptr(alpha), ptr(et), ptr(ws_attn), ws_t, st), "spotv2_gat_attn_fwd")
        ctx.desc, ctx.topo, ctx.Fe, ctx.has_bias, ctx.windows = desc, topo, Fe, bias is not None, windows
        ctx.edge_scale = edge_scale if Fe else None
        ctx.edge_mean = edge_mean if (Fe and edge_scale is not None) else None
        ctx.save_for_backward(x, ea, W, a_src, a_dst, W_e, a_edge, W_aug, v, P_aug, x16, x_blk, p_amax, et, sd32)
        ctx.out_shape, ctx.device = out.shape, dev
        if want_alpha:
            # alpha (after attention dropout) is differentiable, as in PyG: a loss on it reaches every input through the
            # attention backward's d_alpha term.  Unused outputs arrive as None in the backward, not as zeros.
            ctx.set_materialize_grads(False)
            return out, alpha
        return out, None

    @staticmethod
    def backward(ctx, dout, dalpha=None):
        with torch.cuda.device(ctx.device):
            return _GatLayerFn._backward(ctx, dout, dalpha)

    @staticmethod
    def _backward(ctx, dout, dalpha=None):
        lib = _lib.load()
        x, ea, W, a_src, a_dst, W_e, a_edge, W_aug, v, P_aug, x16, x_blk, p_amax, et, sd32 = ctx.saved_tensors
        desc, topo, Fe = ctx.desc, ctx.topo, ctx.Fe
        # d edge_attr: the attention backward hands out dz' (gradient w.r.t. the edge terms), expanded below into rows
        want_dea = bool(ctx.needs_input_grad[1]) and ea is not None
        dev = x.device
        st = stream_ptr(dev)
        H, Cc = desc.H, desc.C
        HC = H * Cc
        # a loss on alpha alone: out received no gradient
        dout = torch.zeros(ctx.out_shape, device=dev, dtype=torch.float32) if dout is None else dout.contiguous()
        # dalpha: [B, H, N, N] gradient w.r.t. the returned coefficients, the _dalpha entry points' extra input
        if dalpha is not None:
            dalpha = dalpha.to(torch.float32).contiguous()
        _, ws_a, ws_p = _workspace(desc)
        ws = torch.empty(max(ws_a, ws_p), device=dev, dtype=torch.uint8)
        # on the tensor-core path the attention backward emits dP directly as the GEMMs' fp16 operand pair
        tc = bool(lib.spotv2_gat_uses_tensor_cores(C.byref(desc)))
        pair = desc.p_format == 1
        dP_aug = dP16 = dp_blk = None
        if pair:
            dP16 = torch.empty_like(P_aug)          # same planes, same padded head pitch
            dp_blk = torch.empty(8, device=dev, dtype=torch.float32)
        elif tc:
            dP16 = torch.empty(2, P_aug.shape[0], lib.spotv2_gat_ld16(HC + 2 * H), device=dev, dtype=torch.float16)
            dp_blk = torch.empty(8, device=dev, dtype=torch.float32)
        else:
            dP_aug = torch.empty_like(P_aug)
        ph, pl = (dP16[0], dP16[1] if dP16.shape[0] > 1 else None) if tc else (None, None)
        dv = torch.empty(H, Fe, device=dev, dtype=torch.float32) if Fe else None
        dbias = torch.empty(dout.shape[1], device=dev, dtype=torch.float32) if ctx.has_bias else None
        win = ctx.windows
        # d(edge terms) out: structured source (dv from the windows), or edge_attr.grad wanted (dv as usual)
        d_et = torch.empty_like(et) if (win is not None or want_dea) else None
        if pair:
            args = (C.byref(desc), ptr(P_aug[0]), ptr(P_aug[1]) if P_aug.shape[0] > 1 else None, ptr(p_amax),
                    ptr(sd32), ptr(ea), ptr(et), ptr(topo.table) if (Fe and win is None) else None, ptr(v),
                    ptr(dout), ptr(ph), ptr(pl), ptr(dp_blk), ptr(dv) if win is None else None,
                    ptr(d_et), ptr(dbias), ptr(ws), ws.numel(), st)
            if dalpha is None:
                check(lib.spotv2_gat_attn_bwd_pair(*args), "spotv2_gat_attn_bwd_pair")
            else:
                check(lib.spotv2_gat_attn_bwd_pair_dalpha(*args, ptr(dalpha)), "spotv2_gat_attn_bwd_pair_dalpha")
        else:
            args = (C.byref(desc), ptr(P_aug), ptr(p_amax), ptr(ea), ptr(et),
                    ptr(topo.table) if (Fe and win is None) else None, ptr(v),
                    ptr(dout), ptr(dP_aug), ptr(ph), ptr(pl), ptr(dp_blk), ptr(dv) if win is None else None,
                    ptr(d_et), ptr(dbias), ptr(ws), ws.numel(), st)
            if dalpha is None:
                check(lib.spotv2_gat_attn_bwd(*args), "spotv2_gat_attn_bwd")
            else:
                check(lib.spotv2_gat_attn_bwd_dalpha(*args, ptr(dalpha)), "spotv2_gat_attn_bwd_dalpha")
        if win is not None:
            wsz = C.c_size_t()
            check(lib.spotv2_windows_dv_workspace_bytes(C.byref(desc), C.byref(wsz)), "windows_dv_workspace_bytes")
            ws_dv = torch.empty(wsz.value, device=dev, dtype=torch.uint8)
            check(lib.spotv2_windows_dv(C.byref(desc), ptr(win.volvol), win.volvol.shape[0], win.L, ptr(win.t0), ptr(d_et),
                                        ptr(dv), ptr(ws_dv), wsz.value, st), "spotv2_windows_dv")
        d_ea = None
        if want_dea:
            # d edge_attr[e, :] = sum_h dz'[e, h] v'_h (v' = the folded, scaled edge vector the forward used); input self
            # loops (rows PyG's remove_self_loops drops) get zero rows
            d_ea = torch.empty_like(ea)
            check(lib.spotv2_gat_edge_rows_grad(C.byref(desc), ptr(d_et), ptr(topo.table), ptr(v), ptr(d_ea), st),
                  "spotv2_gat_edge_rows_grad")
        d_scale = d_mean = None
        if ctx.edge_scale is not None:
            # the layer saw e_hat = (e - mean) * scale through v' = scale * v and the per-head logit shift -<mean, v'> on the
            # d columns.  d/dv = scale * (sum dz' e - mean * sum of ALL dz of the head): the kernels formed the first sum (dv),
            # the second is the column sum of the dd block (LeakyReLU keeps a softmax row's dz from summing to zero).
            T = None
            if ctx.edge_mean is not None:            # (p_format 0 by construction: see _forward)
                if tc:
                    T = ((dP16[0][:, HC + H:HC + 2 * H].float() + dP16[1][:, HC + H:HC + 2 * H].float()).sum(0) * dp_blk[3])
                else:
                    T = dP_aug[:, HC + H:HC + 2 * H].sum(0)
                dv.sub_(T.view(H, 1) * ctx.edge_mean.view(1, Fe))
            # batch statistics that depend on edge_attr (training mode with edge_attr.requires_grad): with g_h = dv here,
            # dL/dscale = sum_h v_h * g_h (v unscaled) and dL/dmean = -sum_h T_h v'_h
            if ctx.needs_input_grad[19]:
                d_scale = (v * dv).sum(0) / ctx.edge_scale
            if ctx.needs_input_grad[20] and T is not None:
                d_mean = -(T.view(H, 1) * v).sum(0)
            dv.mul_(ctx.edge_scale.view(1, Fe))
        if _KEEP is not None:                      # bring-up aid (tools/): the kernel-level gradient of the projection
            _KEEP.update(dP16=dP16, dp_blk=dp_blk, dP_aug=dP_aug, n_aug=lib.spotv2_gat_n_aug(C.byref(desc)),
                         head_pitch=lib.spotv2_gat_head_pitch(C.byref(desc)))
        dW_aug = torch.empty_like(W_aug)
        xh = x16[0] if x16 is not None else None
        xl = x16[1] if x16 is not None else None
        check(lib.spotv2_proj_bwd_weight(C.byref(desc), ptr(x), ptr(xh), ptr(xl), ptr(x_blk), ptr(dP_aug), ptr(ph),
                                         ptr(pl), ptr(dp_blk), ptr(dW_aug), ptr(ws), ws.numel(), st),
              "spotv2_proj_bwd_weight")
        dx = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            check(lib.spotv2_proj_bwd_input(C.byref(desc), ptr(dP_aug), ptr(ph), ptr(pl), ptr(dp_blk), ptr(W_aug),
                                            ptr(dx), ptr(ws), ws.numel(), st), "spotv2_proj_bwd_input")
        dW = torch.empty_like(W)
        da_src = torch.empty_like(a_src)
        da_dst = torch.empty_like(a_dst)
        dW_e = torch.empty_like(W_e) if Fe else None
        da_edge = torch.empty_like(a_edge) if Fe else None
        check(lib.spotv2_gat_unfold(C.byref(desc), ptr(W), ptr(a_src), ptr(a_dst), ptr(W_e) if Fe else None,
                                    ptr(a_edge) if Fe else None, ptr(dW_aug), ptr(dv), ptr(dW), ptr(da_src),
                                    ptr(da_dst), ptr(dW_e), ptr(da_edge), st), "spotv2_gat_unfold")
        if not Fe and W_e is not None:          # layer has lin_edge but was called with edge_attr=None
            dW_e, da_edge = torch.zeros_like(W_e), torch.zeros_like(a_edge)
        return (dx, d_ea, dW, da_src, da_dst, dW_e, da_edge, dbias) + (None,) * 11 + (d_scale, d_mean)


class _AlphaToPyg(torch.autograd.Function):
    """Attention tile [B, H, N, N] -> PyG order [B*R + B*N, H] (input self-loop rows zero), and back for the gradient."""

    @staticmethod
    def forward(ctx, alpha_tile, topo, desc):
        lib = _lib.load()
        dev = alpha_tile.device
        ctx.topo, ctx.desc = topo, desc
        alpha = torch.empty(topo.B * topo.R + topo.B * topo.N, desc.H, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            check(lib.spotv2_alpha_to_pyg(C.byref(desc), ptr(alpha_tile), ptr(topo.table), ptr(alpha), stream_ptr(dev)),
                  "spotv2_alpha_to_pyg")
        return alpha

    @staticmethod
    def backward(ctx, g):
        lib = _lib.load()
        topo, desc = ctx.topo, ctx.desc
        g = g.to(torch.float32).contiguous()
        dev = g.device
        # every tile entry is written once (the table of a complete graph): no zero fill
        d_tile = torch.empty(topo.B, desc.H, topo.N, topo.N, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            check(lib.spotv2_alpha_to_pyg_grad(C.byref(desc), ptr(g), ptr(topo.table), ptr(d_tile), stream_ptr(dev)),
                  "spotv2_alpha_to_pyg_grad")
        return d_tile, None, None


# --------------------------------------------------------------------------- module
def _glorot_(t: Tensor) -> Tensor:
    bound = math.sqrt(6.0 / (t.size(-2) + t.size(-1)))
    with torch.no_grad():
        return t.uniform_(-bound, bound)


class _Linear(nn.Module):
    """Weight holder named like PyG's ``Linear(bias=False, weight_initializer='glorot')``."""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.weight = nn.Parameter(torch.empty(out_channels, in_channels))
        self.reset_parameters()

    def reset_parameters(self):
        _glorot_(self.weight)

    def extra_repr(self):
        return f"{self.in_channels}, {self.out_channels}, bias=False"


class GATConv(nn.Module):
    """``GATConv(in_channels, out_channels, heads=1, concat=True, negative_slope=0.2,
    dropout=0.0, add_self_loops=True, edge_dim=None, fill_value='mean', bias=True)``.

    State-dict keys: ``att_src, att_dst, att_edge, bias, lin_src.weight,
    lin_dst.weight`` (alias of lin_src, as in PyG 2.3.0), ``lin_edge.weight``.
    """

    def __init__(self, in_channels: int, out_channels: int, heads: int = 1, concat: bool = True,
                 negative_slope: float = 0.2, dropout: float = 0.0, add_self_loops: bool = True,
                 edge_dim: Optional[int] = None, fill_value="mean", bias: bool = True, **kwargs):
        super().__init__()
        if not isinstance(in_channels, int):
            raise SpotV2Error("bipartite (tuple) in_channels are outside this library's scope")
        if not add_self_loops or fill_value != "mean":
            raise SpotV2Error("only add_self_loops=True with fill_value='mean' (the PyG defaults the "
                              "reference relies on) is implemented")
        self.in_channels, self.out_channels, self.heads = in_channels, out_channels, heads
        self.concat, self.negative_slope, self.dropout = concat, negative_slope, dropout
        self.add_self_loops, self.edge_dim, self.fill_value = add_self_loops, edge_dim, fill_value
        self.lin_src = _Linear(in_channels, heads * out_channels)
        self.lin_dst = self.lin_src
        self.att_src = nn.Parameter(torch.empty(1, heads, out_channels))
        self.att_dst = nn.Parameter(torch.empty(1, heads, out_channels))
        if edge_dim is not None:
            self.lin_edge = _Linear(edge_dim, heads * out_channels)
            self.att_edge = nn.Parameter(torch.empty(1, heads, out_channels))
        else:
            self.lin_edge = None
            self.register_parameter("att_edge", None)
        if bias:
            self.bias = nn.Parameter(torch.empty(heads * out_channels if concat else out_channels))
        else:
            self.register_parameter("bias", None)
        self.nodes_per_graph: Optional[int] = None     # optional hint; inferred from edge_index otherwise
        # "fp32" (default): every product fp32-accurate (1e-5 parity).  "half": the projection GEMMs issue one fp16
        # tensor-core product with fp32 accumulation (BASELINE config C's reduced-precision variant, ~1e-3).  With the pair
        # format (p_format 1) P, alpha, dout and dP also travel as single fp16 planes through the attention kernels; with
        # p_format 0 the attention kernels stay fp32-accurate and the GEMMs read the fp16 hi plane of dP (DESIGN §6).  Not a PyG ctor
        # argument: set the attribute.
        self.precision = "fp32"
        self.reset_parameters()

    def reset_parameters(self):
        # same RNG draw order as PyG 2.3.0 (SURVEY.md App. A.5)
        self.lin_src.reset_parameters()
        self.lin_dst.reset_parameters()
        if self.lin_edge is not None:
            self.lin_edge.reset_parameters()
        _glorot_(self.att_src)
        _glorot_(self.att_dst)
        if self.att_edge is not None:
            _glorot_(self.att_edge)
        if self.bias is not None:
            with torch.no_grad():
                self.bias.zero_()

    def _load_from_state_dict(self, state_dict, prefix, *args, **kwargs):
        # PyG >= 2.5 checkpoints name the shared projection `lin.weight`
        if prefix + "lin.weight" in state_dict and prefix + "lin_src.weight" not in state_dict:
            w = state_dict.pop(prefix + "lin.weight")
            state_dict[prefix + "lin_src.weight"] = w
            state_dict[prefix + "lin_dst.weight"] = w
        super()._load_from_state_dict(state_dict, prefix, *args, **kwargs)

    def forward(self, x: Tensor, edge_index, edge_attr: Optional[Tensor] = None, size=None,
                return_attention_weights=None, topology: Optional[Topology] = None,
                windows: Optional[WindowSource] = None, edge_scale: Optional[Tensor] = None,
                edge_mean: Optional[Tensor] = None):
        assert x.dim() == 2, "Static graphs not supported in 'GATConv'"
        _lib.require_cuda(x, "x")
        # attention dropout (dropout_att; 0.0 by default, config/GNN_param.yaml:36): a fresh 64-bit Philox key per
        # call from torch's CPU generator (so torch.manual_seed reproduces a run); the kernels derive the mask from it
        drop_p, seed = 0.0, 0
        if self.dropout > 0.0 and self.training:
            if not self.dropout < 1.0:
                raise SpotV2Error("dropout must be in [0, 1)")
            drop_p = float(self.dropout)
            seed = int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).item())
        if edge_attr is not None:
            _lib.require_cuda(edge_attr, "edge_attr")
            if edge_attr.dim() == 1:
                edge_attr = edge_attr.view(-1, 1)
        topo = topology or topology_from_edge_index(edge_index, x.shape[0], self.nodes_per_graph)
        # a caller-supplied topology / window source is checked against this call's tensors: a Topology built for
        # another batch size would make the kernels read and write past x / out
        if x.shape[0] != topo.B * topo.N:
            raise SpotV2Error(f"topology describes {topo.B} graphs of {topo.N} nodes, x has {x.shape[0]} rows")
        if torch.is_tensor(edge_index) and edge_index.dim() == 2 and edge_index.shape[1] != topo.B * topo.R:
            raise SpotV2Error(f"topology describes {topo.B * topo.R} edges, edge_index has {edge_index.shape[1]}")
        if windows is not None:
            if edge_attr is not None:
                windows = None          # a materialised edge_attr always wins (the caller may have edited it)
            elif windows.volvol.dim() != 3 or windows.volvol.shape[1] != topo.N or windows.volvol.shape[2] != topo.N:
                raise SpotV2Error("windows.volvol must be [T, N, N] with this batch's N")
            elif int(windows.t0.numel()) == topo.B and not windows.checked:
                t_hi = int(windows.t0.max().item()) + windows.L          # once per WindowSource (one sync)
                if int(windows.t0.min().item()) < 0 or t_hi > windows.volvol.shape[0]:
                    raise SpotV2Error(f"window [t0, t0 + L) reaches {t_hi} past the {windows.volvol.shape[0]} matrices")
                windows.checked = True
        # structured edge source (batches of spotv2net_b200.WindowDataset): usable when this layer's edge_dim is the
        # dataset's 3L on graphs the fused kernels cover; otherwise the materialised edge_attr is required
        had_windows = windows is not None
        small = topo.N <= 32            # the fused small-graph kernels take the structured source on the pipelined backward only
        if windows is not None and not (self.lin_edge is not None and self.edge_dim == 3 * windows.L and
                                        topo.R == topo.N * (topo.N - 1) and not topo.has_skips and
                                        (not small or ATTN_BWD_ALGO != 1) and windows.t0.numel() == topo.B):
            windows = None
        if had_windows and windows is None and edge_attr is None and self.lin_edge is not None:
            raise SpotV2Error("this batch carries window references instead of a materialised edge_attr, and this layer "
                              "cannot use them (edge_dim != 3 * seq_length, irregular edge order, ...): "
                              "collate with structured=False")
        use_edge = (edge_attr is not None or windows is not None) and self.lin_edge is not None
        if use_edge and windows is None and edge_attr.shape[0] != topo.B * topo.R:
            raise SpotV2Error(f"edge_attr has {edge_attr.shape[0]} rows, edge_index has {topo.B * topo.R} edges")
        want_alpha = isinstance(return_attention_weights, bool)
        # x as the GEMMs' fp16 operand pair, if the collation attached one to this very tensor and nobody wrote to it since
        x_pair = None
        tag = getattr(x, "_spot_pair", None)
        if tag is not None and tag[2] == x._version and tag[0].device == x.device and tag[0].shape[1] == x.shape[0] and \
                tag[0].shape[2] == _lib.load().spotv2_gat_ld16(x.shape[1]):
            x_pair = (tag[0], tag[1])
        out, alpha_tile = _GatLayerFn.apply(
            x, edge_attr if (use_edge and windows is None) else None, self.lin_src.weight, self.att_src, self.att_dst,
            self.lin_edge.weight if self.lin_edge is not None else None, self.att_edge, self.bias,
            topo, self.heads, self.out_channels, self.concat, self.negative_slope, want_alpha, drop_p, seed,
            PRECISIONS[self.precision], windows if use_edge else None, x_pair, edge_scale if use_edge else None,
            edge_mean if use_edge else None)
        if not want_alpha:
            return out
        return out, self._attention_weights(alpha_tile, topo, edge_index)

    def _attention_weights(self, alpha_tile: Tensor, topo: Topology, edge_index: Tensor):
        """(edge_index with self loops appended, alpha [E', H]) in PyG order (App. A.4); alpha carries gradient."""
        lib = _lib.load()
        dev = alpha_tile.device
        H = self.heads
        desc = GatDesc(topo.B, topo.N, self.in_channels, 0, H, self.out_channels, topo.R, int(self.concat),
                       float(self.negative_slope), lib.spotv2_gat_ldp(H, self.out_channels), 0, 0, 0.0, 0, 0, 0)
        n = topo.B * topo.N
        alpha = _AlphaToPyg.apply(alpha_tile, topo, desc)
        loops = torch.arange(n, device=dev, dtype=edge_index.dtype)
        if topo.has_skips:                               # PyG drops input self loops before appending its own
            keep = edge_index[0] != edge_index[1]
            edge_index = edge_index[:, keep]
            alpha = torch.cat([alpha[:topo.B * topo.R][keep], alpha[topo.B * topo.R:]], 0)
        return torch.cat([edge_index, torch.stack([loops, loops])], 1), alpha

    def __repr__(self):
        return f"{self.__class__.__name__}({self.in_channels}, {self.out_channels}, heads={self.heads})"
