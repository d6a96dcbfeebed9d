"""Parity of the CUDA path against the CPU oracle, through the C ABI (run on the B200 box).

Tolerance (SURVEY.md §8d / north_star): max-norm relative error
    ||ours - ref||_inf / ||ref||_inf <= 1e-5
for every output and gradient tensor, ref = the float64 edge-list oracle (PyG 2.3.0 op order).
"""
import ctypes as C
import glob
import os

import numpy as np
import pytest
import torch

import spotv2net_b200 as sv
from spotv2net_b200 import _lib
from spotv2net_b200._lib import GatDesc, check, ptr
from oracle import dense_gat, pyg_gat, synth

pytestmark = pytest.mark.gpu
TOL = 1e-5
GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz")))
DEV = "cuda:0"


def relerr(a, ref):
    a, ref = torch.as_tensor(a).double().cpu(), torch.as_tensor(ref).double().cpu()
    return ((a - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


# (test-name fragment, tensor) pairs that may pass on the "within 3x the fp32 oracle's own error" allowance instead of
# the 1e-5 bar.  Everything else must meet 1e-5 outright.  Filled from a recording run on the B200
# (SPOTV2_PARITY_RECORD=<file> logs every use instead of asserting; tools/runs/ keeps the log it was filled from).
ALLOWANCE_WHITELIST = {
    # d/d att_dst = sum over sources of softmax-gradient rows, which cancel to ~0 (a softmax row's gradient sums to
    # zero): the fp32 PyG-order oracle itself is at 1.5e-4 / 2e-5 on these cases (tools/runs/r2a_allowance.tsv)
    ("test_layer_matches_edge_list_oracle[B3N12F16Fe8H7C12mean", "g_att_dst"),
    ("test_attention_dropout_at_high_rates_with_peaked_rows", "g_att_dst"),
    ("test_golden_fixtures_on_gpu[stress_weights]", "g_att_dst"),
    ("test_model_step_matches_oracle_model[cfg1]", "gat_layers.1.att_dst"),
    # third GAT layer of the 3-layer tanh model: small, heavily cancelled attention-parameter gradients; the fp32
    # oracle is at 2e-5 .. 4.5e-5 itself (tools/runs/r2b_allowance.tsv)
    ("test_model_step_matches_oracle_model[cfg2]", "gat_layers.2.att_src"),
    ("test_model_step_matches_oracle_model[cfg2]", "gat_layers.2.att_dst"),
    ("test_model_step_matches_oracle_model[cfg2]", "gat_layers.2.att_edge"),
    ("test_model_step_matches_oracle_model[cfg2]", "gat_layers.2.lin_edge.weight"),
    ("test_scale_up_reaches_the_edge_features_on_both_batch_kinds", "gat_layers.0.att_dst"),
    # N = 2, H = 1: one real source per target, so these three gradients are identically zero in exact arithmetic and
    # the "relative error" compares rounding noise with rounding noise (ours 3e8..1e9, fp32 oracle 4e8..1.4e9)
    ("test_layer_matches_edge_list_oracle[B2N2F4Fe3H1C2cat", "g_att_dst"),
    ("test_layer_matches_edge_list_oracle[B2N2F4Fe3H1C2cat", "g_att_edge"),
    ("test_layer_matches_edge_list_oracle[B2N2F4Fe3H1C2cat", "g_lin_edge.weight"),
}
ALLOWANCE_USED = []          # (test id, tensor, our error, fp32-oracle error) of this session, for the report


def _current_test():
    return os.environ.get("PYTEST_CURRENT_TEST", "?").split(" ")[0].split("::")[-1]


def parity_failures(ours: dict, ref64: dict, ref32: dict, tol=TOL):
    """The bar: ||ours - ref64||_inf / ||ref64||_inf <= 1e-5.  Some gradients are ill-conditioned in
    fp32 whatever the implementation (d/d att_dst sums softmax-gradient rows that cancel to ~0; with
    N = 2 several gradients are identically zero): for those the PyG-order fp32 oracle itself misses
    1e-5, so a tensor ALSO passes when our error is within 3x the fp32 oracle's own error against fp64 -
    but only for the (test, tensor) pairs listed in ALLOWANCE_WHITELIST; any other use is a failure."""
    bad = {}
    test = _current_test()
    for k, r64 in ref64.items():
        e = relerr(ours[k], r64)
        if e <= tol:
            continue
        e32 = relerr(ref32[k], r64)
        if e <= 3.0 * e32:
            ALLOWANCE_USED.append((test, k, e, e32))
            rec = os.environ.get("SPOTV2_PARITY_RECORD")
            if rec:
                with open(rec, "a") as f:
                    f.write(f"{test}\t{k}\t{e:.3e}\t{e32:.3e}\n")
                continue
            if any(frag in test and k == name for frag, name in ALLOWANCE_WHITELIST):
                continue
            bad[k] = (e, e32, "used the 3x-fp32 allowance without being whitelisted")
            continue
        bad[k] = (e, e32)
    return bad


def st():
    return torch.cuda.current_stream().cuda_stream


def make_layers(Fin, C_, H, concat, Fe, slope, seed, wscale=1.0):
    torch.manual_seed(seed)
    ref = pyg_gat.OracleGATConv(Fin, C_, heads=H, concat=concat, negative_slope=slope, edge_dim=Fe).double()
    with torch.no_grad():
        for p in ref.parameters():
            p.mul_(wscale)
        ref.bias.normal_()
        for p in ref.parameters():
            p.copy_(p.float().double())
    ours = sv.GATConv(Fin, C_, heads=H, concat=concat, negative_slope=slope, edge_dim=Fe)
    ours.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
    return ref, ours.to(DEV)


def oracle_pass(ref, bt, dout, dtype, need_dx):
    import copy
    m = copy.deepcopy(ref).to(dtype)
    x = bt.x.detach().clone().to(dtype).requires_grad_(need_dx)
    out, (ei2, alpha) = m(x, bt.edge_index, bt.edge_attr.to(dtype) if bt.edge_attr is not None else None,
                          return_attention_weights=True)
    out.backward(dout.to(dtype))
    res = {"out": out.detach(), "alpha": alpha.detach()}
    for k, p in m.named_parameters():
        res["g_" + k] = p.grad
    if need_dx:
        res["g_x"] = x.grad
    return res, ei2


def run_both(ref, ours, bt, need_dx=False, seed=0):
    """Returns {tensor: (our error, fp32-oracle error)} for every tensor that misses the bar."""
    g = torch.Generator().manual_seed(seed)
    n_out = ref.heads * ref.out_channels if ref.concat else ref.out_channels
    dout = torch.randn(bt.x.shape[0], n_out, generator=g, dtype=torch.float32)
    r64, ei2 = oracle_pass(ref, bt, dout, torch.float64, need_dx)
    r32, _ = oracle_pass(ref, bt, dout, torch.float32, need_dx)
    xg = bt.x.detach().clone().to(DEV).requires_grad_(need_dx)
    out, (ei2g, alpha) = ours(xg, bt.edge_index.to(DEV), bt.edge_attr.to(DEV) if bt.edge_attr is not None else None,
                              return_attention_weights=True)
    out.backward(dout.to(DEV))
    assert torch.equal(ei2g.cpu(), ei2)
    mine = {"out": out.detach(), "alpha": alpha.detach()}
    for k, p in ours.named_parameters():
        mine["g_" + k] = p.grad
    if need_dx:
        mine["g_x"] = xg.grad
    return parity_failures(mine, r64, r32)


# ------------------------------------------------------------------ individual entry points
def test_fold_and_unfold_entry_points(cuda_lib):
    H, C_, Fin, Fe = 3, 5, 9, 4
    torch.manual_seed(0)
    W, a_s, a_d = torch.randn(H * C_, Fin), torch.randn(1, H, C_), torch.randn(1, H, C_)
    We, a_e = torch.randn(H * C_, Fe), torch.randn(1, H, C_)
    W_aug_ref, v_ref = dense_gat.fold_params(W.double(), a_s.double(), a_d.double(), We.double(), a_e.double(), H, C_)
    d = GatDesc(2, 4, Fin, Fe, H, C_, 12, 0, 0.2, cuda_lib.spotv2_gat_ldp(H, C_), 0, 0)
    g = lambda t: t.to(DEV).contiguous()
    Wg, asg, adg, Weg, aeg = map(g, (W, a_s, a_d, We, a_e))
    W_aug = torch.empty(H * C_ + 2 * H, Fin, device=DEV)
    v = torch.empty(H, Fe, device=DEV)
    check(cuda_lib.spotv2_gat_fold(C.byref(d), ptr(Wg), ptr(asg), ptr(adg), ptr(Weg), ptr(aeg), ptr(W_aug), ptr(v), st()), "fold")
    assert relerr(W_aug, W_aug_ref) < 1e-6 and relerr(v, v_ref) < 1e-6
    dW_aug, dv = torch.randn(H * C_ + 2 * H, Fin), torch.randn(H, Fe)
    ref = dense_gat.unfold_grads(dW_aug.double(), dv.double(), W.double(), a_s.double(), a_d.double(), We.double(),
                                 a_e.double(), H, C_)
    outs = [torch.empty_like(t) for t in (Wg, asg, adg, Weg, aeg)]
    dW_aug_g, dv_g = g(dW_aug), g(dv)          # keep device temporaries alive across the async call
    check(cuda_lib.spotv2_gat_unfold(C.byref(d), ptr(Wg), ptr(asg), ptr(adg), ptr(Weg), ptr(aeg), ptr(dW_aug_g),
                                     ptr(dv_g), *map(ptr, outs), st()), "unfold")
    for o, k in zip(outs, ("lin_weight", "att_src", "att_dst", "lin_edge_weight", "att_edge")):
        assert relerr(o, ref[k]) < 1e-6, k


def f16_pair(cuda_lib, t, split_dim=0, split_at=0):
    """fp16 operand pair of a [rows, cols] fp32 device tensor: (pair [2, rows, ld16], scale block [8])."""
    rows, cols = t.shape
    ld16 = cuda_lib.spotv2_gat_ld16(cols)
    pair = torch.zeros(2, rows, ld16, device=DEV, dtype=torch.float16)
    blk = torch.zeros(8, device=DEV)
    check(cuda_lib.spotv2_split_f16(t.data_ptr(), rows, cols, t.stride(0), split_dim, split_at, ptr(pair[0]), ptr(pair[1]), ld16,
                                    ptr(blk), st()), "split_f16")
    return pair, blk


def pair_value(pair, blk, cols, split_at=None):
    """Reconstruct the fp32 values a pair represents (float64 arithmetic)."""
    val = (pair[0].double() + pair[1].double())[:, :cols]
    inv = blk[2:4].double()
    if split_at is None:
        return val * inv[0]
    scale = torch.where(torch.arange(cols, device=pair.device) >= split_at, inv[1], inv[0])
    return val * scale


@pytest.mark.parametrize("algo", [1, 2], ids=["cuda_cores", "tcgen05"])
@pytest.mark.parametrize("shape", [(2, 30, 1260, 6, 500), (3, 7, 9, 3, 5), (5, 30, 100, 8, 33), (1, 1, 3, 1, 1),
                                   (40, 30, 2048, 8, 256), (64, 30, 256, 2, 50)])
def test_projection_gemms(cuda_lib, shape, algo):
    B, N, Fin, H, C_ = shape
    n, n_aug, HC = B * N, H * C_ + 2 * H, H * C_
    ldp = cuda_lib.spotv2_gat_ldp(H, C_)
    d = GatDesc(B, N, Fin, 0, H, C_, 0, 0, 0.2, ldp, algo, 0)
    torch.manual_seed(1)
    x, W_aug, dP = torch.randn(n, Fin), torch.randn(n_aug, Fin), torch.randn(n, ldp)
    # the folded attention rows of W_aug and the ds|dd columns of dP_aug live on their own scale
    W_aug[HC:] *= 37.0
    dP[:, HC:] *= 1e-3
    xg, Wg, dPg = x.to(DEV), W_aug.to(DEV), dP.to(DEV)
    a, b, c = C.c_size_t(), C.c_size_t(), C.c_size_t()
    check(cuda_lib.spotv2_gat_workspace_bytes(C.byref(d), C.byref(a), C.byref(b), C.byref(c)), "ws")
    ws = torch.empty(max(a.value, c.value), dtype=torch.uint8, device=DEV)

    def grouped_relerr(got, ref, split, dim):
        lo = relerr(got.narrow(dim, 0, split), ref.narrow(dim, 0, split))
        hi = relerr(got.narrow(dim, split, got.shape[dim] - split), ref.narrow(dim, split, got.shape[dim] - split))
        return max(lo, hi)

    P = torch.zeros(n, ldp, device=DEV)
    pmax = torch.zeros(8, device=DEV)
    check(cuda_lib.spotv2_proj_fwd(C.byref(d), ptr(xg), None, None, None, ptr(Wg), ptr(P), ptr(pmax), ptr(ws), ws.numel(), st()), "proj_fwd")
    assert pmax[:1].view(torch.int32).view(torch.float32).item() == P[:, :HC].abs().max().item()   # max|P| as the backward wants it
    assert grouped_relerr(P[:, :n_aug], x.double() @ W_aug.double().t(), HC, 1) < TOL
    dW = torch.empty(n_aug, Fin, device=DEV)
    check(cuda_lib.spotv2_proj_bwd_weight(C.byref(d), ptr(xg), None, None, None, ptr(dPg), None, None, None, ptr(dW), ptr(ws),
                                          ws.numel(), st()), "bwd_w")
    assert grouped_relerr(dW, dP[:, :n_aug].double().t() @ x.double(), HC, 0) < TOL
    dX = torch.empty(n, Fin, device=DEV)
    check(cuda_lib.spotv2_proj_bwd_input(C.byref(d), ptr(dPg), None, None, None, ptr(Wg), ptr(dX), ptr(ws), ws.numel(), st()), "bwd_x")
    assert relerr(dX, dP[:, :n_aug].double() @ W_aug.double()) < TOL
    if algo == 2:       # the same products from caller-provided fp16 operand pairs
        assert cuda_lib.spotv2_gat_uses_tensor_cores(C.byref(d)) == 1
        xs, xblk = f16_pair(cuda_lib, xg)
        ps, pblk = f16_pair(cuda_lib, dPg[:, :n_aug], split_dim=1, split_at=HC)
        assert relerr(pair_value(xs, xblk, Fin), x) < 1e-6
        assert relerr(pair_value(ps, pblk, n_aug, HC), dP[:, :n_aug]) < 1e-6
        assert xs[0].abs().max() < 32800 and xs[0].abs().max() >= 16384       # largest magnitude sits in [2^14, 2^15]
        P2, dW2, dX2 = torch.zeros_like(P), torch.empty_like(dW), torch.empty_like(dX)
        check(cuda_lib.spotv2_proj_fwd(C.byref(d), ptr(xg), ptr(xs[0]), ptr(xs[1]), ptr(xblk), ptr(Wg), ptr(P2), None, ptr(ws),
                                       ws.numel(), st()), "proj_fwd")
        check(cuda_lib.spotv2_proj_bwd_weight(C.byref(d), ptr(xg), ptr(xs[0]), ptr(xs[1]), ptr(xblk), None, ptr(ps[0]),
                                              ptr(ps[1]), ptr(pblk), ptr(dW2), ptr(ws), ws.numel(), st()), "bwd_w")
        check(cuda_lib.spotv2_proj_bwd_input(C.byref(d), None, ptr(ps[0]), ptr(ps[1]), ptr(pblk), ptr(Wg), ptr(dX2), ptr(ws),
                                             ws.numel(), st()), "bwd_x")
        assert torch.equal(P2[:, :n_aug], P[:, :n_aug]) and torch.equal(dW2, dW) and torch.equal(dX2, dX)


def test_f16_pair_keeps_absolute_precision_over_a_wide_dynamic_range(cuda_lib):
    """Operands spanning 12 decades: elements far below the group maximum lose relative precision in the
    pair but not absolute precision, so the max-norm error of the product stays at the fp32 level."""
    torch.manual_seed(5)
    M, N, K = 256, 300, 640
    A = torch.randn(M, K) * torch.logspace(-9, 3, K)[None, :]
    Bm = torch.randn(N, K) * torch.logspace(2, -8, N)[:, None]
    ref = A.double() @ Bm.double().t()
    Ag, Bg = A.to(DEV), Bm.to(DEV)
    Cg = torch.empty(M, N, device=DEV)
    ws = torch.empty(1 << 24, dtype=torch.uint8, device=DEV)
    check(cuda_lib.spotv2_diag_gemm(1, 1, M, N, K, ptr(Ag), K, ptr(Bg), K, ptr(Cg), N, 3, 1, 256, 0, ptr(ws), ws.numel(),
                                    st()), "diag_gemm f16")
    assert relerr(Cg, ref) < 3e-6
    assert relerr(Cg, ref) < 4 * relerr((A @ Bm.t()), ref) + 1e-6          # on par with an fp32 CPU matmul


GEMM_CASES = [
    # a_kc, b_kc, M, N, K, splits, bn, kb_per_chunk
    (1, 1, 128, 256, 32, 1, 256, 4), (1, 1, 128, 256, 256, 1, 256, 4), (1, 1, 300, 520, 1260, 1, 256, 4),
    (1, 1, 300, 520, 1260, 1, 128, 2), (1, 1, 4096, 3012, 1260, 1, 256, 4), (1, 1, 77, 40, 100, 1, 128, 1),
    (0, 0, 3012, 1260, 6000, 3, 256, 4), (0, 0, 280, 100, 999 * 4, 5, 128, 4), (0, 0, 128, 256, 64, 1, 256, 4),
    (1, 0, 500, 1260, 3012, 1, 256, 4), (1, 0, 130, 64, 280, 1, 128, 4), (0, 1, 260, 300, 512, 2, 256, 8),
    # bn = 256 + 16 selects the 16-deep k-block variant (64-byte swizzle, 4-stage ring)
    (1, 1, 300, 520, 1260, 1, 272, 8), (0, 0, 3012, 1260, 6000, 3, 272, 8), (1, 0, 500, 1260, 3012, 1, 272, 0),
    (0, 1, 260, 300, 520, 2, 272, 3),
]


@pytest.mark.parametrize("case", GEMM_CASES, ids=[f"{'KM'[c[0]]}{'KM'[c[1]]}_{c[2]}x{c[3]}x{c[4]}_s{c[5]}_bn{c[6]}_c{c[7]}" for c in GEMM_CASES])
def test_tensor_core_gemm_all_layouts(cuda_lib, case):
    """The tcgen05 kernels (3 = fp16 pairs, the production path; 2 = 3xTF32) against float64, for every
    operand-major combination, ragged tiles, split-K and both tile widths; the CUDA-core kernel (1) is run
    beside them as the yardstick."""
    a_kc, b_kc, M, N, K, splits, bn, kbc = case
    torch.manual_seed(M + N + K)
    A = torch.randn(M, K) if a_kc else torch.randn(K, M + (-M) % 4)
    Bm = torch.randn(N, K + (-K) % 4) if b_kc else torch.randn(K, N + (-N) % 4)
    if a_kc:
        A = torch.randn(M, K + (-K) % 4)
    A64 = (A[:, :K] if a_kc else A[:K, :M].t()).double()
    B64 = (Bm[:, :K] if b_kc else Bm[:K, :N].t()).double()
    ref = A64 @ B64.t()
    Ag, Bg = A.to(DEV), Bm.to(DEV)
    ldc = N + (-N) % 4
    ws = torch.empty(8 * (A.numel() + Bm.numel()) + 4 * splits * M * N + 8192, dtype=torch.uint8, device=DEV)
    for algo in (3, 2, 1):
        Cg = torch.full((M, ldc), float("nan"), device=DEV)
        check(cuda_lib.spotv2_diag_gemm(a_kc, b_kc, M, N, K, ptr(Ag), A.shape[1], ptr(Bg), Bm.shape[1], ptr(Cg), ldc,
                                        algo, splits, bn, kbc, ptr(ws), ws.numel(), st()), f"diag_gemm algo {algo}")
        torch.cuda.synchronize()
        err = relerr(Cg[:, :N], ref)
        assert err < 3e-6, f"algo {algo}: {err}"
        if ldc > N:
            assert torch.isnan(Cg[:, N:]).all()          # nothing written beyond N


def test_edge_table_accepts_reference_order_and_rejects_others(cuda_lib):
    N, B = 30, 3
    bt = synth.random_complete_batch(B, N, 4, 2, seed=0)
    topo = sv.topology_from_edge_index(bt.edge_index.to(DEV), B * N)
    assert (topo.B, topo.N, topo.R, topo.has_skips) == (B, N, N * (N - 1), False)
    local = bt.edge_index[:, :topo.R]
    assert torch.equal(topo.table.cpu(), ((local[1] << 16) | local[0]).int())
    bad = bt.edge_index.clone()
    bad[:, 5] = bad[:, 6]                                   # duplicate one edge, drop another
    with pytest.raises(sv.SpotV2Error, match="complete"):
        sv.topology_from_edge_index(bad.to(DEV), B * N)
    bad = bt.edge_index.clone()
    perm = torch.randperm(topo.R)
    bad[:, topo.R:2 * topo.R] = bad[:, topo.R:2 * topo.R][:, perm]   # second graph in a different edge order
    with pytest.raises(sv.SpotV2Error, match="differs"):
        sv.topology_from_edge_index(bad.to(DEV), B * N)


@pytest.mark.parametrize("bwd_algo", [3, 2, 1], ids=["tcgen05", "pipelined", "phase_serial"])
@pytest.mark.parametrize("geom", [(5, 30, 16, 126, 6, 20), (160, 30, 16, 126, 6, 500), (7, 30, 8, 126, 8, 36), (4, 13, 8, 5, 3, 7),
                                  (300, 30, 8, 126, 6, 500), (9, 31, 8, 10, 7, 44), (6, 2, 8, 4, 2, 8)],
                         ids=["small", "default_channels_2_graphs_per_cta", "H8", "odd", "two_graphs_per_cta_default", "N31_H7", "N2"])
def test_attention_stages_against_dense_oracle(cuda_lib, geom, bwd_algo):
    """attn_fwd / attn_bwd alone (P_aug given), compared stage by stage with oracle/dense_gat.py."""
    _attention_stage_case(cuda_lib, geom, bwd_algo)


@pytest.mark.parametrize("geom", [(2, 40, 8, 126, 6, 20), (2, 77, 8, 5, 3, 7), (1, 131, 8, 36, 8, 12), (1, 500, 8, 126, 6, 500)],
                         ids=["N40", "N77_odd", "N131_H8", "config_D_graph"])
def test_large_universe_attention_stages(cuda_lib, geom):
    """N > 32: the multi-CTA-per-graph kernels (attn_large.cu), same entry points, same stage-by-stage check.
    The last case is one full-size BASELINE config-D graph (500 nodes, 249 500 edge rows, H=6, C=500)."""
    _attention_stage_case(cuda_lib, geom, 0)


def _attention_stage_case(cuda_lib, geom, bwd_algo):
    B, N, Fin, Fe, H, C_ = geom
    for concat in (False, True):
        bt = synth.random_complete_batch(B, N, Fin, Fe, seed=4)
        ref, _ = make_layers(Fin, C_, H, concat, Fe, 0.2, seed=9, wscale=2.0)
        W, a_s, a_d, We, a_e, bias = [p.detach() for p in (ref.lin_src.weight, ref.att_src, ref.att_dst,
                                                           ref.lin_edge.weight, ref.att_edge, ref.bias)]
        T = dense_gat.pyg_to_dense_tile(bt.edge_attr.double(), bt.edge_index, B, N)
        fw = dense_gat.dense_forward(bt.x.double(), T, W, a_s, a_d, We, a_e, bias, H, C_, concat, 0.2)
        ldp = cuda_lib.spotv2_gat_ldp(H, C_)
        # the tcgen05 backward (algo 3) covers head-mean layers with N <= 31, C % 4 == 0, even Fe <= 128 and needs the
        # forward's edge terms: the calls without them, and the shapes outside its range, run the pipelined kernel
        tc5 = bwd_algo == 3 and not concat and N <= 31 and C_ % 4 == 0 and Fe % 2 == 0 and Fe <= 128
        if bwd_algo == 3 and not tc5 and concat is False and geom != (4, 13, 8, 5, 3, 7):
            raise AssertionError("the tcgen05 kernel should apply to this geometry")
        d = GatDesc(B, N, Fin, Fe, H, C_, N * (N - 1), int(concat), 0.2, ldp, 0, 2 if bwd_algo == 3 else bwd_algo)
        d_t = GatDesc(B, N, Fin, Fe, H, C_, N * (N - 1), int(concat), 0.2, ldp, 0, 3 if tc5 else d.attn_bwd_algo)
        P_aug = torch.full((B * N, ldp), float("nan"), device=DEV)       # padding columns may hold anything
        P_aug[:, :H * C_ + 2 * H] = fw["P_aug"].float().to(DEV)
        topo = sv.topology_from_edge_index(bt.edge_index.to(DEV), B * N)
        ea, v, bg = bt.edge_attr.to(DEV), fw["v"].float().to(DEV).contiguous(), bias.float().to(DEV)
        ldo = H * C_ if concat else C_
        out = torch.empty(B * N, ldo, device=DEV)
        alpha = torch.empty(B, H, N, N, device=DEV)
        etb = C.c_size_t()
        check(cuda_lib.spotv2_gat_edge_terms_bytes(C.byref(d), C.byref(etb)), "edge_terms_bytes")
        terms = torch.full((etb.value // 4,), float("nan"), device=DEV)
        check(cuda_lib.spotv2_gat_attn_fwd(C.byref(d), ptr(P_aug), ptr(ea), ptr(topo.table), ptr(v), ptr(bg), ptr(out),
                                           ptr(alpha), ptr(terms), None, 0, st()), "attn_fwd")
        assert relerr(alpha, fw["alpha"].permute(0, 3, 2, 1)) < TOL     # ours is [B, H, j, i]
        assert relerr(out, fw["out"]) < TOL
        # without return_attention_weights the (N > 32) attention tile lives in a workspace: same bits
        wsz = C.c_size_t()
        check(cuda_lib.spotv2_gat_attn_fwd_workspace_bytes(C.byref(d), C.byref(wsz)), "attn_fwd_ws")
        assert (wsz.value > 0) == (N > 32)
        ws_f = torch.empty(max(wsz.value, 1), dtype=torch.uint8, device=DEV)
        out2 = torch.empty_like(out)
        check(cuda_lib.spotv2_gat_attn_fwd(C.byref(d), ptr(P_aug), ptr(ea), ptr(topo.table), ptr(v), ptr(bg), ptr(out2),
                                           None, None, ptr(ws_f), wsz.value, st()), "attn_fwd")
        assert torch.equal(out, out2)
        dout = torch.randn(B * N, ldo)
        gr = dense_gat.dense_backward(fw, bt.x.double(), T, W, a_s, a_d, We, a_e, dout.double(), H, C_, concat, 0.2)
        a, b, c = C.c_size_t(), C.c_size_t(), C.c_size_t()
        check(cuda_lib.spotv2_gat_workspace_bytes(C.byref(d), C.byref(a), C.byref(b), C.byref(c)), "ws")
        ws = torch.empty(b.value, dtype=torch.uint8, device=DEV)
        dP = torch.zeros(B * N, ldp, device=DEV)
        dv, dbias = torch.empty(H, Fe, device=DEV), torch.empty(ldo, device=DEV)
        dout_g = dout.to(DEV)
        check(cuda_lib.spotv2_gat_attn_bwd(C.byref(d), ptr(P_aug), None, ptr(ea), None, ptr(topo.table), ptr(v), ptr(dout_g),
                                           ptr(dP), None, None, None, ptr(dv), None, ptr(dbias), ptr(ws), ws.numel(), st()), "attn_bwd")
        # same call with the edge terms the forward kept (no first pass over the edge rows): same results to rounding
        dP_t = torch.zeros(B * N, ldp, device=DEV)
        dv_t, dbias_t = torch.empty(H, Fe, device=DEV), torch.empty(ldo, device=DEV)
        check(cuda_lib.spotv2_gat_attn_bwd(C.byref(d_t), ptr(P_aug), None, ptr(ea), ptr(terms), ptr(topo.table), ptr(v), ptr(dout_g),
                                           ptr(dP_t), None, None, None, ptr(dv_t), None, ptr(dbias_t), ptr(ws), ws.numel(), st()), "attn_bwd")
        torch.cuda.synchronize()
        assert relerr(dP_t[:, :H * C_ + 2 * H], dP[:, :H * C_ + 2 * H]) < 3e-6 and relerr(dv_t, dv) < 3e-6
        assert torch.equal(dbias_t, dbias) if not tc5 else relerr(dbias_t, dbias) < 2e-6
        # the tensor-core operand form: the fp16 pair reproduces the fp32 gradient to ~2^-22 of each group's scale
        n_aug = H * C_ + 2 * H
        dP16 = torch.zeros(2, B * N, cuda_lib.spotv2_gat_ld16(n_aug), device=DEV, dtype=torch.float16)
        pblk = torch.zeros(8, device=DEV)
        check(cuda_lib.spotv2_gat_attn_bwd(C.byref(d_t), ptr(P_aug), None, ptr(ea), ptr(terms), ptr(topo.table), ptr(v), ptr(dout_g),
                                           None, ptr(dP16[0]), ptr(dP16[1]), ptr(pblk), ptr(dv), None, ptr(dbias), ptr(ws),
                                           ws.numel(), st()), "attn_bwd")
        got = pair_value(dP16, pblk, n_aug, H * C_)
        # (the pair run used the forward's edge terms, the fp32 run recomputed them: two roundings of the same logits)
        assert relerr(got[:, :H * C_], dP[:, :H * C_]) < 3e-6 and relerr(got[:, H * C_:], dP[:, H * C_:n_aug]) < 3e-6
        assert torch.isfinite(dP16.float()).all() and dP16[0].abs().max() < 32800
        HC = H * C_
        assert relerr(dP[:, :HC], gr["dP_aug"][:, :HC]) < TOL
        assert relerr(dP[:, HC:HC + 2 * H], gr["dP_aug"][:, HC:]) < TOL
        assert relerr(dv, gr["dv"]) < TOL and relerr(dbias, gr["bias"]) < TOL
        # (dv / dbias above come from the LAST call, i.e. from d_t's kernel; its fp32 dP against the oracle as well)
        assert relerr(dP_t[:, :HC], gr["dP_aug"][:, :HC]) < TOL and relerr(dP_t[:, HC:HC + 2 * H], gr["dP_aug"][:, HC:]) < TOL
        assert relerr(dv_t, gr["dv"]) < TOL and relerr(dbias_t, gr["bias"]) < TOL


# ------------------------------------------------------------------ the layer, end to end
CASES = [
    # B, N, Fin, Fe, H, C, concat, slope, wscale
    (4, 30, 1260, 126, 6, 500, False, 0.2, 1.0),      # default config geometry (config/GNN_param.yaml)
    (3, 30, 120, 12, 6, 20, True, 0.2, 1.0),
    (2, 30, 64, 126, 8, 256, True, 0.2, 1.0),         # BASELINE config C layer 0
    (2, 30, 2048, 126, 8, 256, False, 0.2, 1.0),      # BASELINE config C layer 1
    (4, 7, 9, 5, 3, 5, False, 0.5, 2.0),              # odd everything -> scalar / unaligned paths
    (3, 12, 16, 8, 7, 12, False, 0.8, 4.0),
    (2, 2, 4, 3, 1, 2, True, 0.05, 1.0),
    (5, 1, 6, 2, 2, 3, False, 0.2, 1.0),              # single-node graphs: only the self loop
    (2, 32, 10, 7, 2, 6, True, 0.2, 1.0),             # N = 32, the kernel's upper bound
    (2, 17, 30, 360, 2, 25, False, 0.1, 1.0),         # seq_length 120 -> Fe = 360 (HPO space), odd C
]


@pytest.fixture
def bwd_kernel(request):
    """Run the test body with a given attention-backward kernel (0 = library's choice: the pipelined kernel,
    1 = the phase-serial any-shape kernel) and GEMM back end."""
    from spotv2net_b200 import gat_conv
    old = (gat_conv.ATTN_BWD_ALGO, gat_conv.GEMM_ALGO)
    gat_conv.ATTN_BWD_ALGO, gat_conv.GEMM_ALGO = request.param
    yield request.param
    gat_conv.ATTN_BWD_ALGO, gat_conv.GEMM_ALGO = old


BACKENDS = [(0, 0), (3, 0), (1, 0), (0, 1), (3, 1)]
BACKEND_IDS = ["piped_bwd+tc_gemm", "tcgen05_bwd+tc_gemm", "serial_bwd+tc_gemm", "piped_bwd+simt_gemm", "tcgen05_bwd+simt_gemm"]


@pytest.mark.parametrize("bwd_kernel", BACKENDS, ids=BACKEND_IDS, indirect=True)
@pytest.mark.parametrize("case", CASES, ids=[f"B{c[0]}N{c[1]}F{c[2]}Fe{c[3]}H{c[4]}C{c[5]}{'cat' if c[6] else 'mean'}" for c in CASES])
def test_layer_matches_edge_list_oracle(cuda_lib, case, bwd_kernel):
    B, N, Fin, Fe, H, C_, concat, slope, wscale = case
    if bwd_kernel[0] == 3 and (concat or N > 31 or N < 2 or C_ % 4 or Fe % 2 or not 0 < Fe <= 128):
        pytest.skip("outside the tcgen05 backward's range (head-mean, 2 <= N <= 31, C % 4 == 0, even Fe <= 128)")
    ref, ours = make_layers(Fin, C_, H, concat, Fe, slope, seed=B + N, wscale=wscale)
    if N == 1:
        bt = synth.Batch(x=torch.randn(B, Fin), edge_index=torch.arange(B).repeat(2, 1),
                         edge_attr=torch.randn(B, Fe), num_graphs=B)     # input = self loops only
        ours.nodes_per_graph = 1
    else:
        bt = synth.random_complete_batch(B, N, Fin, Fe, seed=17)
    bad = run_both(ref, ours, bt, need_dx=True)
    assert not bad, f"(our error, fp32-oracle error) above the bar: {bad}"


LARGE_CASES = [
    # B, N, Fin, Fe, H, C, concat, slope
    (2, 33, 16, 5, 3, 7, True, 0.2),                  # first size past the one-CTA-per-graph kernels
    (3, 64, 20, 126, 6, 20, False, 0.2),
    (2, 100, 12, 9, 8, 33, True, 0.05),               # odd channel count -> scalar GEMM loads
    (1, 131, 10, 126, 2, 10, False, 0.2),             # odd N: unaligned attention-tile rows
    (1, 500, 24, 126, 6, 40, False, 0.2),             # BASELINE config D universe (500 nodes, 249 500 edges)
]


@pytest.mark.parametrize("gemm_algo", [0, 1], ids=["tc_gemm", "simt_gemm"])
@pytest.mark.parametrize("case", LARGE_CASES, ids=[f"B{c[0]}N{c[1]}F{c[2]}Fe{c[3]}H{c[4]}C{c[5]}{'cat' if c[6] else 'mean'}" for c in LARGE_CASES])
def test_large_universe_layer_matches_edge_list_oracle(cuda_lib, case, gemm_algo):
    """BASELINE config D: graphs larger than one CTA's shared memory take the multi-CTA-per-graph path."""
    from spotv2net_b200 import gat_conv
    B, N, Fin, Fe, H, C_, concat, slope = case
    ref, ours = make_layers(Fin, C_, H, concat, Fe, slope, seed=B + N)
    bt = synth.random_complete_batch(B, N, Fin, Fe, seed=23)
    old = gat_conv.GEMM_ALGO
    gat_conv.GEMM_ALGO = gemm_algo
    try:
        bad = run_both(ref, ours, bt, need_dx=True)
    finally:
        gat_conv.GEMM_ALGO = old
    assert not bad, f"(our error, fp32-oracle error) above the bar: {bad}"


@pytest.mark.parametrize("bwd_algo", [0, 1], ids=["pipelined_bwd", "serial_bwd"])
@pytest.mark.parametrize("case", [(3, 30, 40, 126, 6, 20, False), (2, 13, 9, 5, 3, 7, True), (2, 40, 12, 9, 4, 10, False),
                                  (3, 30, 1260, 126, 6, 500, False), (2, 30, 64, 126, 8, 32, True)],
                         ids=["N30_mean", "N13_cat", "N40_large_path", "default_geometry", "H8_cat"])
def test_attention_dropout_in_training_mode_replays_in_the_oracle(cuda_lib, case, bwd_algo):
    """dropout_att > 0 (F.dropout(alpha) in [PyG] gat_conv.py message; HPO range of the reference).  The mask comes
    from the library's own Philox stream, so parity is checked by REPLAYING it: the dropped coefficients returned by
    return_attention_weights give the Bernoulli draw, the oracle applies the same draw, and outputs and every
    gradient (whose backward regenerates the mask from the key) must agree to the usual bar."""
    import copy
    from spotv2net_b200 import gat_conv
    B, N, Fin, Fe, H, C_, concat = case
    pdrop = 0.3
    old_algo = gat_conv.ATTN_BWD_ALGO
    gat_conv.ATTN_BWD_ALGO = bwd_algo
    try:
        _dropout_case(B, N, Fin, Fe, H, C_, concat, pdrop)
    finally:
        gat_conv.ATTN_BWD_ALGO = old_algo


@pytest.mark.parametrize("bwd_algo", [0, 1], ids=["pipelined_bwd", "serial_bwd"])
@pytest.mark.parametrize("pdrop", [0.7, 0.9])
def test_attention_dropout_at_high_rates_with_peaked_rows(cuda_lib, pdrop, bwd_algo):
    """p = 0.7 is the top of the reference's HPO range, 0.9 is beyond it; GATConv accepts any p in [0, 1).  Weights
    scaled x4 concentrate the softmax (rows with one coefficient near 1), so kept coefficients reach 1/(1-p) = 10:
    the backward's fp16 operands must not carry that factor (it rides in the fp32 post-scale) and the bound that
    sizes the dP scale must include it."""
    from spotv2net_b200 import gat_conv
    old_algo = gat_conv.ATTN_BWD_ALGO
    gat_conv.ATTN_BWD_ALGO = bwd_algo
    try:
        _dropout_case(6, 30, 40, 126, 6, 20, False, pdrop, wscale=4.0)
    finally:
        gat_conv.ATTN_BWD_ALGO = old_algo


def _dropout_case(B, N, Fin, Fe, H, C_, concat, pdrop, wscale=1.0):
    import copy
    ref, ours = make_layers(Fin, C_, H, concat, Fe, 0.2, seed=N, wscale=wscale)
    ours.dropout = ref.dropout = pdrop
    bt = synth.random_complete_batch(B, N, Fin, Fe, seed=31)
    dout = torch.randn(B * N, H * C_ if concat else C_)
    xg, eig, eag = bt.x.to(DEV).requires_grad_(True), bt.edge_index.to(DEV), bt.edge_attr.to(DEV)

    def ours_pass(seed):
        ours.zero_grad()
        xg.grad = None
        torch.manual_seed(seed)
        out, (_, a) = ours(xg, eig, eag, return_attention_weights=True)
        out.backward(dout.to(DEV))
        res = {"out": out.detach(), "alpha": a.detach(), "g_x": xg.grad.clone()}
        res.update({"g_" + k: p.grad.clone() for k, p in ours.named_parameters()})
        return res

    ours.train()
    mine = ours_pass(7)
    mask = (mine["alpha"] != 0).cpu()
    keep = mask.float().mean().item()
    assert abs(keep - (1 - pdrop)) < 0.03, keep
    again = ours_pass(7)
    assert all(torch.equal(mine[k], again[k]) for k in mine)            # same torch seed, same key, same bits
    other = ours_pass(8)
    assert not torch.equal((other["alpha"] != 0).cpu(), mask)            # a fresh key per step

    def oracle(dtype):
        m = copy.deepcopy(ref).to(dtype).train()
        x = bt.x.to(dtype).requires_grad_(True)
        out, (_, a) = m(x, bt.edge_index, bt.edge_attr.to(dtype), return_attention_weights=True, dropout_mask=mask)
        out.backward(dout.to(dtype))
        res = {"out": out.detach(), "alpha": a.detach(), "g_x": x.grad}
        res.update({"g_" + k: p.grad for k, p in m.named_parameters()})
        return res

    bad = parity_failures(mine, oracle(torch.float64), oracle(torch.float32))
    assert not bad, bad
    ours.eval()                                                          # eval mode: no dropout
    out_eval, (_, a_eval) = ours(xg, eig, eag, return_attention_weights=True)
    assert (a_eval >= 0).all() and (wscale != 1.0 or (a_eval > 0).all())   # (peaked rows underflow to exact zeros)
    ref_eval = copy.deepcopy(ref).eval()(bt.x.double(), bt.edge_index, bt.edge_attr.double())
    assert relerr(out_eval, ref_eval) < TOL


def test_config_c_two_layer_model_fp32_and_half_precision(cuda_lib):
    """BASELINE config C (8 heads, hidden [256, 256], concat: layer 0 1260 -> 8x256 concat, layer 1 2048 -> 256 mean).

    Two layers multiply the opportunities for a LeakyReLU / ReLU argument to sit within fp32 noise of zero (57 600
    attention logits and 491 520 activations here); one such kink flipping between two implementations moves the
    heavily cancelled attention-parameter gradients by percents in ANY implementation (measured: the fp64 oracle
    evaluated at activations that differ by 2e-6 moves them by 2-5e-2).  So the model is checked layer by layer with
    teacher forcing - the fp64 oracle layer is evaluated at OUR input activations and OUR upstream gradient - on a
    seed whose logits keep a 2e-5 relative margin from the kink (asserted below).
      * fp32 mode: every layer's output and gradients meet the 1e-5 bar;
      * "half" mode (layer.precision = "half": ONE fp16 tensor-core product per projection, fp32 accumulate - 11-bit
        operands, at least bf16's 8; the reduced-precision variant the config names): reported separately, as
        north_star asks - layer outputs within 4e-3, projection-weight and bias gradients within 2e-2."""
    import copy
    N, L, B = 30, 42, 4
    vol, vv = synth.synthetic_matrices(L + B + 2, N, seed=3)
    kw = dict(num_node_features=N * L, num_edge_features=3 * L, num_heads=8, output_node_channels=1,
              dim_hidden_layers=[256, 256], concat_heads=True)
    torch.manual_seed(2)
    ref = pyg_gat.OracleGATModel(**kw).double()
    ours = sv.GATModel(**kw)
    ours.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
    ours.to(DEV)
    cpu = synth.make_batch(vol, vv, list(range(B)), L)
    dev = synth.make_batch(vol, vv, list(range(B)), L).to(DEV)
    topo = sv.topology_from_edge_index(dev.edge_index, dev.x.shape[0])

    def ours_pass():
        ours.zero_grad()
        acts, x = [], dev.x
        for layer in ours.gat_layers:
            x_in = x
            h = layer(x_in, dev.edge_index, dev.edge_attr, topology=topo)
            h.retain_grad()
            acts.append((x_in, h))
            x = torch.relu(h)
        torch.nn.functional.mse_loss(ours.linear(x).view(-1), dev.y_x).backward()
        return acts

    def oracle_layer(k, x_in, dout, dtype):
        m = copy.deepcopy(ref.gat_layers[k]).to(dtype)
        x = x_in.detach().cpu().to(dtype).requires_grad_(True)
        out, (_, alpha) = m(x, cpu.edge_index, cpu.edge_attr.to(dtype), return_attention_weights=True)
        out.backward(dout.detach().cpu().to(dtype))
        res = {"out": out.detach(), "g_x": x.grad}
        res.update({"g_" + n_: p.grad for n_, p in m.named_parameters()})
        return res, out.detach()

    report = {}
    for prec in ("fp32", "half"):
        ours.set_precision(prec)
        acts = ours_pass()
        for k, (x_in, h) in enumerate(acts):
            r64, _ = oracle_layer(k, x_in, h.grad, torch.float64)
            r32, _ = oracle_layer(k, x_in, h.grad, torch.float32)
            mine = {"out": h.detach()}
            mine.update({"g_" + n_: p.grad for n_, p in ours.gat_layers[k].named_parameters()})
            r64.pop("g_x"); r32.pop("g_x")           # dX of both layer geometries is covered by CASES (need_dx=True)
            errs = {t: relerr(mine[t], r64[t]) for t in r64}
            report[(prec, k)] = errs
            if prec == "fp32":
                bad = parity_failures(mine, r64, r32)
                assert not bad, (k, bad)
            else:
                assert errs["out"] < 4e-3, (k, errs)
                assert errs["g_lin_src.weight"] < 2e-2 and errs["g_bias"] < 2e-2, (k, errs)
    for key, errs in report.items():
        print("config C", key, {t: f"{e:.1e}" for t, e in errs.items()})
    # the single-product path really ran: its forward error sits orders of magnitude above the fp32 mode's
    assert report[("half", 0)]["out"] > 20 * report[("fp32", 0)]["out"]
    # kink margin of this seed (fp64, oracle activations): no attention logit within 1e-5 of zero, relative
    x = cpu.x.double()
    T = dense_gat.pyg_to_dense_tile(cpu.edge_attr.double(), cpu.edge_index, B, N)
    for l in ref.gat_layers:
        fw = dense_gat.dense_forward(x, T, l.lin_src.weight.detach(), l.att_src.detach(), l.att_dst.detach(),
                                     l.lin_edge.weight.detach(), l.att_edge.detach(), l.bias.detach(), l.heads,
                                     l.out_channels, l.concat, 0.2)
        assert fw["z"].abs().min() > 1e-5 * fw["z"].abs().max()
        x = torch.relu(fw["out"])


def test_layer_without_edge_attr_and_with_input_self_loops(cuda_lib):
    B, N, Fin, Fe, H, C_ = 3, 9, 10, 4, 2, 6
    ref, ours = make_layers(Fin, C_, H, True, Fe, 0.2, seed=3)
    bt = synth.random_complete_batch(B, N, Fin, Fe, seed=5)
    no_ea = synth.Batch(x=bt.x, edge_index=bt.edge_index, edge_attr=None)
    out_ref = ref(bt.x.double(), bt.edge_index, None)
    out = ours(bt.x.to(DEV), bt.edge_index.to(DEV), None)
    assert relerr(out, out_ref) < TOL                       # Explainer path, 6_results.ipynb:1347
    del no_ea
    # self loops present in the input are dropped and replaced by the mean-filled ones
    ei = torch.cat([bt.edge_index.view(2, B, -1), (torch.arange(B * N).view(1, B, N)).expand(2, B, N)], 2).reshape(2, -1)
    ea = torch.cat([bt.edge_attr.view(B, -1, Fe), 50 * torch.randn(B, N, Fe)], 1).reshape(-1, Fe)
    with_loops = synth.Batch(x=bt.x, edge_index=ei, edge_attr=ea)
    assert not run_both(ref, ours, with_loops)


def test_dense_tile_input(cuda_lib):
    """The collation's dense target-major tile [B, N, N, Fe] is accepted through the same entry point."""
    B, N, Fin, Fe, H, C_ = 3, 30, 8, 12, 6, 10
    bt = synth.random_complete_batch(B, N, Fin, Fe, seed=8)
    ref, _ = make_layers(Fin, C_, H, False, Fe, 0.2, seed=2)
    W, a_s, a_d, We, a_e, bias = [p.detach() for p in (ref.lin_src.weight, ref.att_src, ref.att_dst,
                                                       ref.lin_edge.weight, ref.att_edge, ref.bias)]
    T = dense_gat.pyg_to_dense_tile(bt.edge_attr.double(), bt.edge_index, B, N)
    T = T + torch.eye(N).view(1, N, N, 1) * 1e6            # garbage on the diagonal must be ignored
    fw = dense_gat.dense_forward(bt.x.double(), T, W, a_s, a_d, We, a_e, bias, H, C_, False, 0.2)
    ldp = cuda_lib.spotv2_gat_ldp(H, C_)
    d = GatDesc(B, N, Fin, Fe, H, C_, N * N, 0, 0.2, ldp, 0, 0)
    table = torch.empty(N * N, dtype=torch.int32, device=DEV)
    check(cuda_lib.spotv2_edge_table_dense(N, ptr(table), st()), "table_dense")
    P_aug = torch.zeros(B * N, ldp, device=DEV)
    P_aug[:, :H * C_ + 2 * H] = fw["P_aug"].float().to(DEV)
    out = torch.empty(B * N, C_, device=DEV)
    T_g, v_g, b_g = T.float().to(DEV).contiguous(), fw["v"].float().to(DEV).contiguous(), bias.float().to(DEV)
    check(cuda_lib.spotv2_gat_attn_fwd(C.byref(d), ptr(P_aug), ptr(T_g), ptr(table), ptr(v_g), ptr(b_g), ptr(out),
                                       None, None, None, 0, st()), "attn_fwd")
    assert relerr(out, fw["out"]) < TOL


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_golden_fixtures_on_gpu(cuda_lib, path):
    z = np.load(path)
    B, N, Fin, Fe, H, C_, concat = [int(v) for v in z["meta"]]
    layer = sv.GATConv(Fin, C_, heads=H, concat=bool(concat), negative_slope=float(z["slope"]), edge_dim=Fe)
    t = lambda k: torch.from_numpy(z[k])
    layer.load_state_dict({"att_src": t("att_src"), "att_dst": t("att_dst"), "att_edge": t("att_edge"),
                           "bias": t("bias"), "lin_src.weight": t("lin_weight"), "lin_dst.weight": t("lin_weight"),
                           "lin_edge.weight": t("lin_edge_weight")})
    layer.to(DEV)
    out, (ei2, alpha) = layer(t("x").to(DEV), t("edge_index").to(DEV), t("edge_attr").to(DEV), return_attention_weights=True)
    out.backward(t("dout").to(DEV))
    assert (ei2.cpu().numpy() == z["edge_index_with_loops"]).all()
    names = ("lin_weight", "att_src", "att_dst", "lin_edge_weight", "att_edge", "bias")
    # fp32 PyG-order oracle on the same fixture, to calibrate ill-conditioned gradients (see parity_failures)
    p32 = [t(k).clone().requires_grad_() for k in names]
    o32, (_, a32) = pyg_gat.gat_conv_edgelist(t("x"), t("edge_index"), t("edge_attr"), *p32, H, C_, bool(concat),
                                              float(z["slope"]), return_attention_weights=True)
    o32.backward(t("dout"))
    mine = {"out": out.detach(), "alpha": alpha.detach()}
    r64 = {"out": torch.from_numpy(z["out"]), "alpha": torch.from_numpy(z["alpha"])}
    r32 = {"out": o32.detach(), "alpha": a32.detach()}
    for k, p, q in zip(names, (layer.lin_src.weight, layer.att_src, layer.att_dst, layer.lin_edge.weight,
                               layer.att_edge, layer.bias), p32):
        mine["g_" + k], r64["g_" + k], r32["g_" + k] = p.grad, torch.from_numpy(z["g_" + k]), q.grad
    assert not parity_failures(mine, r64, r32)


# ------------------------------------------------------------------ model + collation
@pytest.mark.parametrize("cfg", [dict(dim_hidden_layers=[40], concat_heads=True),
                                 dict(dim_hidden_layers=[24, 16], concat_heads=True),
                                 dict(dim_hidden_layers=[24, 16, 8], concat_heads=False, activation="tanh"),
                                 dict(dim_hidden_layers=[20], concat_heads=False, standardize=True)])
def test_model_step_matches_oracle_model(cuda_lib, cfg):
    N, L, B = 30, 3, 6
    vol, vv = synth.synthetic_matrices(L + B + 2, N, seed=21)
    bt = synth.make_batch(vol, vv, list(range(B)), L)
    kw = dict(num_node_features=N * L, num_edge_features=3 * L, num_heads=3, output_node_channels=1, **cfg)
    torch.manual_seed(0)
    ref = pyg_gat.OracleGATModel(**kw).double()
    ours = sv.GATModel(**kw)
    ours.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
    ours.to(DEV)
    ref.train(); ours.train()
    d64 = synth.Batch(x=bt.x.double(), edge_index=bt.edge_index, edge_attr=bt.edge_attr.double())
    loss_ref = torch.nn.functional.mse_loss(ref(d64), bt.y_x.double())
    loss_ref.backward()
    loss = torch.nn.functional.mse_loss(ours(bt.to(DEV)), bt.y_x.to(DEV))
    loss.backward()
    import copy
    ref32 = copy.deepcopy(ref).float()
    ref32.zero_grad()
    torch.nn.functional.mse_loss(ref32(synth.Batch(x=bt.x.cpu(), edge_index=bt.edge_index.cpu(), edge_attr=bt.edge_attr.cpu())),
                                 bt.y_x.cpu()).backward()
    assert abs(loss.item() - loss_ref.item()) <= 2e-5 * abs(loss_ref.item())
    mine = {k: p.grad for k, p in ours.named_parameters()}
    bad = parity_failures(mine, {k: p.grad for k, p in ref.named_parameters()},
                          {k: p.grad for k, p in ref32.named_parameters()})
    assert not bad, bad


def test_device_collation_matches_reference_layouts(cuda_lib):
    N, L, T = 30, 5, 40
    vol, vv = synth.synthetic_matrices(T, N, seed=33)
    ds = sv.WindowDataset(vol, vv, seq_length=L, device=DEV, drop_first=3)
    assert len(ds) == T - L - 3
    idx = [0, 7, 31, 2]
    ours = ds.collate(idx)
    ref = synth.make_batch(vol, vv, [i + 3 for i in idx], L)
    assert torch.equal(ours.x.cpu(), ref.x) and torch.equal(ours.edge_attr.cpu(), ref.edge_attr)
    assert torch.equal(ours.y_x.cpu(), ref.y_x) and torch.equal(ours.edge_index.cpu(), ref.edge_index)
    assert torch.equal(ours.batch.cpu(), ref.batch) and torch.equal(ours.ptr.cpu(), ref.ptr)
    loader = sv.WindowLoader(ds[:20], batch_size=8, shuffle=False)
    sizes = [b.num_graphs for b in loader]
    assert sizes == [8, 8, 4] and len(loader) == 3


def test_multi_output_variant_collation_and_model_step(cuda_lib):
    """output_node_channels = 14 (config/GNN_param.yaml:29 HPO space; 5_train_SpotV2Net.py:66-76 switches to
    CovarianceLaggedMultiOutputDataset, utils/dataset.py:293-412): targets are the next K diagonals per node."""
    N, L, T, K = 30, 4, 40, 14
    vol, vv = synth.synthetic_matrices(T, N, seed=12)
    ds = sv.WindowDataset(vol, vv, seq_length=L, device=DEV, drop_first=2, future_steps=K)
    assert len(ds) == T - L - K + 1 - 2
    idx = [0, 5, len(ds) - 1]
    ours_bt = ds.collate(idx)
    ref_bt = synth.make_batch(vol, vv, [i + 2 for i in idx], L, future_steps=K)
    assert ours_bt.y_x.shape == (len(idx) * N * K,)
    assert torch.equal(ours_bt.y_x.cpu(), ref_bt.y_x) and torch.equal(ours_bt.x.cpu(), ref_bt.x)
    assert torch.equal(ours_bt.edge_attr.cpu(), ref_bt.edge_attr)
    kw = dict(num_node_features=N * L, num_edge_features=3 * L, num_heads=3, output_node_channels=K,
              dim_hidden_layers=[20], concat_heads=False)
    torch.manual_seed(1)
    ref = pyg_gat.OracleGATModel(**kw).double()
    ours = sv.GATModel(**kw)
    ours.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
    ours.to(DEV)
    d64 = synth.Batch(x=ref_bt.x.double(), edge_index=ref_bt.edge_index, edge_attr=ref_bt.edge_attr.double())
    loss_ref = torch.nn.functional.mse_loss(ref(d64), ref_bt.y_x.double())
    loss_ref.backward()
    loss = torch.nn.functional.mse_loss(ours(ours_bt), ours_bt.y_x)
    loss.backward()
    assert abs(loss.item() - loss_ref.item()) <= 2e-5 * abs(loss_ref.item())
    import copy
    ref32 = copy.deepcopy(ref).float()
    ref32.zero_grad()
    torch.nn.functional.mse_loss(ref32(synth.Batch(x=ref_bt.x, edge_index=ref_bt.edge_index, edge_attr=ref_bt.edge_attr)),
                                 ref_bt.y_x).backward()
    bad = parity_failures({k: p.grad for k, p in ours.named_parameters()}, {k: p.grad for k, p in ref.named_parameters()},
                          {k: p.grad for k, p in ref32.named_parameters()})
    assert not bad, bad


def test_evaluation_loop_and_attention_export_match_the_oracle_model(cuda_lib):
    """6_results.ipynb: batched no-grad evaluation with de-standardised predictions, and the per-layer attention
    coefficients of the notebook's GATModel variant."""
    N, L, T = 30, 3, 30
    vol, vv = synth.synthetic_matrices(T, N, seed=44)
    kw = dict(num_node_features=N * L, num_edge_features=3 * L, num_heads=4, output_node_channels=1,
              dim_hidden_layers=[12, 8], concat_heads=True)
    torch.manual_seed(3)
    ref = pyg_gat.OracleGATModel(**kw).double().eval()
    ours = sv.GATModel(**kw)
    ours.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
    ours.to(DEV)
    ds = sv.WindowDataset(vol, vv, seq_length=L, device=DEV, drop_first=1)
    mean, std = 0.37, 2.5
    res = sv.evaluate(ours, sv.WindowLoader(ds, batch_size=8, shuffle=False), mean=mean, std=std)
    assert ours.training                                   # mode restored
    preds, actual, losses = [], [], []
    with torch.no_grad():
        for s0 in range(0, len(ds), 8):
            bt = synth.make_batch(vol, vv, [i + 1 for i in range(s0, min(s0 + 8, len(ds)))], L)
            d64 = synth.Batch(x=bt.x.double(), edge_index=bt.edge_index, edge_attr=bt.edge_attr.double())
            yh, y = ref(d64) * std + mean, bt.y_x.double() * std + mean
            preds.append(yh); actual.append(y); losses.append(torch.nn.functional.mse_loss(yh, y).item())
    assert relerr(res["preds"], torch.cat(preds)) < TOL and relerr(res["actual"], torch.cat(actual)) < 1e-6
    assert abs(res["mse"] - sum(losses) / len(losses)) <= 2e-5 * abs(sum(losses) / len(losses))
    assert res["preds"].view(-1, N).shape[0] == len(ds)
    # attention export, layer by layer
    bt = synth.make_batch(vol, vv, [1, 2, 3], L)
    att = sv.attention_weights(ours, ds.collate([0, 1, 2]))
    x = bt.x.double()
    for layer, (ei2, alpha) in zip(ref.gat_layers, att):
        x, (ei_ref, a_ref) = layer(x, bt.edge_index, bt.edge_attr.double(), return_attention_weights=True)
        assert torch.equal(ei2.cpu(), ei_ref) and relerr(alpha, a_ref) < TOL
        x = torch.relu(x)


@pytest.mark.parametrize("geom", [(6, 30, 42, 6, 500, False), (5, 30, 7, 8, 24, True), (4, 13, 3, 3, 10, False),
                                  (2, 40, 5, 4, 12, False), (2, 77, 3, 3, 7, True), (1, 300, 4, 6, 16, False),
                                  (1, 40, 50, 2, 8, False)],
                         ids=["default", "H8_cat", "N13", "N40_large", "N77_large_cat", "N300_large", "N40_L50"])
def test_structured_edge_source_layer_parity(cuda_lib, geom):
    """SURVEY 8f-2: a layer given the dataset's window references (spot_windows) reads the [L, N, N] co-volatility
    windows instead of the materialised edge rows.  Same operator, so: outputs, attention coefficients and every
    gradient against the fp64 edge-list oracle on the MATERIALISED batch, to the usual bar."""
    B, N, L, H, C_, concat = geom
    vol, vv = synth.synthetic_matrices(L + B + 3, N, seed=61)
    ds = sv.WindowDataset(vol, vv, seq_length=L, device=DEV, drop_first=1, structured=True)
    idx = list(range(B))
    bt_s = ds.collate(idx)
    assert bt_s.edge_attr is None and bt_s.spot_windows is not None
    bt = synth.make_batch(vol, vv, [i + 1 for i in idx], L)
    ref, ours = make_layers(N * L, C_, H, concat, 3 * L, 0.2, seed=N + L)
    g = torch.Generator().manual_seed(2)
    dout = torch.randn(B * N, H * C_ if concat else C_, generator=g)
    r64, ei2 = oracle_pass(ref, bt, dout, torch.float64, True)
    r32, _ = oracle_pass(ref, bt, dout, torch.float32, True)
    xg = bt_s.x.detach().clone().requires_grad_(True)
    out, (ei2g, alpha) = ours(xg, bt_s.edge_index, None, return_attention_weights=True, topology=bt_s.spot_topology,
                              windows=bt_s.spot_windows)
    out.backward(dout.to(DEV))
    assert torch.equal(ei2g.cpu(), ei2)
    mine = {"out": out.detach(), "alpha": alpha.detach(), "g_x": xg.grad}
    mine.update({"g_" + k: p.grad for k, p in ours.named_parameters()})
    bad = parity_failures(mine, r64, r32)
    assert not bad, bad


@pytest.mark.parametrize("geom", [(6, 30, 42, 6, 500, False), (5, 30, 7, 8, 24, True), (4, 13, 3, 3, 10, False), (3, 30, 4, 3, 20, False)],
                         ids=["default", "H8_cat", "N13", "L4_H3"])
def test_structured_edge_source_stages(cuda_lib, geom):
    """The structured entry points against the generic ones on the same inputs: edge terms from the windows ==
    edge terms the generic forward keeps; forward outputs; dP_aug; dv from the windows == dv from the edge rows."""
    B, N, L, H, C_, concat = geom
    Fin, Fe = 8, 3 * L
    vol, vv = synth.synthetic_matrices(L + B + 2, N, seed=5)
    bt = synth.make_batch(vol, vv, list(range(B)), L)
    ref, _ = make_layers(Fin, C_, H, concat, Fe, 0.2, seed=9, wscale=2.0)
    W, a_s, a_d, We, a_e, bias = [p.detach() for p in (ref.lin_src.weight, ref.att_src, ref.att_dst,
                                                       ref.lin_edge.weight, ref.att_edge, ref.bias)]
    x = torch.randn(B * N, Fin, dtype=torch.float64)
    T = dense_gat.pyg_to_dense_tile(bt.edge_attr.double(), bt.edge_index, B, N)
    fw = dense_gat.dense_forward(x, T, W, a_s, a_d, We, a_e, bias, H, C_, concat, 0.2)
    ldp = cuda_lib.spotv2_gat_ldp(H, C_)
    ldo = H * C_ if concat else C_
    P_aug = torch.zeros(B * N, ldp, device=DEV)
    P_aug[:, :H * C_ + 2 * H] = fw["P_aug"].float().to(DEV)
    topo = sv.topology_from_edge_index(bt.edge_index.to(DEV), B * N)
    ea, v, bg = bt.edge_attr.to(DEV), fw["v"].float().to(DEV).contiguous(), bias.float().to(DEV)
    vv_g = torch.as_tensor(vv).float().to(DEV).contiguous()
    t0 = torch.arange(B, dtype=torch.int32, device=DEV)
    dout = torch.randn(B * N, ldo).to(DEV)
    res = {}
    for mode in (0, 1):
        d = GatDesc(B, N, Fin, Fe, H, C_, N * (N - 1), int(concat), 0.2, ldp, 0, 0, 0.0, mode)
        etb = C.c_size_t()
        check(cuda_lib.spotv2_gat_edge_terms_bytes(C.byref(d), C.byref(etb)), "edge_terms_bytes")
        terms = torch.full((etb.value // 4,), float("nan"), device=DEV)      # every byte the kernels read must be written
        if mode == 1:
            wse = C.c_size_t()
            check(cuda_lib.spotv2_edge_terms_from_windows_workspace_bytes(C.byref(d), C.byref(wse)), "edge_terms ws")
            ws_e = torch.empty(max(wse.value, 1), dtype=torch.uint8, device=DEV)
            check(cuda_lib.spotv2_edge_terms_from_windows(C.byref(d), ptr(vv_g), vv_g.shape[0], L, ptr(t0), ptr(v), ptr(terms),
                                                          ptr(ws_e), wse.value, st()), "edge_terms_from_windows")
        out = torch.empty(B * N, ldo, device=DEV)
        check(cuda_lib.spotv2_gat_attn_fwd(C.byref(d), ptr(P_aug), ptr(ea) if mode == 0 else None,
                                           ptr(topo.table) if mode == 0 else None, ptr(v), ptr(bg), ptr(out), None, ptr(terms),
                                           None, 0, st()), "attn_fwd")
        a, b, c = C.c_size_t(), C.c_size_t(), C.c_size_t()
        check(cuda_lib.spotv2_gat_workspace_bytes(C.byref(d), C.byref(a), C.byref(b), C.byref(c)), "ws")
        ws = torch.empty(b.value, dtype=torch.uint8, device=DEV)
        dP = torch.full((B * N, ldp), float("nan"), device=DEV)
        dv, dbias = torch.zeros(H, Fe, device=DEV), torch.empty(ldo, device=DEV)
        d_terms = torch.full_like(terms, float("nan")) if mode == 1 else None
        check(cuda_lib.spotv2_gat_attn_bwd(C.byref(d), ptr(P_aug), None, ptr(ea) if mode == 0 else None, ptr(terms),
                                           ptr(topo.table) if mode == 0 else None, ptr(v), ptr(dout), ptr(dP), None, None, None,
                                           ptr(dv) if mode == 0 else None, ptr(d_terms), ptr(dbias), ptr(ws), ws.numel(), st()),
              "attn_bwd")
        if mode == 1:
            wsz = C.c_size_t()
            check(cuda_lib.spotv2_windows_dv_workspace_bytes(C.byref(d), C.byref(wsz)), "windows_dv ws")
            ws2 = torch.empty(wsz.value, dtype=torch.uint8, device=DEV)
            check(cuda_lib.spotv2_windows_dv(C.byref(d), ptr(vv_g), vv_g.shape[0], L, ptr(t0), ptr(d_terms), ptr(dv), ptr(ws2),
                                             wsz.value, st()), "windows_dv")
        # the tensor-core operand form of the same gradient
        n_aug_ = H * C_ + 2 * H
        dP16 = torch.zeros(2, B * N, cuda_lib.spotv2_gat_ld16(n_aug_), device=DEV, dtype=torch.float16)
        pblk = torch.zeros(8, device=DEV)
        dv2 = torch.zeros(H, Fe, device=DEV)
        check(cuda_lib.spotv2_gat_attn_bwd(C.byref(d), ptr(P_aug), None, ptr(ea) if mode == 0 else None, ptr(terms),
                                           ptr(topo.table) if mode == 0 else None, ptr(v), ptr(dout), None, ptr(dP16[0]),
                                           ptr(dP16[1]), ptr(pblk), ptr(dv2) if mode == 0 else None, ptr(d_terms), ptr(dbias),
                                           ptr(ws), ws.numel(), st()), "attn_bwd")
        got = pair_value(dP16, pblk, n_aug_, H * C_)
        assert relerr(got[:, :H * C_], dP[:, :H * C_]) < 3e-6 and relerr(got[:, H * C_:], dP[:, H * C_:n_aug_]) < 3e-6, mode
        torch.cuda.synchronize()
        res[mode] = dict(terms=terms.view(B, H, N, 36)[..., :N].clone(), out=out, dP=dP, dv=dv, dbias=dbias)
    off = ~torch.eye(N, dtype=torch.bool, device=DEV)
    g_ref = fw["g"].permute(0, 3, 2, 1).float().to(DEV)              # [b, h, j, i]
    for mode in (0, 1):
        assert relerr(res[mode]["terms"][..., off], g_ref[..., off]) < TOL, mode
    assert relerr(res[1]["out"], fw["out"]) < TOL
    n_aug = H * C_ + 2 * H
    assert relerr(res[1]["dP"][:, :n_aug], res[0]["dP"][:, :n_aug]) < 3e-6
    assert relerr(res[1]["dv"], res[0]["dv"]) < 3e-6 and torch.equal(res[1]["dbias"], res[0]["dbias"])


def test_structured_edge_source_with_attention_dropout(cuda_lib):
    """Same Philox key, same element indexing: the structured and the materialised path drop the same coefficients."""
    N, L, B, H, C_ = 30, 6, 4, 4, 16
    vol, vv = synth.synthetic_matrices(L + B + 2, N, seed=19)
    _, layer = make_layers(N * L, C_, H, False, 3 * L, 0.2, seed=5)
    layer.dropout = 0.25
    layer.train()
    res = []
    for structured in (False, True):
        ds = sv.WindowDataset(vol, vv, seq_length=L, device=DEV, drop_first=0, structured=structured)
        bt = ds.collate(list(range(B)))
        layer.zero_grad()
        torch.manual_seed(11)
        out, (_, alpha) = layer(bt.x, bt.edge_index, bt.edge_attr, return_attention_weights=True, topology=bt.spot_topology,
                                windows=bt.spot_windows if structured else None)
        out.sum().backward()
        res.append((out.detach(), alpha.detach(), {k: p.grad.clone() for k, p in layer.named_parameters()}))
    assert torch.equal(res[0][1] != 0, res[1][1] != 0) and 0.6 < (res[0][1] != 0).float().mean() < 0.9
    assert relerr(res[1][0], res[0][0]) < 3e-6
    for k in res[0][2]:
        assert relerr(res[1][2][k], res[0][2][k]) < 2e-5, k


def test_structured_and_materialised_model_steps_agree(cuda_lib):
    """GATModel on a structured batch (no edge_attr in HBM at all) vs the same batch with edge_attr materialised."""
    N, L, B = 30, 5, 7
    vol, vv = synth.synthetic_matrices(L + B + 2, N, seed=8)
    kw = dict(num_node_features=N * L, num_edge_features=3 * L, num_heads=4, output_node_channels=1,
              dim_hidden_layers=[16, 12], concat_heads=True)
    torch.manual_seed(4)
    model = sv.GATModel(**kw).to(DEV)
    grads = []
    for structured in (False, True):
        ds = sv.WindowDataset(vol, vv, seq_length=L, device=DEV, drop_first=0, structured=structured)
        bt = ds.collate(list(range(B)))
        model.zero_grad()
        loss = torch.nn.functional.mse_loss(model(bt), bt.y_x)
        loss.backward()
        grads.append((loss.item(), {k: p.grad.clone() for k, p in model.named_parameters()}))
    assert abs(grads[0][0] - grads[1][0]) <= 1e-5 * abs(grads[0][0])
    # layer-1 gradients are exact functions of the same activations; layer-0's pass through a ReLU (kinks): 1e-4
    for k in grads[0][1]:
        assert relerr(grads[1][1][k], grads[0][1][k]) < 1e-4, k


@pytest.mark.parametrize("layers", [[20], [16, 12]], ids=["one_layer", "two_layers"])
def test_standardize_on_every_batch_kind_matches_the_oracle_model(cuda_lib, layers):
    """standardize=True (BatchNorm1d(affine=False) on x and on the real edges, utils/models.py:80-82,142-144) without a
    normalising pass over edge_attr: the edge statistics ride into the layers as (mean, scale), from torch sums (a PyG-style
    batch), from the dataset's per-matrix sums (WindowDataset, materialised) or with no edge tensor at all (structured).
    Data with a clear offset (means of 2 .. 3 standard deviations), so the mean's cancellation in the softmax and its
    correction in dv are both exercised.  Loss, every gradient, the running statistics and the eval-mode output against
    OracleGATModel(standardize=True) in fp64."""
    import copy
    N, L, B = 30, 4, 7
    vol, vv = synth.synthetic_matrices(L + B + 2, N, seed=13)
    vol, vv = vol * 0.7 + 2.0, vv * 0.4 + 1.2                # not standardised: that is when the flag is used
    kw = dict(num_node_features=N * L, num_edge_features=3 * L, num_heads=3, output_node_channels=1, dim_hidden_layers=layers,
              concat_heads=True, standardize=True)
    torch.manual_seed(2)
    ref = pyg_gat.OracleGATModel(**kw).double()
    sd0 = {k: v.clone() for k, v in ref.state_dict().items()}           # weights and FRESH running statistics
    bt = synth.make_batch(vol, vv, list(range(B)), L)
    d64 = synth.Batch(x=bt.x.double(), edge_index=bt.edge_index, edge_attr=bt.edge_attr.double())
    ref.train()
    loss_ref = torch.nn.functional.mse_loss(ref(d64), bt.y_x.double())
    loss_ref.backward()
    ref32 = pyg_gat.OracleGATModel(**kw)
    ref32.load_state_dict({k: (v.float() if v.is_floating_point() else v) for k, v in sd0.items()})
    ref32.train()
    torch.nn.functional.mse_loss(ref32(synth.Batch(x=bt.x, edge_index=bt.edge_index, edge_attr=bt.edge_attr)), bt.y_x).backward()
    ref.eval()
    out_eval_ref = ref(d64).detach()                          # eval: the running statistics after ONE training step
    g64 = {k: p.grad for k, p in ref.named_parameters()}
    g32 = {k: p.grad for k, p in ref32.named_parameters()}
    for kind in ("pyg_batch", "materialised", "structured"):
        ours = sv.GATModel(**kw)
        ours.load_state_dict({k: (v.float() if v.is_floating_point() else v) for k, v in sd0.items()})
        ours.to(DEV)
        if kind == "pyg_batch":
            data = copy.deepcopy(bt).to(DEV)
        else:
            ds = sv.WindowDataset(vol, vv, seq_length=L, device=DEV, drop_first=0, structured=kind == "structured")
            data = ds.collate(list(range(B)))
            assert (data.edge_attr is None) == (kind == "structured")
        ours.train()
        loss = torch.nn.functional.mse_loss(ours(data), data.y_x)
        loss.backward()
        assert abs(loss.item() - loss_ref.item()) <= 2e-5 * abs(loss_ref.item()), kind
        bad = parity_failures({k: p.grad for k, p in ours.named_parameters()}, g64, g32)
        assert not bad, (kind, bad)
        for name in ("bnorm_node", "bnorm_edge"):
            mine, want = getattr(ours, name), getattr(ref, name)
            assert relerr(mine.running_mean, want.running_mean) < 1e-5 and relerr(mine.running_var, want.running_var) < 1e-5, (kind, name)
            assert int(mine.num_batches_tracked) == 1
        ours.eval()
        with torch.no_grad():
            assert relerr(ours(data), out_eval_ref) < 2e-5, kind


def test_scale_up_reaches_the_edge_features_on_both_batch_kinds(cuda_lib):
    """train()'s scale_up multiplies x, edge_attr and y_x (5_train_SpotV2Net.py:145-147).  A materialised batch must use
    the scaled edge_attr (never the raw windows), a structured batch gets its window stack scaled: same loss, same
    gradients, and both differ from the un-scaled edge features."""
    from spotv2net_b200.train import _scaled
    N, L, B, SCALE = 30, 5, 6, 4.0
    vol, vv = synth.synthetic_matrices(L + B + 2, N, seed=9)
    torch.manual_seed(3)
    model = sv.GATModel(N * L, 3 * L, 3, 1, [12]).to(DEV)

    def oracle(dtype, edge_scale):
        ref = pyg_gat.OracleGATModel(N * L, 3 * L, 3, 1, [12]).to(dtype)
        ref.load_state_dict({k: v.to(dtype).cpu() for k, v in model.state_dict().items()})
        bt = synth.make_batch(vol, vv, list(range(B)), L)
        bt.x, bt.edge_attr, bt.y_x = bt.x.to(dtype) * SCALE, bt.edge_attr.to(dtype) * edge_scale, bt.y_x.to(dtype) * SCALE
        loss = torch.nn.functional.mse_loss(ref(bt), bt.y_x)
        loss.backward()
        return loss.item(), {k: p.grad for k, p in ref.named_parameters()}

    loss64, g64 = oracle(torch.float64, SCALE)
    _, g32 = oracle(torch.float32, SCALE)
    _, g_unscaled_edges = oracle(torch.float64, 1.0)          # what the round-1 bug computed
    assert relerr(g_unscaled_edges["gat_layers.0.lin_edge.weight"], g64["gat_layers.0.lin_edge.weight"]) > 1e-2
    for structured in (False, True):
        ds = sv.WindowDataset(vol, vv, seq_length=L, device=DEV, drop_first=0, structured=structured)
        bt = _scaled(ds.collate(list(range(B))), SCALE)
        model.zero_grad()
        loss = torch.nn.functional.mse_loss(model(bt), bt.y_x)
        loss.backward()
        assert abs(loss.item() - loss64) <= 1e-5 * abs(loss64)
        bad = parity_failures({k: p.grad for k, p in model.named_parameters()}, g64, g32)
        assert not bad, (structured, bad)


# ------------------------------------------------------------------ full-size properties
def test_full_batch_properties(cuda_lib):
    """B = 4096 at the default geometry (BASELINE config 2).  The oracle cannot run this size, so:
    graphs are independent (a graph's rows equal the small-batch result bit for bit), attention
    rows sum to one, and the weight gradient is additive over a split of the batch."""
    B, N, L, H, C_ = 4096, 30, 42, 6, 500
    Fin, Fe = N * L, 3 * L
    torch.manual_seed(5)
    layer = sv.GATConv(Fin, C_, heads=H, concat=False, edge_dim=Fe).to(DEV)
    g = torch.Generator(device=DEV).manual_seed(1)
    x = torch.randn(B * N, Fin, device=DEV, generator=g)
    ea = torch.randn(B * N * (N - 1), Fe, device=DEV, generator=g)
    ei, topo = sv.batched_topology(B, N, DEV)
    out, (ei2, alpha) = layer(x, ei, ea, return_attention_weights=True)
    sums = torch.zeros(B * N, H, device=DEV).index_add_(0, ei2[1], alpha)
    assert (sums - 1).abs().max() < 1e-5
    dout = torch.randn(out.shape, device=DEV, generator=g)
    out.backward(dout)
    gW = layer.lin_src.weight.grad.clone()
    layer.zero_grad()
    # graph independence + oracle on a few graphs
    pick = [0, 1, 2047, 4095]
    rows = torch.cat([torch.arange(b * N, (b + 1) * N) for b in pick]).to(DEV)
    erow = torch.cat([torch.arange(b * N * (N - 1), (b + 1) * N * (N - 1)) for b in pick]).to(DEV)
    ei_s, _ = sv.batched_topology(len(pick), N, DEV)
    out_s = layer(x[rows], ei_s, ea[erow])
    assert torch.equal(out_s, out[rows])
    ref = pyg_gat.OracleGATConv(Fin, C_, heads=H, concat=False, edge_dim=Fe).double()
    ref.load_state_dict({k: v.double().cpu() for k, v in layer.state_dict().items()})
    out_ref = ref(x[rows].double().cpu(), ei_s.cpu(), ea[erow].double().cpu())
    assert relerr(out_s, out_ref) < TOL
    # additivity of dW over a 2-way split of the batch
    half = B // 2
    ei_h, _ = sv.batched_topology(half, N, DEV)
    acc = torch.zeros_like(gW)
    for s in range(2):
        layer.zero_grad()
        o = layer(x[s * half * N:(s + 1) * half * N], ei_h, ea[s * half * N * (N - 1):(s + 1) * half * N * (N - 1)])
        o.backward(dout[s * half * N:(s + 1) * half * N])
        acc += layer.lin_src.weight.grad
    assert relerr(acc, gW) < TOL


def test_full_batch_gradients_match_chunked_oracle(cuda_lib):
    """B = 4096 at the default geometry: EVERY parameter gradient against the fp64 edge-list oracle.  The oracle
    cannot hold 4096 graphs (2 x 44 GB of PyG intermediates), but its parameter gradients are sums over graphs, so it
    runs in 64 chunks of 64 graphs and autograd accumulates them in fp64.  Covers what the small cases cannot: the
    per-CTA partial reductions of dv / dbias / ds|dd over 4096 graphs on 148 CTAs and the 16-way split-K of the
    weight-gradient GEMM (what the reference does in one pass: 5_train_SpotV2Net.py:150-159), and the input gradient
    (proj_bwd_input on the padded dP pair over 960 row tiles), chunk by chunk."""
    import copy
    B, N, L, H, C_ = 4096, 30, 42, 6, 500
    Fin, Fe, chunk = N * L, 3 * L, 64
    torch.manual_seed(11)
    ref = pyg_gat.OracleGATConv(Fin, C_, heads=H, concat=False, edge_dim=Fe)
    with torch.no_grad():
        ref.bias.normal_()
    ours = sv.GATConv(Fin, C_, heads=H, concat=False, edge_dim=Fe)
    ours.load_state_dict(ref.state_dict())
    ours.to(DEV)
    g = torch.Generator(device=DEV).manual_seed(3)
    x = torch.randn(B * N, Fin, device=DEV, generator=g).requires_grad_()
    ea = torch.randn(B * N * (N - 1), Fe, device=DEV, generator=g)
    dout = torch.randn(B * N, C_, device=DEV, generator=g)
    ei, _ = sv.batched_topology(B, N, DEV)
    out = ours(x, ei, ea)
    out.backward(dout)
    torch.cuda.synchronize()
    ei_c = sv.batched_topology(chunk, N, "cuda:0")[0].cpu()
    torch.set_num_threads(os.cpu_count() or 1)

    def oracle_grads(dtype):
        m = copy.deepcopy(ref).to(dtype)
        worst, worst_dx = 0.0, 0.0
        for c0 in range(0, B, chunk):
            rows, erows = slice(c0 * N, (c0 + chunk) * N), slice(c0 * N * (N - 1), (c0 + chunk) * N * (N - 1))
            xc = x[rows].detach().cpu().to(dtype).requires_grad_()
            o = m(xc, ei_c, ea[erows].cpu().to(dtype))
            o.backward(dout[rows].cpu().to(dtype))            # .grad accumulates over the chunks
            worst = max(worst, relerr(out[rows], o.detach()))
            worst_dx = max(worst_dx, relerr(x.grad[rows], xc.grad))
        return {"g_" + k: p.grad for k, p in m.named_parameters()}, worst, worst_dx

    g64, worst_out, worst_dx = oracle_grads(torch.float64)
    print(f"B=4096 chunked fp64 oracle: worst out error {worst_out:.2e}, worst x.grad error {worst_dx:.2e}")
    assert worst_out < TOL, worst_out
    assert worst_dx < TOL, worst_dx
    mine = {"g_" + k: p.grad for k, p in ours.named_parameters()}
    errs = {k: relerr(mine[k], g64[k]) for k in g64}
    print("B=4096 gradient errors vs the chunked fp64 oracle:", {k: f"{v:.2e}" for k, v in errs.items()})
    bad = {}
    if max(errs.values()) > TOL:        # only then pay for the fp32 oracle (calibrates ill-conditioned sums; whitelisted uses only)
        bad = parity_failures(mine, g64, oracle_grads(torch.float32)[0])
    assert not bad, f"(our error, fp32-oracle error) above the bar at B=4096: {bad}"


# ------------------------------------------------------------------ the caller: training harness
@pytest.mark.parametrize("scale_up", [None, 100.0], ids=["no_scale_up", "scale_up_100"])
def test_training_harness_loss_curve_matches_oracle_loop(cuda_lib, tmp_path, scale_up):
    """spotv2net_b200.train.train (5_train_SpotV2Net.py:23-203 restated) against the same loop run with the
    oracle model on the CPU: same seed, same split, same shuffle, Adam; per-epoch train/test losses agree."""
    from spotv2net_b200.train import train
    N, L, T = 30, 3, 46
    vol, vv = synth.synthetic_matrices(T, N, seed=77)
    p = dict(modelname="t", modeltype="gat", seq_length=L, batch_size=8, dim_hidden_layers=[16], output_node_channels=1,
             num_heads=3, concat_heads=True, activation="relu", optimizer="adam", learning_rate=1e-3, negative_slope=0.2,
             dropout_att=0.0, dropout=0.0, standardize=False, num_epochs=2, tolerance=1e-9, split_proportion=0.8,
             scale_up=scale_up, seed=5)      # scale_up: x, edge_attr AND targets scaled (5_train_SpotV2Net.py:145-147)
    tr, te = train(p=dict(p), vol=vol, volvol=vv, device=DEV, output_root=str(tmp_path), drop_first=2, verbose=False)
    assert os.path.exists(tmp_path / "t_3" / "t_weights_seed_5.pth") and os.path.exists(tmp_path / "t_3" / "test_losses_seed_5.npy")
    # oracle loop, in fp32 (what the reference runs) and in fp64 (the yardstick)
    n = T - L - 2
    n_train = int(0.8 * n)

    def oracle_loop(dtype):
        torch.manual_seed(5)
        model = pyg_gat.OracleGATModel(N * L, 3 * L, 3, 1, [16], concat_heads=True).to(dtype)
        opt = torch.optim.Adam(model.parameters(), lr=1e-3)
        gen = torch.Generator().manual_seed(5)
        crit = torch.nn.MSELoss()
        tr_ref, te_ref = [], []

        def prep(bt):
            s_ = scale_up if scale_up else 1.0
            return synth.Batch(x=(bt.x * s_).to(dtype), edge_index=bt.edge_index, edge_attr=(bt.edge_attr * s_).to(dtype)), (bt.y_x * s_).to(dtype)

        for _ in range(2):
            model.train()
            order = torch.randperm(n_train, generator=gen)
            tot, steps = 0.0, 0
            for s in range(0, n_train, 8):
                bt, y = prep(synth.make_batch(vol, vv, [int(i) + 2 for i in order[s:s + 8]], L))
                loss = crit(model(bt), y)
                opt.zero_grad(); loss.backward(); opt.step()
                tot += loss.item(); steps += 1
            tr_ref.append(tot / steps)
            model.eval()
            tot, nb = 0.0, 0
            with torch.no_grad():
                for s in range(n_train, n, 8):
                    bt, y = prep(synth.make_batch(vol, vv, [i + 2 for i in range(s, min(s + 8, n))], L))
                    tot += crit(model(bt), y).item(); nb += 1
            te_ref.append(tot / nb)
        return np.array(tr_ref), np.array(te_ref), model

    tr32, te32, model = oracle_loop(torch.float32)
    tr64, te64, _ = oracle_loop(torch.float64)
    # The bar is 2e-4 against the fp64 loop (3x the fp32 reference loop's own distance where that is larger).  One exception,
    # measured (tools/pair_model_check.py): with scale_up = 100 every logit is 100x larger, the softmax saturates, and the
    # gradient w.r.t. att_dst - a per-target shift the softmax is invariant to, up to LeakyReLU kinks - is max|dd| = 3.9e-6
    # against max|ds| = 11.5, i.e. ONE fp32 ulp of the dz entries it sums.  Adam normalises that rounding noise into full-size
    # steps of att_dst, which move kinks; from the second epoch on the loss curve of ANY fp32 implementation depends on its
    # summation order at the 1e-3 level (p_format 0 lands at 3e-6, p_format 1 at 8e-4, both with identical per-step
    # gradients to 3e-7 for every other parameter).  So: epoch 1 at the bar, later epochs of the scaled run at 2e-3.
    tr, te = np.array(tr), np.array(te)
    for name, ours_, r32, r64 in (("train", tr, tr32, tr64), ("test", te, te32, te64)):
        err = np.abs(ours_ - r64) / np.abs(r64)
        ref_err = np.abs(r32 - r64) / np.abs(r64)
        bar = np.maximum(2e-4, 3.0 * ref_err)
        if scale_up:
            bar[1:] = np.maximum(bar[1:], 2e-3)
        if (err > 2e-4).any() or os.environ.get("SPOTV2_VERBOSE_TESTS"):
            print(f"training harness [{'scale_up' if scale_up else 'plain'}] {name} loss: ours {err}, fp32 reference loop {ref_err} (relative to the fp64 loop)")
        assert (err <= bar).all(), (name, ours_, r32, r64)
    sd = torch.load(tmp_path / "t_3" / "t_weights_seed_5.pth")
    assert list(sd.keys()) == list(model.state_dict().keys())


# ------------------------------------------------------------------ p_format 1: the projection as an fp16 operand pair
@pytest.mark.parametrize("shape", [(8, 30, 500, 1), (593, 30, 500, 1), (1184, 30, 500, 1), (70, 30, 256, 8), (300, 7, 12, 3), (5, 1, 1024, 1)],
                         ids=lambda s: "B%dN%dC%dupg%d" % s)
def test_dout_operand_pair_prepass(cuda_lib, shape):
    """csrc/attn_prep.cu through spotv2_diag_dout_pair: one pass turns dout into hi | lo planes with one power-of-two
    scale per unit (a graph, or a (graph, head) block of a concat layer), the bias gradient and max|dout|.  Units whose
    magnitudes differ by orders (rows scaled by a random factor) each keep 22 bits; more units than CTAs (593, 1184)."""
    B, N, C_, upg = shape
    ldo = upg * C_
    g = torch.Generator(device=DEV).manual_seed(B)
    dout = torch.randn(B * N, ldo, device=DEV, generator=g) * torch.rand(B, 1, 1, device=DEV, generator=g).expand(B, N, 1).reshape(B * N, 1) ** 4
    ld16 = cuda_lib.spotv2_gat_ld16(ldo)
    planes = torch.zeros(2, B * N, ld16, device=DEV, dtype=torch.float16)
    scales, blk, dbias = torch.zeros(B * upg, device=DEV), torch.zeros(8, device=DEV), torch.zeros(ldo, device=DEV)
    ws = torch.empty(cuda_lib.spotv2_diag_dout_pair_ws_bytes(B, C_, upg), device=DEV, dtype=torch.uint8)
    check(cuda_lib.spotv2_diag_dout_pair(ptr(dout), B, N, C_, upg, ptr(planes[0]), ptr(planes[1]), ld16, ptr(scales), ptr(blk),
                                         ptr(dbias), ptr(ws), st()), "spotv2_diag_dout_pair")
    units = dout.view(B, N, upg, C_)
    umax = units.abs().amax(dim=(1, 3))
    want_s = torch.where(umax > 0, torch.exp2(15 - torch.frexp(umax)[1].float()), torch.ones_like(umax))
    assert torch.equal(scales.view(B, upg), want_s)                                  # amax * scale in [2^14, 2^15): exact rule
    assert (planes[0].float().abs().max() < 32768.5)
    rec = (planes[0, :, :ldo].double() + planes[1, :, :ldo].double()).view(B, N, upg, C_) / scales.view(B, 1, upg, 1).double()
    per_unit = (rec - units.double()).abs().amax(dim=(1, 3)) / umax.double().clamp_min(1e-300)
    assert per_unit.max().item() < 2.0 ** -21                                        # 22 bits relative to EACH unit's maximum
    assert blk.view(torch.int32)[0].item() == units.abs().max().view(torch.int32).item()
    assert relerr(dbias, dout.double().sum(0)) < 2e-6


@pytest.mark.parametrize("geom", [(4, 30, 1260, 6, 500, 0), (3, 30, 90, 3, 16, 0), (2, 30, 2048, 8, 256, 0), (2, 7, 33, 5, 12, 0), (4, 30, 1260, 8, 256, 3)],
                         ids=lambda g_: "B%dN%dF%dH%dC%dalgo%d" % g_)
def test_projection_as_an_operand_pair(cuda_lib, geom):
    """spotv2_proj_fwd_pair: P never exists in fp32 - the GEMM epilogue emits hi | lo planes in the padded head pitch with
    the a-priori scale (max|x| * row-L1 bound), and the logit terms s | d in fp32 beside them.  Against an fp64 matmul:
    hi + lo to 1e-5 of max|P| (fp32 class) or 2e-3 (half class: hi plane only), pad columns exactly zero, the bound holds."""
    B, N, Fin, H, C_, algo = geom
    n = B * N
    d = GatDesc(B, N, Fin, 0, H, C_, 0, 0, 0.2, cuda_lib.spotv2_gat_ldp(H, C_), algo, 0, 0.0, 0, 0, 0, 1)
    Cp, n_aug = cuda_lib.spotv2_gat_head_pitch(C.byref(d)), cuda_lib.spotv2_gat_n_aug(C.byref(d))
    assert Cp % 8 == 0 and Cp >= C_ and n_aug == H * Cp + 2 * H
    g = torch.Generator(device=DEV).manual_seed(Fin)
    x = torch.randn(n, Fin, device=DEV, generator=g) * 3.0
    W = torch.randn(H * C_, Fin, device=DEV, generator=g) * 0.05
    a_s, a_d = torch.randn(1, H, C_, device=DEV, generator=g), torch.randn(1, H, C_, device=DEV, generator=g)
    W_aug = torch.empty(n_aug, Fin, device=DEV)
    check(cuda_lib.spotv2_gat_fold(C.byref(d), ptr(W), ptr(a_s), ptr(a_d), None, None, ptr(W_aug), None, st()), "fold")
    Wv = W_aug[:H * Cp].view(H, Cp, Fin)
    assert torch.equal(Wv[:, :C_].reshape(H * C_, Fin), W) and (Wv[:, C_:] == 0).all()      # padded rows are zero rows
    ldx = cuda_lib.spotv2_gat_ld16(Fin)
    x16, xblk = torch.empty(2, n, ldx, device=DEV, dtype=torch.float16), torch.empty(8, device=DEV)
    check(cuda_lib.spotv2_split_f16(ptr(x), n, Fin, Fin, 0, 0, ptr(x16[0]), ptr(x16[1]), ldx, ptr(xblk), st()), "split_f16")
    ldp16 = cuda_lib.spotv2_gat_ld16(n_aug)
    P16 = torch.full((2, n, ldp16), float("nan"), device=DEV, dtype=torch.float16)
    pblk, sd = torch.empty(8, device=DEV), torch.empty(n, 2 * H, device=DEV)
    a_, _, _ = (C.c_size_t(), C.c_size_t(), C.c_size_t())
    check(cuda_lib.spotv2_gat_workspace_bytes(C.byref(d), C.byref(a_), None, None), "ws")
    ws = torch.empty(a_.value, device=DEV, dtype=torch.uint8)
    check(cuda_lib.spotv2_proj_fwd_pair(C.byref(d), ptr(x16[0]), ptr(x16[1]), ptr(xblk), ptr(W_aug), ptr(P16[0]),
                                        ptr(P16[1]) if algo != 3 else None, ptr(pblk), ptr(sd), ptr(ws), ws.numel(), st()), "proj_fwd_pair")
    ref = x.double() @ W_aug.double().t()                                             # [n, n_aug]
    full = P16[0, :, :n_aug].double() + (P16[1, :, :n_aug].double() if algo != 3 else 0.0)
    P = full[:, :H * Cp] * pblk[2].double()
    tol = 2e-3 if algo == 3 else TOL
    assert relerr(P, ref[:, :H * Cp]) < tol
    assert (full[:, :H * Cp].view(n, H, Cp)[:, :, C_:] == 0).all()                    # pad columns: exact zeros
    assert relerr(sd, ref[:, H * Cp:]) < tol                                          # fp32 logit terms
    assert relerr(full[:, H * Cp:] * pblk[3].double(), ref[:, H * Cp:]) < tol         # and their copy in the planes' second group
    bound = pblk[:2].double()
    assert ref[:, :H * Cp].abs().max() <= bound[0] and ref[:, H * Cp:].abs().max() <= bound[1]
    assert (full.abs().max() < 32768.0) and float(pblk[4]) * float(pblk[2]) == 1.0


@pytest.mark.parametrize("case", [(6, 30, 1260, 126, 6, 500, False), (5, 30, 64, 126, 8, 256, True), (4, 13, 9, 5, 3, 8, True), (7, 30, 90, 9, 3, 16, True),
                                  (3, 30, 40, 0, 4, 36, False), (3, 17, 40, 360, 2, 64, True), (300, 32, 24, 200, 8, 72, False), (2, 2, 8, 4, 2, 1024, False)],
                         ids=lambda c: "B%dN%dF%dFe%dH%dC%d%s" % (c[:6] + ("cat" if c[6] else "mean",)))
def test_both_projection_formats_agree(cuda_lib, case, monkeypatch):
    """One layer step with P as fp32 (p_format 0) and as the operand pair (p_format 1): same operator, same logits (the
    s | d terms and the edge terms are bit-identical by construction, so every LeakyReLU kink falls on the same side),
    outputs and gradients equal to fp32 rounding."""
    from spotv2net_b200 import gat_conv
    B, N, Fin, Fe, H, C_, concat = case
    torch.manual_seed(B)
    layer = sv.GATConv(Fin, C_, heads=H, concat=concat, edge_dim=Fe or None).to(DEV)
    g = torch.Generator(device=DEV).manual_seed(1)
    x0 = torch.randn(B * N, Fin, device=DEV, generator=g)
    ea = torch.randn(B * N * (N - 1), Fe, device=DEV, generator=g) if Fe else None
    dout = torch.randn(B * N, H * C_ if concat else C_, device=DEV, generator=g)
    ei, _ = sv.batched_topology(B, N, DEV)
    res = {}
    for pf in (0, 1):
        monkeypatch.setattr(gat_conv, "P_FORMAT", pf)
        layer.zero_grad()
        x = x0.clone().requires_grad_()
        out = layer(x, ei, ea)
        out.backward(dout)
        res[pf] = dict(out=out.detach(), dx=x.grad, **{k: p.grad.clone() for k, p in layer.named_parameters() if p.grad is not None})
    d = gat_conv._desc(sv.batched_topology(B, N, DEV)[1], Fin, Fe, H, C_, concat, 0.2)
    assert d.p_format == 1, "the library should have chosen the pair format for this shape"
    for k in res[0]:
        assert relerr(res[1][k], res[0][k]) < 2e-6, k


@pytest.mark.parametrize("geom", [(5, 30, 64, 126, 6, 500, False), (3, 13, 16, 5, 3, 8, True), (2, 32, 24, 40, 8, 72, False)],
                         ids=lambda g_: "B%dN%dF%dFe%dH%dC%d%s" % (g_[:6] + ("cat" if g_[6] else "mean",)))
def test_forward_record_for_the_backward(cuda_lib, geom):
    """p_format 1 without attention dropout: what spotv2_gat_attn_fwd_pair leaves in edge_terms is its attention
    coefficients ([B, H, j, 36] tile rows, target i inside a row) with the LeakyReLU side of the logit in the sign bit -
    the backward redoes neither logits nor softmax.  |record| must be the returned alpha bit for bit, the signs those of
    the fp64 oracle's logits (away from the kink), pad columns zero; with dropout the record is the edge terms."""
    B, N, Fin, Fe, H, C_, concat = geom
    bt = synth.random_complete_batch(B, N, Fin, Fe, seed=11)
    ref, _ = make_layers(Fin, C_, H, concat, Fe, 0.2, seed=5, wscale=1.5)
    W, a_s, a_d, We, a_e, bias = [p.detach() for p in (ref.lin_src.weight, ref.att_src, ref.att_dst,
                                                       ref.lin_edge.weight, ref.att_edge, ref.bias)]
    T = dense_gat.pyg_to_dense_tile(bt.edge_attr.double(), bt.edge_index, B, N)
    fw = dense_gat.dense_forward(bt.x.double(), T, W, a_s, a_d, We, a_e, bias, H, C_, concat, 0.2)
    n = B * N
    topo = sv.topology_from_edge_index(bt.edge_index.to(DEV), n)
    for pdrop in (0.0, 0.25):
        d = GatDesc(B, N, Fin, Fe, H, C_, N * (N - 1), int(concat), 0.2, cuda_lib.spotv2_gat_ldp(H, C_), 0, 0, pdrop, 0, 7, 0, 1)
        assert cuda_lib.spotv2_gat_pair_format_supported(C.byref(d)) == 1
        Cp, n_aug = cuda_lib.spotv2_gat_head_pitch(C.byref(d)), cuda_lib.spotv2_gat_n_aug(C.byref(d))
        W_aug, v = torch.empty(n_aug, Fin, device=DEV), torch.empty(H, Fe, device=DEV)
        Wg, asg, adg, Weg, aeg, bg = [t_.float().to(DEV).contiguous() for t_ in (W, a_s, a_d, We, a_e, bias)]
        check(cuda_lib.spotv2_gat_fold(C.byref(d), ptr(Wg), ptr(asg), ptr(adg), ptr(Weg), ptr(aeg), ptr(W_aug), ptr(v), st()), "fold")
        x, ea = bt.x.to(DEV), bt.edge_attr.to(DEV)
        ldx = cuda_lib.spotv2_gat_ld16(Fin)
        x16, xblk = torch.empty(2, n, ldx, device=DEV, dtype=torch.float16), torch.empty(8, device=DEV)
        check(cuda_lib.spotv2_split_f16(ptr(x), n, Fin, Fin, 0, 0, ptr(x16[0]), ptr(x16[1]), ldx, ptr(xblk), st()), "split_f16")
        ldp16 = cuda_lib.spotv2_gat_ld16(n_aug)
        P16 = torch.zeros(2, n, ldp16, device=DEV, dtype=torch.float16)
        pblk, sd = torch.empty(8, device=DEV), torch.empty(n, 2 * H, device=DEV)
        a_ = C.c_size_t()
        check(cuda_lib.spotv2_gat_workspace_bytes(C.byref(d), C.byref(a_), None, None), "ws")
        ws = torch.empty(a_.value, device=DEV, dtype=torch.uint8)
        check(cuda_lib.spotv2_proj_fwd_pair(C.byref(d), ptr(x16[0]), ptr(x16[1]), ptr(xblk), ptr(W_aug), ptr(P16[0]), ptr(P16[1]),
                                            ptr(pblk), ptr(sd), ptr(ws), ws.numel(), st()), "proj_fwd_pair")
        etb = C.c_size_t()
        check(cuda_lib.spotv2_gat_edge_terms_bytes(C.byref(d), C.byref(etb)), "edge_terms_bytes")
        rec = torch.full((etb.value // 4,), float("nan"), device=DEV)
        out = torch.empty(n, H * C_ if concat else C_, device=DEV)
        alpha = torch.empty(B, H, N, N, device=DEV)
        check(cuda_lib.spotv2_gat_attn_fwd_pair(C.byref(d), ptr(P16[0]), ptr(P16[1]), ptr(pblk), ptr(sd), ptr(ea),
                                                ptr(topo.table), ptr(v), ptr(bg), ptr(out), ptr(alpha), ptr(rec), st()),
              "attn_fwd_pair")
        torch.cuda.synchronize()
        rec = rec.view(B, H, N, 36)
        assert torch.isfinite(rec).all()                                               # every byte of the record is written
        g64 = fw["g"].permute(0, 3, 2, 1)                                              # edge terms [B, H, j, i]
        off = ~torch.eye(N, dtype=torch.bool)
        if pdrop > 0:
            assert relerr(rec[..., :N].cpu()[..., off], g64[..., off]) < TOL           # dropout: the edge terms, as before
            continue
        assert relerr(out, fw["out"]) < TOL
        assert torch.equal(rec[..., :N].abs(), alpha)                                  # the coefficients, bit for bit
        assert (rec[..., N:] == 0).all()
        z = fw["z"].permute(0, 3, 2, 1)                                                # logits [B, H, j, i]
        clear = z.abs() > 1e-4 * z.abs().max()
        neg = torch.signbit(rec[..., :N]).cpu()
        assert torch.equal(neg[clear], (z <= 0)[clear])
        assert 0.05 < neg.float().mean() < 0.95                                        # both sides occur
