"""The large-graph attention path (N > 32: csrc/attn_large.cu, the batched GEMMs of csrc/gemm_simt.cu and the N > 32 half
of csrc/windows.cu) stage by stage against float64, with several graphs per batch and every error taken per graph.

The path spreads one graph over many CTAs.  Which kernels run depends on the shape (lg_plan and attn_large_bwd):
  - the ring chunk CR of the edge-row passes: 64 rows, shrunk to 48, 32 or 16 when two stages and v's MMA fragments
    exceed 110 KB of shared memory (Fe of about 200 and more);
  - the dv kernel lg_dv_kernel<KPT, RG>, KPT = ceil(Fe / 128): <1, 4>, <2, 2> or <4, 1>;
  - the copy into the ring: 1-D bulk copies when the edge block is 16-byte aligned and R Fe % 4 == 0, else the
    cooperative copies (lg_copy and the inline copy of lg_dv_kernel);
  - the batched GEMMs: 3xTF32 mma.sync (gemm_algo 0) or exact-fp32 FFMA2 (gemm_algo 1).
GEOMS reaches every one of them; test_plan_coverage_of_the_geometry_grid restates the rules and says which variant the
grid no longer reaches if they change.

Operands are plain fp32 and the reference (tests/test_half_precision.py dense_attention, on the device in float64) runs
on exactly those values.  Each graph's P rows and dout rows carry their own power of two, per (graph, head) for concat
layers, and every error is max over units of |ours_u - ref_u|_inf / |ref_u|_inf (unit = graph, or (graph, head) for
concat layers) against the project's 1e-5, so that a fault confined to one graph cannot hide under another graph's
larger values.  Two quantities cancel by construction and are measured against the magnitude of what they sum:
  dd_i = sum_j dz_ij   (a softmax row's gradient sums to zero before the LeakyReLU factor): against max_i sum_j |dz_ij|
  dz'_ij = dz_ij + dz_ii / (N - 1):                        against max |dz_ij| + |dz_ii| / (N - 1)
"""
import ctypes as C
import math
from collections import namedtuple
from pathlib import Path

import pytest
import torch

import spotv2net_b200 as sv
from spotv2net_b200._lib import GatDesc, check, ptr
from oracle import dense_gat, synth
from test_half_precision import dense_attention, dense_logits, workspace
from test_pair_format_stages import keep_mask, per_graph

DEV = "cuda:0"
TOL = 1e-5
PAIR_TOL = 3e-6                # the fp16-pair dP output against the fp32 one (22 bits of each group's scale)
SEED_LO, SEED_HI = 0x2468ACE, 0x13579BDF
CSRC = Path(__file__).resolve().parent.parent / "spotv2net_b200" / "csrc"

Geom = namedtuple("Geom", "B N Fe H C concat pdrop rows", defaults=(0.0, "pyg"))
# rows: "pyg" = the N (N - 1) real edges in PyG order; "loops" = N^2 rows, the input's self loops (skipped rows) at
# scattered positions of a permuted edge order; "dense" = the dense target-major tile with a garbage diagonal
GEOMS = [
    Geom(3, 33, 200, 7, 12, True),              # CR 48, <2,2>
    Geom(2, 77, 129, 1, 33, True),              # CR 64 with <2,2>, H = 1, a ragged last chunk (5852 = 91 * 64 + 28)
    Geom(4, 64, 256, 8, 16, False),             # CR 32, <2,2>, H = 8
    Geom(2, 131, 257, 3, 20, False),            # cooperative copies (R Fe % 4 == 2), CR 32, <4,1>
    Geom(2, 131, 5, 4, 9, False),               # cooperative copies with <1,4>
    Geom(2, 129, 360, 6, 128, True),            # CR 16, <4,1>, one past the 128-row GEMM tile, C exactly one tile
    Geom(3, 127, 512, 8, 8, False),             # Fe at its limit, KS = 64
    Geom(2, 200, 0, 6, 40, False),              # no edge_attr: the softmax without edge terms
    Geom(3, 500, 126, 6, 500, False),           # BASELINE config D's layer, several graphs
    Geom(3, 40, 7, 5, 12, False, 0.0, "loops"),  # input self loops, odd Fe (bulk copies: R Fe % 4 == 0)
    Geom(2, 131, 33, 3, 16, True, 0.0, "loops"),  # input self loops, odd Fe and odd R: cooperative copies
    Geom(2, 64, 12, 6, 10, False, 0.0, "dense"),  # spotv2_edge_table_dense, garbage on the diagonal
    Geom(2, 77, 129, 1, 33, True, 0.3),         # attention dropout
    Geom(2, 77, 129, 1, 33, True, 0.9),
    Geom(2, 500, 126, 6, 40, False, 0.3),
    Geom(2, 500, 126, 6, 40, False, 0.9),
]
GEMM_ALGOS = (0, 1)             # batched GEMMs: 3xTF32 bgemm_tc_kernel, exact-fp32 FFMA2 bgemm_kernel


def geom_id(g):
    return (f"B{g.B}N{g.N}Fe{g.Fe}H{g.H}C{g.C}{'cat' if g.concat else 'mean'}" + (f"_p{g.pdrop:g}" if g.pdrop else "")
            + ("" if g.rows == "pyg" else "_" + g.rows))


# ======================================================================================== the plan, restated
def round_up(x, a):
    return (x + a - 1) // a * a


def lg_plan(Fe, H):
    """lg_plan (csrc/attn_large.cu): (KS, CR) of the edge-row ring, None for a layer without edge features."""
    if Fe <= 0:
        return None
    KS = ((Fe + 7) // 8 + 7) // 8 * 8
    NT = (H + 7) // 8
    off_stage = round_up(128 + NT * KS * 32 * 16, 128)
    CR = 64
    while CR > 16 and off_stage + 2 * round_up(CR * Fe * 4, 128) > 110 * 1024:
        CR -= 16
    return KS, CR


def dv_kernel(Fe):
    """lg_dv_kernel<KPT, RG> that attn_large_bwd launches: KPT = ceil(Fe / 128)."""
    kpt = (Fe + 127) // 128
    return (1, 4) if kpt <= 1 else (2, 2) if kpt <= 2 else (4, 1)


def rows_per_graph(g):
    return g.N * g.N if g.rows in ("loops", "dense") else g.N * (g.N - 1)


def bulk_ok(g):
    """attn_params_of (csrc/attn_bwd.cu): bulk copies when the edge block is 16-byte aligned (every buffer these tests
    allocate is) and R Fe % 4 == 0."""
    return g.Fe > 0 and rows_per_graph(g) * g.Fe % 4 == 0


# the source lines restated above: if one of them changes, the restatement (and what the grid reaches) needs a new look
RESTATED = {
    "attn_large.cu": [
        "pl.KS = ((p.Fe + 7) / 8 + 7) / 8 * 8;",
        "pl.NT = (p.H + 7) / 8;",
        "const size_t vfrag = (size_t)pl.NT * pl.KS * 32 * 16;",
        "pl.off_stage = (uint32_t)round_up(128 + vfrag, 128);",
        "pl.CR = 64;",
        "while (pl.CR > 16 && pl.off_stage + 2 * round_up((size_t)pl.CR * p.Fe * 4, 128) > 110 * 1024) pl.CR -= 16;",
        "const int kpt = (p.Fe + kLgThreads - 1) / kLgThreads;",
        "if (kpt <= 1) rc = launch(lg_dv_kernel<1, 4>, 4);",
        "else if (kpt <= 2) rc = launch(lg_dv_kernel<2, 2>, 2);",
        "else rc = launch(lg_dv_kernel<4, 1>, 1);",
        "constexpr int kLgThreads = 128;",
        "g.tensor_cores = p.lg_tensor_cores;",
    ],
    "attn_bwd.cu": [
        "p.bulk_ok = d->Fe > 0 && aligned16(e.rows) && ((size_t)d->R * d->Fe) % 4 == 0;",
        "p.lg_tensor_cores = d->gemm_algo != 1;",
    ],
}


def test_plan_coverage_of_the_geometry_grid():
    """Without a device: the grid reaches CR 16, 32, 48 and 64, all three dv kernels, both copy paths, a layer without
    edge features and both batched-GEMM back ends; the restated rules are still the library's."""
    for src, lines in RESTATED.items():
        text = " ".join((CSRC / src).read_text().split())
        changed = [ln for ln in lines if " ".join(ln.split()) not in text]
        assert not changed, f"{src} no longer holds these lines restated by this test: {changed}"
    assert [lg_plan(Fe, 6)[1] for Fe in (126, 190, 200, 230, 256, 257, 300, 360, 384, 512)] == \
        [64, 64, 48, 48, 32, 32, 32, 16, 16, 16]
    assert lg_plan(512, 8)[0] == 64
    edge = [g for g in GEOMS if g.Fe > 0]
    reached = {
        "CR": {lg_plan(g.Fe, g.H)[1] for g in edge},
        "dv kernel": {dv_kernel(g.Fe) for g in edge},
        "bulk copies": {bulk_ok(g) for g in edge},
        "no edge features": {g.Fe == 0 for g in GEOMS},
        "gemm_algo": set(GEMM_ALGOS),
        "row source": {g.rows for g in GEOMS},
        "dropout": {g.pdrop > 0 for g in GEOMS},
    }
    wanted = {
        "CR": {16, 32, 48, 64},
        "dv kernel": {(1, 4), (2, 2), (4, 1)},
        "bulk copies": {True, False},
        "no edge features": {True, False},
        "gemm_algo": {0, 1},
        "row source": {"pyg", "loops", "dense"},
        "dropout": {True, False},
    }
    missing = {k: sorted(wanted[k] - reached[k], key=str) for k in wanted if wanted[k] - reached[k]}
    assert not missing, f"variants of the large-graph path the grid no longer reaches: {missing}"
    # a partial last chunk (rows % 16 != 0) under the 16-row MMA tiles of the logit kernel, with each copy path
    partial = {bulk_ok(g) for g in edge if rows_per_graph(g) % lg_plan(g.Fe, g.H)[1] % 16}
    assert partial == {True, False}
    assert all(g.N > 32 for g in GEOMS) and max(g.N for g in GEOMS) == 500


# ======================================================================================== one geometry end to end
def st():
    return torch.cuda.current_stream().cuda_stream


def units(t, B, U, node_major):
    """Rows of the error groups: [B, N, H, ...] (node_major) or [B, H, ...] -> [B * U, -1], U = H for concat layers (one
    group per (graph, head)), 1 for head-mean layers (one group per graph)."""
    if U == 1:
        return t.reshape(B, -1)
    if node_major:
        t = t.reshape(B, t.shape[1], U, -1).transpose(1, 2)
    return t.reshape(B * U, -1)


class LargeCase:
    """fp32 operands of one geometry, the row table, and the float64 reference on the device."""

    def __init__(self, cuda_lib, g, seed=0):
        self.g = g
        B, N, Fe, H, C_, concat = g.B, g.N, g.Fe, g.H, g.C, g.concat
        n = self.n = B * N
        self.R = R = rows_per_graph(g)
        self.U = U = H if concat else 1
        self.HC, self.ldo = H * C_, (H * C_ if concat else C_)
        self.ldp = cuda_lib.spotv2_gat_ldp(H, C_)
        gen = self.gen = torch.Generator(device=DEV).manual_seed(7919 * seed + 31 * N + Fe + H)
        # per-unit exponents of P (k) and dout (m): one unit at each end of [-8, 8]
        k = torch.randint(-8, 9, (B, U), generator=gen, device=DEV)
        m = torch.randint(-8, 9, (B, U), generator=gen, device=DEV)
        k[0, 0], k[-1, -1], m[0, -1], m[-1, 0] = 8, -8, -8, 8
        self.k, self.m = k, m
        P = torch.randn(B, N, H, C_, generator=gen, device=DEV) * torch.exp2(k.float()).view(B, 1, U, 1)
        self.P64 = P.double()
        # edge rows, the row table and the fp64 target-major tile T[b, i, j] (edge j -> i)
        if Fe and g.rows == "dense":
            T = torch.randn(B, N, N, Fe, generator=gen, device=DEV)
            T += 1e6 * torch.eye(N, device=DEV).view(1, N, N, 1)              # the diagonal must be ignored
            self.ea = T.reshape(B * R, Fe).contiguous()
            self.table = torch.empty(R, dtype=torch.int32, device=DEV)
            check(cuda_lib.spotv2_edge_table_dense(N, ptr(self.table), st()), "edge_table_dense")
            self.T = T.double()
        elif Fe:
            local = synth.complete_graph_edge_index(N).to(DEV)
            if g.rows == "loops":
                loops = torch.arange(N, device=DEV).view(1, N).expand(2, N)
                local = torch.cat([local, loops], 1)
                local = local[:, torch.randperm(R, generator=gen, device=DEV)]      # skipped rows all over the ring
            self.edge_index = torch.cat([local + b * N for b in range(B)], 1).contiguous()
            topo = sv.topology_from_edge_index(self.edge_index, n)
            assert (topo.B, topo.N, topo.R, topo.has_skips) == (B, N, R, g.rows == "loops")
            self.table = topo.table
            self.ea = torch.randn(B * R, Fe, generator=gen, device=DEV)
            if g.rows == "loops":                                             # loud values on the skipped rows
                is_loop = (local[0] == local[1]).repeat(B)
                self.ea[is_loop] *= 50.0
            self.T = dense_gat.pyg_to_dense_tile(self.ea.double(), self.edge_index, B, N)
        else:
            self.ea, self.table, self.T = None, None, None
        self.v = (torch.randn(H, Fe, generator=gen, device=DEV) / math.sqrt(Fe)).contiguous() if Fe else None
        # s | d, with no logit within fp32 noise of the LeakyReLU kink (the backward's slope would differ there)
        sd = torch.randn(n, 2 * H, generator=gen, device=DEV)
        for _ in range(12):
            z = self.logits(sd)
            near = (z.abs() < 2e-5 * z.abs().max()).any(2).view(n, H)
            if not near.any():
                break
            sd[:, H:][near] += 1e-4 * z.abs().max().item()
        z = self.logits(sd)
        assert not (z.abs() < 2e-5 * z.abs().max()).any(), "a logit is left at the LeakyReLU kink"
        self.sd = sd
        self.P_aug = torch.full((n, self.ldp), float("nan"), device=DEV)        # padding columns may hold anything
        self.P_aug[:, :self.HC] = P.reshape(n, self.HC)
        self.P_aug[:, self.HC:self.HC + 2 * H] = sd
        self.bias = torch.randn(self.ldo, generator=gen, device=DEV)
        dout = torch.randn(B, N, U, self.ldo // U, generator=gen, device=DEV) * torch.exp2(m.float()).view(B, 1, U, 1)
        self.dout = dout.reshape(n, self.ldo).contiguous()
        self.keep = keep_mask(B, H, N, g.pdrop, SEED_LO, SEED_HI) if g.pdrop > 0 else None       # [b, h, i, j]
        self.off = ~torch.eye(N, dtype=torch.bool, device=DEV)

    def desc(self, algo, B=None):
        g = self.g
        return GatDesc(B or g.B, g.N, 16, g.Fe, g.H, g.C, self.R, int(g.concat), 0.2, self.ldp, algo, 0, g.pdrop, 0,
                       SEED_LO, SEED_HI, 0)

    def logits(self, sd):
        B, N, H = self.g.B, self.g.N, self.g.H
        return dense_logits(sd[:, :H].double().view(B, N, H), sd[:, H:].double().view(B, N, H), self.T,
                            self.v.double() if self.v is not None else None)

    def reference(self, G=None):
        """G: d_alpha [B, H, j, i] of the _dalpha backward, or None."""
        B, N, H = self.g.B, self.g.N, self.g.H
        mask = self.keep.permute(0, 2, 3, 1) if self.keep is not None else None             # [b, i, j, h]
        return dense_attention(self.P64, self.sd[:, :H].double().view(B, N, H), self.sd[:, H:].double().view(B, N, H),
                               self.T, self.v.double() if self.v is not None else None, self.bias.double(),
                               self.dout.double(), H, self.g.concat, 0.2, mask, 1.0 / (1.0 - self.g.pdrop),
                               d_alpha=None if G is None else G.double().permute(0, 3, 2, 1))

    def edge_terms(self):
        """<e_ij, v_h> in the tile layout [B, H, j, i] (fp64)."""
        return torch.einsum("bijf,hf->bhji", self.T, self.v.double())

    def d_alpha(self):
        """A gradient through the returned coefficients of the size of g dO P^T in every unit, [B, H, j, i]."""
        g = self.g
        s = torch.exp2((self.k + self.m).float()) * math.sqrt(g.C) / (1 if g.concat else g.H)
        s = s.view(g.B, self.U, 1, 1).expand(g.B, g.H, 1, 1) if g.concat else s.view(g.B, 1, 1, 1)
        return (torch.randn(g.B, g.H, g.N, g.N, generator=self.gen, device=DEV) * s).contiguous()

    # -------------------------------------------------------------------------------------------- the calls
    def forward(self, cuda_lib, algo, keep_alpha=True, keep_terms=True, B=None, P_aug=None, ea=None):
        """attn_fwd with NaN-prefilled outputs; without alpha the attention tile lives in a workspace."""
        g = self.g
        B = B or g.B
        d = self.desc(algo, B)
        P_aug = self.P_aug if P_aug is None else P_aug
        ea = self.ea if ea is None else ea
        out = torch.full((B * g.N, self.ldo), float("nan"), device=DEV)
        alpha = torch.full((B, g.H, g.N, g.N), float("nan"), device=DEV) if keep_alpha else None
        terms = torch.full((B, g.H, g.N, g.N), float("nan"), device=DEV) if keep_terms and g.Fe else None
        if terms is not None:
            etb = C.c_size_t()
            check(cuda_lib.spotv2_gat_edge_terms_bytes(C.byref(d), C.byref(etb)), "edge_terms_bytes")
            assert etb.value == terms.numel() * 4
        ws = None
        if alpha is None:
            wsb = C.c_size_t()
            check(cuda_lib.spotv2_gat_attn_fwd_workspace_bytes(C.byref(d), C.byref(wsb)), "attn_fwd_workspace_bytes")
            assert wsb.value >= B * g.H * g.N * g.N * 4
            ws = torch.empty(wsb.value, dtype=torch.uint8, device=DEV)
        check(cuda_lib.spotv2_gat_attn_fwd(C.byref(d), ptr(P_aug), ptr(ea), ptr(self.table), ptr(self.v), ptr(self.bias),
                                           ptr(out), ptr(alpha), ptr(terms), ptr(ws), ws.numel() if ws is not None else 0,
                                           st()), "attn_fwd")
        torch.cuda.synchronize()
        return dict(out=out, alpha=alpha, terms=terms)

    def backward(self, cuda_lib, algo, terms=None, G=None, pair=False, B=None, P_aug=None, ea=None, dout=None):
        """attn_bwd (or attn_bwd_dalpha with G) with NaN-prefilled outputs; terms: the forward's edge terms, or None to
        recompute them from the edge rows; pair: dP as the fp16 pair instead of fp32."""
        g = self.g
        B = B or g.B
        n, H, Fe = B * g.N, g.H, g.Fe
        d = self.desc(algo, B)
        P_aug = self.P_aug if P_aug is None else P_aug
        ea = self.ea if ea is None else ea
        dout = self.dout if dout is None else dout
        dP, dP16, dblk = None, None, None
        if pair:
            dP16 = torch.full((2, n, cuda_lib.spotv2_gat_ld16(self.HC + 2 * H)), float("nan"), device=DEV, dtype=torch.float16)
            dblk = torch.full((8,), float("nan"), device=DEV)
        else:
            dP = torch.full((n, self.ldp), float("nan"), device=DEV)
        dv = torch.full((H, Fe), float("nan"), device=DEV) if Fe else None
        d_et = torch.full((B, H, g.N, g.N), float("nan"), device=DEV) if Fe else None
        dbias = torch.full((self.ldo,), float("nan"), device=DEV)
        ws = workspace(cuda_lib, d)
        args = [C.byref(d), ptr(P_aug), None, ptr(ea), ptr(terms), ptr(self.table), ptr(self.v), ptr(dout), ptr(dP),
                ptr(dP16[0]) if pair else None, ptr(dP16[1]) if pair else None, ptr(dblk), ptr(dv), ptr(d_et), ptr(dbias),
                ptr(ws), ws.numel(), st()]
        if G is None:
            check(cuda_lib.spotv2_gat_attn_bwd(*args), "attn_bwd")
        else:
            check(cuda_lib.spotv2_gat_attn_bwd_dalpha(*args, ptr(G)), "attn_bwd_dalpha")
        torch.cuda.synchronize()
        return dict(dP=dP, dP16=dP16, dblk=dblk, dv=dv, d_et=d_et, dbias=dbias)

    # ------------------------------------------------------------------------------------------------ checks
    def check_forward(self, f, r):
        g, B, U = self.g, self.g.B, self.U
        errs = {}
        assert torch.isfinite(f["out"]).all() and torch.isfinite(f["alpha"]).all()
        if self.keep is not None:
            assert torch.equal(f["alpha"] != 0, self.keep.transpose(2, 3)), "dropout mask differs from its documented layout"
        errs["alpha"] = per_graph(units(f["alpha"], B, U, False), units(r["alpha"].permute(0, 3, 2, 1), B, U, False), B * U)
        errs["out"] = per_graph(units(f["out"].view(B, g.N, -1), B, U, True), units(r["out"].view(B, g.N, -1), B, U, True),
                                B * U)
        if g.Fe:
            got = f["terms"][..., self.off]
            assert torch.isfinite(got).all()
            errs["edge terms"] = per_graph(units(got, B, U, False), units(self.edge_terms()[..., self.off], B, U, False), B * U)
        return errs

    def check_backward(self, bw, r):
        g, B, U, N, H, HC = self.g, self.g.B, self.U, self.g.N, self.g.H, self.HC
        dP = bw["dP"]
        assert torch.isfinite(dP[:, :HC + 2 * H]).all()
        errs = {}
        errs["dP"] = per_graph(units(dP[:, :HC].view(B, N, -1), B, U, True), units(r["dP"].reshape(B, N, -1), B, U, True),
                               B * U)
        dz = r["dz"]                                                             # [b, i, j, h]
        errs["ds"] = per_graph(units(dP[:, HC:HC + H].view(B, N, H), B, U, True), units(r["ds"], B, U, True), B * U)
        errs["dd"] = per_graph(units(dP[:, HC + H:HC + 2 * H].view(B, N, H), B, U, True), units(r["dd"], B, U, True), B * U,
                               scale=units(dz.abs().sum(2), B, U, True))
        errs["dbias"] = per_graph(bw["dbias"].view(U, -1), r["dbias"].view(U, -1), U)
        if g.Fe:
            d_et = bw["d_et"]
            assert (d_et.diagonal(dim1=2, dim2=3) == 0).all(), "d_edge_terms is not exactly 0 on the diagonal"
            diag = torch.diagonal(dz, dim1=1, dim2=2).permute(0, 2, 1).abs()       # [b, i, h]
            terms = (dz.abs() + diag.unsqueeze(2) / (N - 1)).permute(0, 3, 2, 1)[..., self.off]
            errs["dz'"] = per_graph(units(d_et[..., self.off], B, U, False),
                                    units(r["dzp"].permute(0, 3, 2, 1)[..., self.off], B, U, False), B * U,
                                    scale=units(terms, B, U, False))
            errs["dv"] = per_graph(bw["dv"], r["dv"], H)                         # per head: a batch reduction
        return errs


def report(label, errs, tol=TOL):
    print(f"{label}: " + ", ".join(f"{k} {e:.2e}" for k, e in errs.items()))
    bad = {k: e for k, e in errs.items() if not e <= tol}
    assert not bad, (label, bad)


def pair_value(dP16, dblk, HC, cols):
    """The fp32 values an fp16 dP pair stands for: columns < HC at group 0's scale, the ds | dd columns at group 1's."""
    val = dP16[0, :, :cols].double() + dP16[1, :, :cols].double()
    inv = torch.where(torch.arange(cols, device=DEV) >= HC, dblk[3].double(), dblk[2].double())
    return val * inv


def same_bits(a, b):
    """Bit equality of two fp32 tensors, NaN included: cells a call leaves alone keep their NaN prefill (the diagonal of
    the edge terms, the padding columns of dP_aug) and must be left alone in both."""
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def relerr(a, ref):
    return ((a.double() - ref.double()).abs().max() / ref.double().abs().max().clamp_min(1e-300)).item()


# ======================================================================================== 1. stages against fp64
@pytest.mark.gpu
@pytest.mark.parametrize("geom", GEOMS, ids=geom_id)
def test_large_graph_attention_stages_against_fp64(cuda_lib, geom):
    """attn_fwd, attn_bwd (logits recomputed, and from the forward's edge terms), its fp16-pair dP output and
    attn_bwd_dalpha against float64, per graph, with both batched-GEMM back ends."""
    case = LargeCase(cuda_lib, geom)
    g, HC, H = geom, case.HC, geom.H
    r = case.reference()
    G = case.d_alpha()
    r_ga = case.reference(G)
    for algo in GEMM_ALGOS:
        label = f"{geom_id(g)} gemm_algo {algo}"
        f = case.forward(cuda_lib, algo)
        report(f"{label} forward", case.check_forward(f, r))
        f_ws = case.forward(cuda_lib, algo, keep_alpha=False, keep_terms=False)
        assert torch.equal(f_ws["out"], f["out"]), "out differs when the attention tile lives in the workspace"
        modes = [("recomputed logits", None)] + ([("forward's edge terms", f["terms"])] if g.Fe else [])
        for mode, terms in modes:
            bw = case.backward(cuda_lib, algo, terms=terms)
            report(f"{label} backward, {mode}", case.check_backward(bw, r))
        # (terms, bw: the last mode - the forward's edge terms when the layer has edge features)
        # the tensor-core operand form of dP against the fp32 gradient of the same call
        bp = case.backward(cuda_lib, algo, terms=terms, pair=True)
        got = pair_value(bp["dP16"], bp["dblk"], HC, HC + 2 * H)
        assert torch.isfinite(got).all()
        report(f"{label} fp16-pair dP", {"dP": relerr(got[:, :HC], bw["dP"][:, :HC]),
                                         "ds|dd": relerr(got[:, HC:], bw["dP"][:, HC:HC + 2 * H])}, PAIR_TOL)
        assert torch.equal(bp["dbias"], bw["dbias"]) and (not g.Fe or torch.equal(bp["dv"], bw["dv"]))
        # the gradient through the returned coefficients joins dalpha before the dropout factor
        bg = case.backward(cuda_lib, algo, terms=terms, G=G)
        report(f"{label} backward with d_alpha", case.check_backward(bg, r_ga))


# ======================================================================================== 3. batch independence
# (without dropout: the mask is keyed by batch position, so a graph's coefficients move with it only when it stays put)
INDEP = [Geom(5, 131, 5, 4, 9, False), Geom(3, 33, 200, 7, 12, True), Geom(3, 129, 360, 6, 128, True),
         Geom(4, 40, 7, 5, 12, False, 0.0, "loops"), Geom(3, 64, 0, 3, 20, False)]


@pytest.mark.gpu
@pytest.mark.parametrize("geom", INDEP, ids=geom_id)
@pytest.mark.parametrize("algo", GEMM_ALGOS, ids=["tf32x3_gemm", "ffma2_gemm"])
def test_large_graph_outputs_are_independent_of_batch_position(cuda_lib, geom, algo):
    """A graph's out, alpha, edge terms, dP_aug rows and d_edge_terms are the same bits whether it runs alone, in the
    batch, or in a permutation of the batch; two identical calls give the same bits for every output, dv and dbias (the
    two batch reductions) included."""
    case = LargeCase(cuda_lib, geom, seed=1)
    B, N, R, Fe = geom.B, geom.N, case.R, geom.Fe
    f = case.forward(cuda_lib, algo)
    bw = case.backward(cuda_lib, algo, terms=f["terms"])
    f2 = case.forward(cuda_lib, algo)
    bw2 = case.backward(cuda_lib, algo, terms=f2["terms"])
    for k in ("out", "alpha", "terms"):
        assert (f[k] is None and Fe == 0) or same_bits(f[k], f2[k]), ("repeat", k)
    for k in ("dP", "dv", "d_et", "dbias"):
        assert (bw[k] is None and Fe == 0) or same_bits(bw[k], bw2[k]), ("repeat", k)

    def sub(rows_of, edges_of, nb):
        P = case.P_aug[rows_of].contiguous()
        ea = case.ea[edges_of].contiguous() if Fe else None
        fo = case.forward(cuda_lib, algo, B=nb, P_aug=P, ea=ea)
        bo = case.backward(cuda_lib, algo, terms=fo["terms"], B=nb, P_aug=P, ea=ea, dout=case.dout[rows_of].contiguous())
        return fo, bo

    def same(fo, bo, rows, graphs):
        assert same_bits(fo["out"], f["out"][rows]), "out"
        assert same_bits(fo["alpha"], f["alpha"][graphs]), "alpha"
        assert same_bits(bo["dP"], bw["dP"][rows]), "dP_aug rows"
        if Fe:
            assert same_bits(fo["terms"], f["terms"][graphs]), "edge terms"
            assert same_bits(bo["d_et"], bw["d_et"][graphs]), "d_edge_terms"

    for b in sorted({0, B // 2, B - 1}):
        rows = torch.arange(b * N, (b + 1) * N, device=DEV)
        fo, bo = sub(rows, torch.arange(b * R, (b + 1) * R, device=DEV), 1)
        same(fo, bo, rows, torch.tensor([b], device=DEV))
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(3)).to(DEV)
    rows = (perm.view(B, 1) * N + torch.arange(N, device=DEV)).reshape(-1)
    fo, bo = sub(rows, (perm.view(B, 1) * R + torch.arange(R, device=DEV)).reshape(-1), B)
    same(fo, bo, rows, perm)


# ======================================================================================== 4. structured source at N > 32
# B, N, L, H, t0 (unsorted, repeated): H = 1, 3, 5, 8 -> HT = 2, 4, 6, 8 of win_dv_large2_kernel<6, HT> (L <= 48);
# L = 49 -> win_dv_large_kernel; N = 33, 256, 257 around the 8-row and 256-column work items
WINDOWS = [
    (5, 33, 48, 1, [7, 0, 7, 3, 1]),
    (3, 256, 48, 3, [4, 0, 4]),
    (2, 257, 48, 5, [2, 2]),
    (3, 33, 48, 8, [5, 1, 5]),
    (2, 257, 49, 8, [3, 0]),
    (4, 33, 49, 3, [2, 0, 2, 1]),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", WINDOWS, ids=lambda c: "B%dN%dL%dH%d" % c[:4])
def test_structured_source_against_fp64(cuda_lib, case):
    """spotv2_edge_terms_from_windows and spotv2_windows_dv (N > 32) against a float64 einsum over the windows.  Edge
    j -> i, r = min(i, j), c = max(i, j):  g_ij,h = <vv[.][r][c], v_h[0:L]> + <vv[.][j][j], v_h[L:2L]> + <vv[.][i][i], v_h[2L:3L]>
    (only the upper triangle is read: the windows here are not symmetric), and dv is the transpose of that map."""
    B, N, L, H, t0s = case
    Fe = 3 * L
    gen = torch.Generator(device=DEV).manual_seed(N * 100 + L * 10 + H)
    Tn = max(t0s) + L + 1
    # every lag its own power of two: the graphs' windows differ in scale
    vv = torch.randn(Tn, N, N, generator=gen, device=DEV) * torch.exp2(torch.randint(-4, 5, (Tn, 1, 1), generator=gen, device=DEV).float())
    v = torch.randn(H, Fe, generator=gen, device=DEV)
    t0 = torch.tensor(t0s, dtype=torch.int32, device=DEV)
    d = GatDesc(B, N, 16, Fe, H, 8, N * (N - 1), 0, 0.2, cuda_lib.spotv2_gat_ldp(H, 8), 0, 0, 0.0, 1, 0, 0, 0)
    # the float64 reference
    W = torch.stack([vv[t:t + L] for t in t0s]).double()                          # [B, L, N, N]
    up = torch.triu(W, 1)
    S = up + up.transpose(2, 3)                                                   # vv[min][max] off the diagonal
    D = torch.diagonal(W, dim1=2, dim2=3)                                         # [B, L, N]
    v64 = v.double()
    a = torch.einsum("btn,ht->bhn", D, v64[:, L:2 * L])                           # source node j
    c = torch.einsum("btn,ht->bhn", D, v64[:, 2 * L:])                            # target node i
    Z = torch.einsum("btji,ht->bhji", S, v64[:, :L]) + a.unsqueeze(3) + c.unsqueeze(2)
    off = ~torch.eye(N, dtype=torch.bool, device=DEV)
    terms = torch.full((B, H, N, N), float("nan"), device=DEV)
    wse = C.c_size_t()
    check(cuda_lib.spotv2_edge_terms_from_windows_workspace_bytes(C.byref(d), C.byref(wse)), "edge_terms ws")
    ws_e = torch.empty(max(wse.value, 256), dtype=torch.uint8, device=DEV)
    check(cuda_lib.spotv2_edge_terms_from_windows(C.byref(d), ptr(vv), Tn, L, ptr(t0), ptr(v), ptr(terms), ptr(ws_e),
                                                  ws_e.numel(), st()), "edge_terms_from_windows")
    # dv from d(edge terms) w [B, H, j, i] (diagonal 0), each graph at its own power of two
    w = torch.randn(B, H, N, N, generator=gen, device=DEV) * torch.exp2(torch.randint(-6, 7, (B, 1, 1, 1), generator=gen, device=DEV).float())
    w[..., ~off] = 0.0
    w64 = w.double()
    dv64 = torch.cat([torch.einsum("bhji,btji->ht", w64, S), torch.einsum("bhji,btj->ht", w64, D),
                      torch.einsum("bhji,bti->ht", w64, D)], 1)
    dv = torch.full((H, Fe), float("nan"), device=DEV)
    wsz = C.c_size_t()
    check(cuda_lib.spotv2_windows_dv_workspace_bytes(C.byref(d), C.byref(wsz)), "windows_dv ws")
    ws2 = torch.empty(max(wsz.value, 256), dtype=torch.uint8, device=DEV)
    check(cuda_lib.spotv2_windows_dv(C.byref(d), ptr(vv), Tn, L, ptr(t0), ptr(w), ptr(dv), ptr(ws2), ws2.numel(), st()),
          "windows_dv")
    torch.cuda.synchronize()
    assert torch.isfinite(terms[..., off]).all() and torch.isfinite(dv).all()
    errs = {"edge terms": per_graph(terms[..., off], Z[..., off], B),
            "dv": per_graph(dv, dv64, H),
            "dv lag block": per_graph(dv[:, :L], dv64[:, :L], H),
            "dv source-diagonal block": per_graph(dv[:, L:2 * L], dv64[:, L:2 * L], H),
            "dv target-diagonal block": per_graph(dv[:, 2 * L:], dv64[:, 2 * L:], H)}
    report("B%dN%dL%dH%d" % case[:4], errs)
