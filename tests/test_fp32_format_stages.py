"""The fp32 P_aug attention path at N <= 32 (p_format 0) stage by stage against float64, with several graphs per CTA and
every error taken per graph.

p_format 0 runs for every layer of GATModel(standardize=True), for layers the pair format does not cover (Fe > 384,
C % 4 != 0, concat with C % 8 != 0) and under gemm_algo 1, attn_bwd_algo 1 or 3.  Its kernels:
  - attn_fwd.cu: the forward, NPAIRS 4 / 8 / 15 / 16, VEC2 (C even), the FIX default-geometry instantiation, an edge-row
    ring of 48, 32 or 16 rows, bulk or cooperative copies into it, and a P-tile ring of 24 slots (8 where 24 do not fit);
  - attn_bwd2.cu, P16 = false: the pipelined backward (attn_bwd_algo 0 when its plan fits), whose two big products run on
    fp16 pairs of P and dout at ONE scale for the whole batch (s_P from p_amax, s_dO from max|dout|);
  - attn_bwd.cu: the phase-serial backward (attn_bwd_algo 1, and algo 0 where the pipelined plan does not fit), 2G CTAs;
  - attn_bwd3.cu: the tcgen05 backward (attn_bwd_algo 3; head-mean layers, N <= 31, the forward's edge terms), with its own
    H = 6 instantiation.
test_plan_coverage_of_the_geometry_grid restates the plan rules of all four and names any variant GEOMS no longer reaches;
test_every_documented_shape_has_a_plan sweeps the documented domain.

The operands and the float64 reference are those of tests/test_large_graph_stages.py (LargeCase): plain fp32, each graph's
P rows and dout rows at their own power of two in [2^-8, 2^8], per (graph, head) for concat layers, NaN in P_aug's pad
columns, dense_attention on the device in float64.  Batches hold G, 2G + 1 or 3G - 5 graphs (G = SM count = the grid of
the persistent kernels; the phase-serial kernel's 2G CTAs then hold one or two graphs).  Errors are per graph (per
(graph, head) for concat) against 1e-5; dd and dz' are measured against the magnitude of the terms they sum.

The pipelined kernel's single batch-wide scale gives every graph the same absolute floor: an fp16 pair at scale s resolves
2^-25 / s (half the spacing of subnormal lo values), and s maps the batch maximum below 2^15, so the floor is about 2^-39 of
the batch maximum (DESIGN.md section 4).  test_batch_wide_scale_floor holds a graph 2^-30 below the rest to the elementwise
bound that follows from the scales the kernel used:
  P and dout:  |dP~ - P| <= 2^-22 |P| + 2^-25 / s_P,   |dO~ - dO| <= 2^-22 |dO| + 2^-25 / s_dO   (hi | lo split)
  dP_j   <= g sum_i a_ij (A 2^-22 |dO_i| + 2^-25 / s_dO) + 2^-23 |dP_j|
  da_ij  <= E_ij = g sum_c (A 2^-22 |dO_ic| |P_jc| + 2^-25 |dO_ic| / s_P + 2^-25 |P_jc| / s_dO)
  dz_ij  <= a_ij (E_ij + sum_k a_ik E_ik);  dd_i <= sum_j dz-bound_ij;  ds_j <= sum_i dz-bound_ij;  dz'_ij <= dz_ij + dz_ii / (N - 1)
with A = 32 as in tests/test_pair_format_stages.py, each bound plus 1e-5 of the graph's own magnitude for the fp32 steps.
"""
import ctypes as C
import math
from pathlib import Path

import pytest
import torch

from spotv2net_b200._lib import GatDesc, check, ptr
from oracle import dense_gat, synth
from test_half_precision import workspace
from test_large_graph_stages import Geom, LargeCase, pair_value, report, rows_per_graph, same_bits, units
from test_pair_format_stages import per_graph

DEV = "cuda:0"
TOL = 1e-5
PAIR_TOL = 3e-6                # the fp16-pair dP output against the fp32 one (22 bits of the batch's scale)
A_BOUND = 32.0
ET_NS = 36                     # the edge-term layout for N <= 32: [B][H][N(j)][36(i)]
SMEM_CAP = 227 * 1024
CSRC = Path(__file__).resolve().parent.parent / "spotv2net_b200" / "csrc"
PIPELINED, PHASE_SERIAL, TCGEN05 = 0, 1, 3        # attn_bwd_algo

# B is (a, c): a G + c graphs.  rows as in test_large_graph_stages: "pyg", "loops" (N^2 rows, the input's self loops at
# scattered positions of a permuted edge order), "dense" (the dense target-major tile with a garbage diagonal)
GEOMS = [
    Geom((2, 1), 30, 126, 6, 500, False),           # the default: FIX forward and pipelined kernels, tcgen05 H = 6
    Geom((1, 0), 30, 126, 8, 256, True),            # forward ring 32, n_rounds 3, phase-serial ring 16
    Geom((3, -5), 7, 5, 3, 5, False),               # NPAIRS 4, odd C (no VEC2, no TMA), cooperative copies
    Geom((2, 1), 2, 3, 1, 2, True),                 # N = 2: the logit gradients cancel
    Geom((1, 0), 13, 0, 3, 7, True),                # no edge features
    Geom((2, 1), 32, 96, 8, 12, True),              # NPAIRS 16, pipelined chunk 64 with ksplit 1
    Geom((3, -5), 31, 40, 7, 44, False),            # tcgen05 at N = 31 with a run-time H; chunk 96, n_rounds 2
    Geom((1, 0), 16, 190, 4, 33, False),            # chunk 32, dv_rg 2, no TMA
    Geom((2, 1), 24, 200, 5, 20, True),             # forward ring 32, dv_rg 1
    Geom((3, -5), 9, 64, 8, 10, False),             # chunk 80
    Geom((1, 0), 17, 360, 2, 25, False),            # forward ring 16
    Geom((2, 1), 30, 360, 6, 500, False),           # the 8-slot forward (GATModel(standardize=True), seq_length 120)
    Geom((1, 0), 30, 512, 6, 500, False),           # Fe at its limit: the pipelined plan does not fit, phase-serial runs
    Geom((3, -5), 32, 512, 1, 4, False),
    Geom((2, 1), 11, 7, 5, 12, False, 0.0, "loops"),     # input self loops, R Fe % 4 == 3: cooperative copies
    Geom((1, 0), 20, 33, 3, 16, True, 0.0, "loops"),     # input self loops, bulk copies
    Geom((2, 1), 16, 12, 6, 10, False, 0.0, "dense"),    # spotv2_edge_table_dense, garbage on the diagonal
    Geom((2, 1), 30, 126, 6, 500, False, 0.3),      # attention dropout on the default geometry (FIX + DROP)
    Geom((1, 0), 30, 126, 6, 500, False, 0.9),
    Geom((3, -5), 24, 200, 5, 20, True, 0.3),       # and on a concat layer
    Geom((1, 0), 24, 200, 5, 20, True, 0.9),
]


def geom_id(g):
    return (f"B{g.B[0]}G{g.B[1]:+d}N{g.N}Fe{g.Fe}H{g.H}C{g.C}{'cat' if g.concat else 'mean'}"
            + (f"_p{g.pdrop:g}" if g.pdrop else "") + ("" if g.rows == "pyg" else "_" + g.rows))


# ======================================================================================== the plans, restated
def round_up(x, a):
    return (x + a - 1) // a * a


def ldp_of(H, C_):
    return max(round_up(H * C_ + 2 * H, 4), 32)


def npairs_of(N):
    np_ = (N + 1) // 2
    return 4 if np_ <= 4 else 8 if np_ <= 8 else 15 if np_ <= 15 else 16


def common_plan(N, Fe, H, R, npairs, rows):
    """attn_smem_plan (attn_common.cuh): (NS, KS, offset of s|d, base total, ring stage bytes)."""
    NS, KS, NT = (2 * npairs + 3) // 4 * 4, ((Fe + 7) // 8 + 7) // 8 * 8, (H + 7) // 8
    off_sd = 512 + round_up(R * 4, 16) + NT * KS * 32 * 16
    base = off_sd + round_up(N * 2 * H * 4, 16) + round_up(H * N * NS * 4, 16)
    return NS, KS, off_sd, base, round_up(rows * Fe * 4, 128)


def bulk_ok(Fe, R):
    """attn_params_of (attn_bwd.cu): bulk copies when the edge block is 16-byte aligned (every buffer here is) and
    R Fe % 4 == 0."""
    return Fe > 0 and R * Fe % 4 == 0


def fwd_plan(N, Fe, H, C_, R, concat):
    """launch_fwd (attn_fwd.cu): dict(npairs, vec2, rows, slots, total, fix, bulk)."""
    npairs = npairs_of(N)

    def total(rows, slots):
        _, KS, off_sd, _, ring = common_plan(N, Fe, H, R, npairs, rows)
        off_tile = off_sd + 2 * round_up(N * 2 * H * 4, 16)
        off_ring = round_up(off_tile + 2 * round_up(H * N * 36 * 4, 16), 128)
        return round_up(off_ring + 2 * ring + 256, 1024) + (slots + 2) * 4096, KS

    def plan(slots):
        rows = 48
        while rows - 16 >= 16 and total(rows, slots)[0] > SMEM_CAP:
            rows -= 16
        return rows

    slots, rows = 24, plan(24)
    if total(rows, 24)[0] > SMEM_CAP:
        slots, rows = 8, plan(8)
    t, KS = total(rows, slots)
    vec2, bulk = C_ % 2 == 0, bulk_ok(Fe, R)
    fix = (npairs == 15 and vec2 and N == 30 and H == 6 and C_ == 500 and Fe == 126 and R == 870 and not concat
           and ldp_of(H, C_) == 3012 and bulk and KS == 16 and rows == 48 and slots == 24)
    return dict(npairs=npairs, vec2=vec2, rows=rows, slots=slots, total=t, fix=fix, bulk=bulk)


def bwd2_plan(N, Fe, H, C_, R, concat):
    """make_plan (attn_bwd2.cu), P16 = false: None when it does not fit, else dict(chunk, ksplit, dv_rg, n_rounds, tma,
    n_slots, total, fix)."""
    KS = ((Fe + 7) // 8 + 7) // 8 * 8
    hpr = 3 if concat else 6
    ldo = H * C_ if concat else C_
    o = 128 + round_up(max(R, 1) * 4, 16) + (KS if Fe > 0 else 0) * 32 * 16 + round_up(N * 2 * H * 4, 16)
    o += 2 * round_up(H * N * 4, 16) + 2 * H * 32 * 4 + round_up(ldo * 4, 16) + round_up(H * N * 36 * 4, 16)
    o = round_up(o, 1024) + round_up(H * N * 36 * 4, 16)
    off_slots = round_up(o, 1024)
    slot = 7 * 4096
    if Fe > 0 and round_up(16 * Fe * 4, 1024) > slot:
        slot = round_up(16 * Fe * 4, 1024)
    avail = SMEM_CAP - 256 - off_slots if SMEM_CAP - 256 > off_slots else 0
    n_slots = min(avail // slot, 8)
    if n_slots < 3:
        return None
    chunk, ksplit, rg, nchunks = 0, 1, None, 0
    if Fe > 0:
        chunk = min(slot // (Fe * 4) // 16 * 16, 96)
        if chunk > R:
            chunk = round_up(R, 16)
        nchunks = -(-R // chunk)
    n_mt = chunk // 16
    ksplit = 2 if (n_mt > 0 and 2 * n_mt <= 6 and KS >= 16) else 1
    if Fe > 0:
        rg = min(24 // ((Fe + 15) // 16), (chunk + 7) // 8, 3)
        if rg < 1:
            return None
    fix = (N == 30 and H == 6 and C_ == 500 and Fe == 126 and R == 870 and not concat and bulk_ok(Fe, R) and KS == 16
           and chunk == 48 and nchunks == 19 and n_slots == 5 and slot == 7 * 4096)
    return dict(chunk=chunk, ksplit=ksplit, dv_rg=rg, n_rounds=-(-H // hpr), tma=C_ % 4 == 0, n_slots=n_slots,
                total=off_slots + n_slots * slot + 256, fix=fix)


def serial_plan(N, Fe, H, C_, R, concat):
    """bwd_smem_plan + launch_bwd (attn_bwd.cu): (NPAIRS, ring rows, total); the ring shrinks toward 113 KB."""
    npairs = npairs_of(N)
    ldo = H * C_ if concat else C_
    NP5 = (N + 4) // 5 * 5

    def total(rows):
        NS, _, _, base, ring = common_plan(N, Fe, H, R, npairs, rows)
        o = base + round_up(H * N * NS * 4, 16) + 2 * round_up(H * N * 4, 16) + round_up(ldo * 4, 16)
        stage = H * NP5 * 20 * 4 + (H if concat else 1) * NP5 * 20 * 4
        return round_up(o, 128) + max(2 * stage, 2 * ring)

    rows = 48
    while rows - 16 >= 16 and total(rows) > 113 * 1024:
        rows -= 16
    return npairs, rows, total(rows)


def bwd3_applies(N, Fe, H, C_, R, concat, terms=True, terms_in=False):
    """attn_bwd3_applies (attn_bwd3.cu) short of its shared-memory plan (the calls below fail if that does not fit)."""
    if N > 31 or N < 1 or H > 8 or concat or C_ % 4 != 0 or ldp_of(H, C_) % 4 != 0:
        return False
    if Fe <= 0 or not terms:
        return False
    return terms_in or (Fe <= 128 and Fe % 2 == 0 and bulk_ok(Fe, R))


def bwd_kernels(N, Fe, H, C_, R, concat, terms=True):
    """choose_bwd_kernel (attn_bwd.cu): attn_bwd_algo -> the kernel that runs ("pipelined", "phase-serial", "tcgen05")."""
    k = {PIPELINED: "pipelined" if bwd2_plan(N, Fe, H, C_, R, concat) else "phase-serial", PHASE_SERIAL: "phase-serial"}
    if bwd3_applies(N, Fe, H, C_, R, concat, terms):
        k[TCGEN05] = "tcgen05"
    return k


# the source lines restated above: if one of them changes, the restatement (and what the grid reaches) needs a new look
RESTATED = {
    "attn_fwd.cu": [
        "constexpr int kFwdChunkRows3 = 48;", "constexpr int kPSlots = 24;", "constexpr int kPSlotsLean = kCbPerPass;",
        "constexpr int kCbPerPass = 8;", "constexpr int kPTileBytes = 32 * 128;", "const int NS = 36;",
        "s.off_tile = s.off_sd + 2 * sd_bytes;", "s.off_ring = round_up(s.off_tile + 2 * tile_bytes, 128);",
        "auto ptile_off = [&](const AttnSmem& s) { return round_up(s.off_ring + 2 * s.ring_stage_bytes + 256, 1024); };",
        "auto total = [&](const AttnSmem& s, int slots) { return ptile_off(s) + (size_t)(slots + 2) * kPTileBytes; };",
        "for (int rows = kFwdChunkRows3 - 16; rows >= 16 && total(s, slots) > 227 * 1024; rows -= 16)",
        "const bool lean = total(sm, kPSlots) > 227 * 1024;", "if (lean) sm = plan(kPSlotsLean);",
        "if (np <= 4) return dispatch_vec<4>(a, st);", "if (np <= 8) return dispatch_vec<8>(a, st);",
        "if (np <= 15) return dispatch_vec<15>(a, st);", "if (np <= 16) return dispatch_vec<16>(a, st);",
        "const bool fix = NPAIRS == 15 && VEC2 && p.N == 30 && p.H == 6 && p.C == 500 && p.Fe == 126 && p.R == 870 && "
        "!p.concat && p.ldp == 3012 && p.ldo == 500 && p.bulk_ok && sm.NS == 36 && sm.KS == 16 && sm.chunk_rows == kFwdChunkRows3;",
    ],
    "attn_common.cuh": [
        "s.NS = (2 * npairs + 3) / 4 * 4;", "s.KS = ((Fe + 7) / 8 + 7) / 8 * 8;", "s.NT = (H + 7) / 8;",
        "s.off_bar = o; o += 512;", "s.off_table = o; o += round_up((size_t)R * 4, 16);",
        "s.off_vfrag = o; o += (size_t)s.NT * s.KS * 32 * 16;", "s.off_sd = o; o += round_up((size_t)N * 2 * H * 4, 16);",
        "s.off_tile = o; o += round_up((size_t)H * N * s.NS * 4, 16);",
        "s.ring_stage_bytes = round_up((size_t)chunk_rows * Fe * 4, 128);", "constexpr int kBwdChunkRows = 48;",
    ],
    "attn_bwd2.cu": [
        "s.hpr = p.concat ? 3 : 6;", "s.tma_ok = (C % 4 == 0) ? 1 : 0;", "constexpr int kMaxSlots = 8;",
        "s.off_bar = o; o += 128;", "s.off_table = o; o += (uint32_t)round_up((size_t)(p.R > 0 ? p.R : 1) * 4, 16);",
        "s.off_vfrag = o; o += (uint32_t)((Fe > 0 ? s.KS : 0) * 32 * 16);",
        "s.off_mask = o; o += 2 * (uint32_t)round_up((size_t)H * N * 4, 16);", "s.off_dspart = o; o += (uint32_t)(2 * H * 32 * 4);",
        "s.off_dbias = o; o += (uint32_t)round_up((size_t)p.ldo * 4, 16);",
        "s.off_tile = o; o += (uint32_t)round_up((size_t)H * N * kNS2 * 4, 16);", "o = (uint32_t)round_up(o, 1024);",
        "s.off_D = o; o += (uint32_t)round_up((size_t)H * N * kNS2 * 4, 16);", "s.off_slots = (uint32_t)round_up(o, 1024);",
        "s.slot_bytes = kGrpTiles * kTile;",
        "if (Fe > 0 && (uint32_t)round_up((size_t)16 * Fe * 4, 1024) > s.slot_bytes) s.slot_bytes = (uint32_t)round_up((size_t)16 * Fe * 4, 1024);",
        "const uint32_t avail = 227 * 1024 - 256 > s.off_slots ? 227 * 1024 - 256 - s.off_slots : 0;",
        "if (s.n_slots < 3) { s.total = 0xffffffffu; return s; }",
        "s.chunk_rows = (int)(s.slot_bytes / ((uint32_t)Fe * 4)) / 16 * 16;", "if (s.chunk_rows > 96) s.chunk_rows = 96;",
        "if (s.chunk_rows > p.R) s.chunk_rows = (p.R + 15) / 16 * 16;",
        "s.ksplit = (s.n_mt_chunk > 0 && 2 * s.n_mt_chunk <= kW / 2 && s.KS >= 16) ? 2 : 1;",
        "int rg = (kMaxDvUnits * kW) / s.n_mtiles;", "const int rg_max = (s.chunk_rows + 7) / 8;", "if (rg > 3) rg = 3;",
        "static constexpr int KS = 16, chunk_rows = 48, nchunks = 19, n_cb = 16, hpr = 6, n_rounds = 1, n_mt_chunk = 3, ksplit = 2;",
        "static constexpr int n_mtiles = 8, dv_rg = 3, dv_rpu = 16, dv_units = 24, cbs_per_grp_d = 7, n_slots = 5;",
    ],
    "attn_bwd.cu": [
        "const int ldo = concat ? H * C : C;", "s.off_D = o; o += round_up((size_t)H * N * s.a.NS * 4, 16);",
        "s.off_mask = o; o += 2 * round_up((size_t)H * N * 4, 16);", "s.off_dbias = o; o += round_up((size_t)ldo * 4, 16);",
        "s.off_union = round_up(o, 128);", "s.stage_P_bytes = (size_t)H * s.NP5 * kCKP * 4;",
        "s.stage_G_bytes = (size_t)(concat ? H : 1) * s.NP5 * kCKP * 4;", "constexpr int kCKP = 20;",
        "for (int rows = kBwdChunkRows - 16; rows >= 16 && sm.total > 113 * 1024; rows -= 16)",
        "if (d->attn_bwd_algo == 1 || (d->attn_bwd_algo != 2 && !attn_bwd2_fits(p))) *k = BwdKernel::kPhaseSerial;",
        "int grid = 2 * sm_count();",
        "p.bulk_ok = d->Fe > 0 && aligned16(e.rows) && ((size_t)d->R * d->Fe) % 4 == 0;",
    ],
    "attn_bwd3.cu": [
        "if (p.N > 31 || p.N < 1 || p.H > kMaxHeads || p.concat || p.C % 4 != 0 || p.ldp % 4 != 0) return false;",
        "if (p.Fe <= 0 || !p.edge_terms) return false;",
        "if (!p.terms_in && (p.Fe > 128 || p.Fe % 2 != 0 || !p.bulk_ok || !p.edge_rows || !p.table)) return false;",
        "auto kern = p.H == 6 ? (drop ? gat_attn_bwd3_kernel<true, 6> : gat_attn_bwd3_kernel<false, 6>)",
    ],
    "api.cu": ["const int32_t w = (H * C + 2 * H + 3) / 4 * 4;"],
}


def assert_restated():
    for src, lines in RESTATED.items():
        text = " ".join((CSRC / src).read_text().split())
        changed = [ln for ln in lines if " ".join(ln.split()) not in text]
        assert not changed, f"{src} no longer holds these lines restated by this test: {changed}"


def reached_variants(geoms):
    out = {k: set() for k in ("fwd NPAIRS", "fwd VEC2", "fwd FIX", "fwd ring rows", "fwd P slots", "fwd copies",
                              "pipelined fits", "pipelined chunk", "pipelined ksplit", "pipelined dv_rg",
                              "pipelined n_rounds", "pipelined tma", "pipelined FIX", "pipelined DROP",
                              "serial NPAIRS", "serial ring rows", "tcgen05 H", "no edge features", "row source")}
    for g in geoms:
        R = rows_per_graph(g)
        f = fwd_plan(g.N, g.Fe, g.H, g.C, R, g.concat)
        out["fwd NPAIRS"].add(f["npairs"]); out["fwd VEC2"].add(f["vec2"]); out["fwd FIX"].add(f["fix"])
        out["fwd P slots"].add(f["slots"])
        if g.Fe:
            out["fwd ring rows"].add(f["rows"]); out["fwd copies"].add("bulk" if f["bulk"] else "cooperative")
        b = bwd2_plan(g.N, g.Fe, g.H, g.C, R, g.concat)
        out["pipelined fits"].add(b is not None)
        if b:
            out["pipelined n_rounds"].add(b["n_rounds"]); out["pipelined tma"].add(b["tma"]); out["pipelined FIX"].add(b["fix"])
            out["pipelined DROP"].add(g.pdrop > 0)
            if g.Fe:
                out["pipelined chunk"].add(b["chunk"]); out["pipelined ksplit"].add(b["ksplit"])
                out["pipelined dv_rg"].add(b["dv_rg"])
        npairs, rows, _ = serial_plan(g.N, g.Fe, g.H, g.C, R, g.concat)
        out["serial NPAIRS"].add(npairs)
        if g.Fe:
            out["serial ring rows"].add(rows)
        if bwd3_applies(g.N, g.Fe, g.H, g.C, R, g.concat):
            out["tcgen05 H"].add("6" if g.H == 6 else "run-time")
        out["no edge features"].add(g.Fe == 0); out["row source"].add(g.rows)
    return out


def test_plan_coverage_of_the_geometry_grid():
    """Without a device: the grid reaches every variant of the four kernels' plans (forward NPAIRS, VEC2, FIX, ring rows,
    P slots and copy path; pipelined fit, chunk rows, ksplit, dv_rg, n_rounds, TMA, FIX and DROP; phase-serial NPAIRS and
    ring rows; both tcgen05 instantiations); the restated rules are still the library's."""
    assert_restated()
    # 24 P slots at N = 30, H = 6, C = 500 fit up to Fe = 330 (233 472 B at Fe = 331)
    assert fwd_plan(30, 330, 6, 500, 870, False)["slots"] == 24 and fwd_plan(30, 331, 6, 500, 870, False)["slots"] == 8
    assert fwd_plan(32, 512, 8, 16, 992, False)["total"] == 222208
    reached = reached_variants(GEOMS)
    wanted = {
        "fwd NPAIRS": {4, 8, 15, 16}, "fwd VEC2": {True, False}, "fwd FIX": {True, False}, "fwd ring rows": {48, 32, 16},
        "fwd P slots": {24, 8}, "fwd copies": {"bulk", "cooperative"},
        "pipelined fits": {True, False}, "pipelined chunk": {16, 32, 48, 64, 80, 96}, "pipelined ksplit": {1, 2},
        "pipelined dv_rg": {1, 2, 3}, "pipelined n_rounds": {1, 2, 3}, "pipelined tma": {True, False},
        "pipelined FIX": {True, False}, "pipelined DROP": {True, False},
        "serial NPAIRS": {4, 8, 15, 16}, "serial ring rows": {48, 32, 16},
        "tcgen05 H": {"6", "run-time"}, "no edge features": {True, False}, "row source": {"pyg", "loops", "dense"},
    }
    missing = {k: sorted(wanted[k] - reached[k], key=str) for k in wanted if wanted[k] - reached[k]}
    assert not missing, f"variants of the p_format 0 path the grid no longer reaches: {missing}"
    assert all(g.N <= 32 for g in GEOMS)


def test_every_documented_shape_has_a_plan():
    """Without a device: every N in 1..32, H in 1..8, Fe in 0..512, head mean and concat (C from 1 to 1024) has a
    forward plan within 227 KB and a backward kernel whose plan fits (the pipelined one, else the phase-serial one), by
    the library's rules as restated above."""
    assert_restated()
    no_fwd, no_bwd = [], []
    for N in range(1, 33):
        R = N * (N - 1)
        for H in range(1, 9):
            for Fe in range(0, 513 if R else 1):                      # (check_desc: Fe > 0 needs edges)
                if fwd_plan(N, Fe, H, 16, R, False)["total"] > SMEM_CAP:
                    no_fwd.append((N, H, Fe))
                for C_ in (1, 500, 1024):
                    for concat in (False, True):
                        if bwd2_plan(N, Fe, H, C_, R, concat) is None and serial_plan(N, Fe, H, C_, R, concat)[2] > SMEM_CAP:
                            no_bwd.append((N, H, Fe, C_, concat))
    assert not no_fwd, f"{len(no_fwd)} shapes (N, H, Fe) without a forward plan, e.g. {no_fwd[:5]}"
    assert not no_bwd, f"{len(no_bwd)} shapes (N, H, Fe, C, concat) without a backward plan, e.g. {no_bwd[:5]}"


# ======================================================================================== one geometry end to end
def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def st():
    return torch.cuda.current_stream().cuda_stream


class Fp32Case(LargeCase):
    """LargeCase's operands and float64 reference at N <= 32: the calls take attn_bwd_algo, and the edge terms travel in
    the [B][H][N][36] layout (views [..., :N] are what the checks read)."""

    def __init__(self, cuda_lib, g, seed=0, edge_mode=0):
        self.edge_mode = edge_mode
        super().__init__(cuda_lib, g, seed)

    def desc(self, bwd_algo, B=None):
        g = self.g
        return GatDesc(B or g.B, g.N, 16, g.Fe, g.H, g.C, self.R, int(g.concat), 0.2, self.ldp, 0, bwd_algo, g.pdrop,
                       self.edge_mode, 0x2468ACE, 0x13579BDF, 0)

    def forward(self, cuda_lib, B=None, P_aug=None, ea=None, terms_in=None):
        """attn_fwd with NaN-prefilled outputs (terms_in: the edge terms of edge_mode 1)."""
        g = self.g
        B = B or g.B
        d = self.desc(PIPELINED, B)
        P_aug = self.P_aug if P_aug is None else P_aug
        ea = self.ea if ea is None else ea
        out = torch.full((B * g.N, self.ldo), float("nan"), device=DEV)
        alpha = torch.full((B, g.H, g.N, g.N), float("nan"), device=DEV)
        t36 = terms_in
        if t36 is None and g.Fe:
            t36 = torch.full((B, g.H, g.N, ET_NS), float("nan"), device=DEV)
            etb = C.c_size_t()
            check(cuda_lib.spotv2_gat_edge_terms_bytes(C.byref(d), C.byref(etb)), "edge_terms_bytes")
            assert etb.value == t36.numel() * 4
        check(cuda_lib.spotv2_gat_attn_fwd(C.byref(d), ptr(P_aug), ptr(ea) if terms_in is None else None,
                                           ptr(self.table) if terms_in is None else None, ptr(self.v), ptr(self.bias),
                                           ptr(out), ptr(alpha), ptr(t36), None, 0, st()), "attn_fwd")
        torch.cuda.synchronize()
        return dict(out=out, alpha=alpha, t36=t36, terms=t36[..., :g.N] if t36 is not None else None)

    def backward(self, cuda_lib, bwd_algo, t36=None, G=None, pair=False, B=None, P_aug=None, ea=None, dout=None,
                 p_amax=None, structured=False):
        """attn_bwd (attn_bwd_dalpha with G), NaN-prefilled outputs; t36: the forward's edge terms, or None to recompute
        them; pair: dP as the fp16 pair."""
        g = self.g
        B = B or g.B
        n, H, Fe = B * g.N, g.H, g.Fe
        d = self.desc(bwd_algo, B)
        P_aug = self.P_aug if P_aug is None else P_aug
        ea = None if structured else self.ea if ea is None else ea
        dout = self.dout if dout is None else dout
        dP, dP16, dblk = None, None, None
        if pair:
            dP16 = torch.full((2, n, cuda_lib.spotv2_gat_ld16(self.HC + 2 * H)), float("nan"), device=DEV, dtype=torch.float16)
            dblk = torch.full((8,), float("nan"), device=DEV)
        else:
            dP = torch.full((n, self.ldp), float("nan"), device=DEV)
        dv = torch.full((H, Fe), float("nan"), device=DEV) if Fe and not structured else None
        d_et = torch.full((B, H, g.N, ET_NS), float("nan"), device=DEV) if Fe else None
        dbias = torch.full((self.ldo,), float("nan"), device=DEV)
        ws = workspace(cuda_lib, d)
        args = [C.byref(d), ptr(P_aug), ptr(p_amax), ptr(ea), ptr(t36), None if structured else ptr(self.table), ptr(self.v),
                ptr(dout), ptr(dP), ptr(dP16[0]) if pair else None, ptr(dP16[1]) if pair else None, ptr(dblk), ptr(dv),
                ptr(d_et), ptr(dbias), ptr(ws), ws.numel(), st()]
        if G is None:
            check(cuda_lib.spotv2_gat_attn_bwd(*args), "attn_bwd")
        else:
            check(cuda_lib.spotv2_gat_attn_bwd_dalpha(*args, ptr(G)), "attn_bwd_dalpha")
        torch.cuda.synchronize()
        return dict(dP=dP, dP16=dP16, dblk=dblk, dv=dv, d_et36=d_et, d_et=d_et[..., :g.N] if Fe else None, dbias=dbias)


    def check_backward(self, bw, r):
        """LargeCase's checks, with ds_j = sum_i dz_ij measured against sum_i |dz_ij| like dd: at N = 2 the two terms of
        each sum nearly cancel (a target's two coefficients move only through their difference)."""
        errs = super().check_backward(bw, r)
        g, B, U, N, H, HC = self.g, self.g.B, self.U, self.g.N, self.g.H, self.HC
        errs["ds"] = per_graph(units(bw["dP"][:, HC:HC + H].reshape(B, N, H), B, U, True), units(r["ds"], B, U, True), B * U,
                               scale=units(r["dz"].abs().sum(1), B, U, True))
        return errs


def with_batch(g):
    a, c = g.B
    return g._replace(B=a * sm_count() + c)


def pair_errors(bp, bw, B, HC, H):
    """Per graph: the fp16-pair dP against the fp32 one of the same kernel, relative to PAIR_TOL |fp32_b| + the pair's
    absolute resolution at the batch's scale (2^-25 / scale: half the spacing of subnormal lo values)."""
    got = pair_value(bp["dP16"], bp["dblk"], HC, HC + 2 * H)
    assert torch.isfinite(got).all()
    ref = bw["dP"][:, :HC + 2 * H].double()
    errs = {}
    for name, cols, inv in (("dP", slice(0, HC), bp["dblk"][2]), ("ds|dd", slice(HC, HC + 2 * H), bp["dblk"][3])):
        d = (got[:, cols] - ref[:, cols]).abs().reshape(B, -1).amax(1)
        allow = PAIR_TOL * ref[:, cols].abs().reshape(B, -1).amax(1) + inv.double() * 2.0 ** -25
        errs[name] = (d / allow.clamp_min(1e-300)).max().item() * PAIR_TOL
    return errs


# ======================================================================================== 1. stages against fp64
@pytest.mark.gpu
@pytest.mark.parametrize("geom", GEOMS, ids=geom_id)
def test_fp32_attention_stages_against_fp64(cuda_lib, geom):
    """attn_fwd, then each backward that applies (pipelined or its phase-serial fallback, phase-serial, tcgen05), once
    recomputing the logits and once from the forward's edge terms, plain and with d_alpha, and the fp16-pair dP output,
    against float64, per graph."""
    g = with_batch(geom)
    case = Fp32Case(cuda_lib, g)
    B, HC, H = g.B, case.HC, g.H
    r = case.reference()
    G = case.d_alpha()
    r_ga = case.reference(G)
    label = geom_id(geom) + f" (B = {B})"
    f = case.forward(cuda_lib)
    report(f"{label} forward", case.check_forward(f, r))
    kernels = bwd_kernels(g.N, g.Fe, H, g.C, case.R, g.concat)
    assert (geom.Fe, geom.H, geom.N) != (512, 6, 30) or kernels[PIPELINED] == "phase-serial"
    for algo, kern in kernels.items():
        modes = ([("recomputed logits", None)] if kern != "tcgen05" else []) + ([("edge terms", f["t36"])] if g.Fe else [])
        for mode, t36 in modes:
            bw = case.backward(cuda_lib, algo, t36=t36)
            report(f"{label} {kern} backward, {mode}", case.check_backward(bw, r))
            bg = case.backward(cuda_lib, algo, t36=t36, G=G)
            report(f"{label} {kern} backward with d_alpha, {mode}", case.check_backward(bg, r_ga))
        bp = case.backward(cuda_lib, algo, t36=t36, pair=True)
        report(f"{label} {kern} fp16-pair dP", pair_errors(bp, bw, B, HC, H), PAIR_TOL)
        assert torch.equal(bp["dbias"], bw["dbias"]) and (not g.Fe or torch.equal(bp["dv"], bw["dv"]))


# ======================================================================================== 2. the batch-wide scale
def scale_of(amax):
    """dp_scale_from_amax (attn_bwd.cuh): 2^(15 - e), amax = m 2^e with m in [0.5, 1)."""
    return 2.0 ** (15 - math.frexp(amax)[1])


@pytest.mark.gpu
def test_batch_wide_scale_floor(cuda_lib):
    """Pipelined kernel: one graph 2^-30 below the rest of the batch is held to the elementwise bound of the module
    docstring, built from the scales the kernel used; the other graphs, spread over 2^+-8, still meet 1e-5 per graph."""
    g = with_batch(Geom((2, 1), 30, 126, 6, 500, False))
    case = Fp32Case(cuda_lib, g, seed=5)
    B, N, H, HC, tiny = g.B, g.N, g.H, case.HC, g.B // 3
    P = case.P_aug[:, :HC].view(B, N, HC)
    P[tiny] *= 2.0 ** -30                                           # exact: powers of two
    case.dout.view(B, N, -1)[tiny] *= 2.0 ** -30
    case.P64 = P.view(B, N, H, g.C).double()
    amax_P = P.abs().max().item()
    p_amax = torch.zeros(8, device=DEV)
    p_amax[0] = amax_P                                              # (the bits of max|P|, read back as a float)
    s_P, s_dO = scale_of(amax_P), scale_of(case.dout.abs().max().item())
    r = case.reference()
    f = case.forward(cuda_lib)
    bw = case.backward(cuda_lib, PIPELINED, t36=f["t36"], p_amax=p_amax)
    assert bwd2_plan(N, g.Fe, H, g.C, case.R, False)["fix"]
    others = torch.arange(B, device=DEV) != tiny
    # the rest of the batch: 1e-5 per graph
    dz = r["dz"]
    errs = {"dP": per_graph(bw["dP"][:, :HC].reshape(B, -1)[others], r["dP"].reshape(B, -1)[others], B - 1)}
    errs["dd"] = per_graph(bw["dP"][:, HC + H:HC + 2 * H].reshape(B, -1)[others], r["dd"].reshape(B, -1)[others], B - 1,
                           scale=dz.abs().sum(2).reshape(B, -1)[others])
    errs["ds"] = per_graph(bw["dP"][:, HC:HC + H].reshape(B, -1)[others], r["ds"].reshape(B, -1)[others], B - 1,
                           scale=dz.abs().sum(1).reshape(B, -1)[others])
    report(f"graphs at 2^+-8 beside one at 2^-30 (B = {B})", errs)
    # the elementwise bound, every graph
    a = r["alpha"]                                                  # [b, i, j, h]
    Pa, dOa = case.P64.abs(), r["dO"].abs()                         # dO carries g = 1/H
    gsc = 1.0 / H
    E = (A_BOUND * 2.0 ** -22 * torch.einsum("bihc,bjhc->bijh", dOa, Pa)
         + 2.0 ** -25 / s_P * dOa.sum(3).unsqueeze(2) + 2.0 ** -25 / s_dO * gsc * Pa.sum(3).unsqueeze(1))
    Bz = a * (E + (a * E).sum(2, keepdim=True))
    mag = lambda t: t.abs().reshape(B, -1).amax(1).view(B, *([1] * (t.dim() - 1)))
    bound_dP = (A_BOUND * 2.0 ** -22 * r["adO"] + gsc * 2.0 ** -25 / s_dO * a.sum(1).unsqueeze(3)
                + 2.0 ** -39 * dOa.sum(1).unsqueeze(1) + 2.0 ** -23 * r["dP"].abs() + TOL * mag(r["dP"]))
    got_dP = bw["dP"][:, :HC].double().reshape(B, N, H, g.C)
    dzsum_i = dz.abs().sum(2)
    checks = {
        "dP": ((got_dP - r["dP"]).abs(), bound_dP),
        "dd": ((bw["dP"][:, HC + H:HC + 2 * H].double().reshape(B, N, H) - r["dd"]).abs(), Bz.sum(2) + TOL * mag(dzsum_i)),
        "ds": ((bw["dP"][:, HC:HC + H].double().reshape(B, N, H) - r["ds"]).abs(), Bz.sum(1) + TOL * mag(dz.abs().sum(1))),
    }
    diagB = torch.diagonal(Bz, dim1=1, dim2=2).permute(0, 2, 1)     # [b, i, h]
    bz_p = (Bz + diagB.unsqueeze(2) / (N - 1)).permute(0, 3, 2, 1)[..., case.off]
    got_zp = bw["d_et"][..., case.off].double()
    ref_zp = r["dzp"].permute(0, 3, 2, 1)[..., case.off]
    checks["dz'"] = ((got_zp - ref_zp).abs(), bz_p + TOL * mag(dz.abs()).view(B, 1, 1))
    for name, (err, bound) in checks.items():
        ratio = (err / bound).reshape(B, -1).amax(1)
        print(f"{name}: worst error / bound {ratio.max().item():.3f}, tiny graph {ratio[tiny].item():.3f}")
        assert (err <= bound).all(), (name, ratio.max().item())
    # what the floor means for the tiny graph on its own scale
    rel_tiny = ((got_dP[tiny] - r["dP"][tiny]).abs().max() / r["dP"][tiny].abs().max()).item()
    print(f"tiny graph: dP error {rel_tiny:.2e} of its own maximum")


# ======================================================================================== 3. independence
INDEP = [Geom((2, 1), 30, 126, 6, 500, False), Geom((3, -5), 7, 5, 3, 5, False), Geom((2, 1), 24, 200, 5, 20, True),
         Geom((1, 0), 30, 360, 6, 500, False), Geom((2, 1), 11, 7, 5, 12, False, 0.0, "loops")]


@pytest.mark.gpu
@pytest.mark.parametrize("geom", INDEP, ids=geom_id)
def test_fp32_outputs_are_independent_of_batch_position(cuda_lib, geom):
    """The forward's out, alpha and edge terms are the same bits alone, in the batch and in a permuted batch; every
    backward's per-graph outputs are the same bits under permutation (the batch maxima do not move); the phase-serial and
    tcgen05 dP, and the pipelined kernel's outputs when the graph's maxima lie in the binade of the batch's, are the same
    bits alone; two identical calls give the same bits for everything, dv and dbias included."""
    g = with_batch(geom)
    case = Fp32Case(cuda_lib, g, seed=1)
    B, N, R, Fe, H, U = g.B, g.N, case.R, g.Fe, g.H, case.U
    # one power of two for the whole batch, so that graphs share the binade of the batch maxima
    case.P_aug[:, :case.HC].view(B, N, U, -1).mul_(torch.exp2(-case.k.float()).view(B, 1, U, 1))
    case.dout.view(B, N, U, -1).mul_(torch.exp2(-case.m.float()).view(B, 1, U, 1))
    HC = case.HC
    P_rows, dout_rows = case.P_aug[:, :HC].view(B, N, HC), case.dout.view(B, N, -1)

    def binade(t):
        return math.frexp(t.abs().max().item())[1]

    for rows in (P_rows, dout_rows):                                # graph B // 2 into the binade of the batch maximum
        rows[B // 2] *= 2.0 ** (binade(rows) - binade(rows[B // 2]))
    same_binade = [b for b in range(B) if binade(P_rows[b]) == binade(P_rows) and binade(dout_rows[b]) == binade(dout_rows)]
    assert B // 2 in same_binade
    kernels = bwd_kernels(N, Fe, H, g.C, R, g.concat)
    f, f2 = case.forward(cuda_lib), case.forward(cuda_lib)
    for k in ("out", "alpha", "terms"):
        assert (f[k] is None and Fe == 0) or same_bits(f[k][..., case.off] if k == "terms" else f[k], f2[k][..., case.off]
                                                       if k == "terms" else f2[k]), ("repeat", k)
    bws = {}
    for algo in kernels:
        bws[algo] = case.backward(cuda_lib, algo, t36=f["t36"])
        again = case.backward(cuda_lib, algo, t36=f2["t36"])
        for k in ("dP", "dv", "d_et36", "dbias"):
            assert (bws[algo][k] is None and Fe == 0) or same_bits(bws[algo][k], again[k]), ("repeat", kernels[algo], k)

    def run(rows_of, graphs, nb):
        P = case.P_aug[rows_of].contiguous()
        ea = case.ea[(graphs.view(-1, 1) * R + torch.arange(R, device=DEV)).reshape(-1)].contiguous() if Fe else None
        fo = case.forward(cuda_lib, B=nb, P_aug=P, ea=ea)
        bo = {algo: case.backward(cuda_lib, algo, t36=fo["t36"], B=nb, P_aug=P, ea=ea, dout=case.dout[rows_of].contiguous())
              for algo in kernels}
        assert same_bits(fo["out"], f["out"][rows_of]), "out"
        assert same_bits(fo["alpha"], f["alpha"][graphs]), "alpha"
        if Fe:                                                      # (the diagonal holds stale values no consumer reads)
            assert same_bits(fo["terms"][..., case.off], f["terms"][graphs][..., case.off]), "edge terms"
        return bo

    perm = torch.randperm(B, generator=torch.Generator().manual_seed(3)).to(DEV)
    rows = (perm.view(B, 1) * N + torch.arange(N, device=DEV)).reshape(-1)
    bo = run(rows, perm, B)
    for algo, kern in kernels.items():
        assert same_bits(bo[algo]["dP"], bws[algo]["dP"][rows]), (kern, "dP_aug rows under permutation")
        if Fe:
            assert same_bits(bo[algo]["d_et36"], bws[algo]["d_et36"][perm]), (kern, "d_edge_terms under permutation")
    alone = sorted({0, B // 2, B - 1})
    for b in alone:
        rows = torch.arange(b * N, (b + 1) * N, device=DEV)
        bo = run(rows, torch.tensor([b], device=DEV), 1)
        for algo, kern in kernels.items():
            if kern == "pipelined" and b not in same_binade:
                continue
            cols = slice(0, HC) if kern != "pipelined" else slice(None)
            assert same_bits(bo[algo]["dP"][:, cols], bws[algo]["dP"][rows][:, cols]), (kern, b, "dP alone")
            if kern == "pipelined" and Fe:
                assert same_bits(bo[algo]["d_et36"], bws[algo]["d_et36"][b:b + 1]), (kern, b, "d_edge_terms alone")


# ======================================================================================== 4. edge_mode 1
@pytest.mark.gpu
def test_structured_edge_source_chain_on_the_fp32_path(cuda_lib):
    """edge_terms_from_windows -> attn_fwd -> the pipelined backward -> windows_dv on p_format 0 at N = 30, H = 6 and
    seq_length 120 (Fe = 360: the 8-slot forward), B = 2G + 1, against fp64 from the reference's edge rows."""
    N, L, H, C_ = 30, 120, 6, 500
    Fe = 3 * L
    B = 2 * sm_count() + 1
    g = Geom(B, N, Fe, H, C_, False)
    assert fwd_plan(N, Fe, H, C_, N * (N - 1), False)["slots"] == 8
    vol, vv = synth.synthetic_matrices(L + B + 2, N, seed=21)
    bt = synth.make_batch(vol, vv, list(range(B)), L)
    case = Fp32Case(cuda_lib, g, seed=2, edge_mode=1)
    assert torch.equal(bt.edge_index.to(DEV), case.edge_index)
    case.ea = bt.edge_attr.float().to(DEV).contiguous()
    case.T = dense_gat.pyg_to_dense_tile(case.ea.double(), case.edge_index, B, N)
    for _ in range(12):                                             # off the LeakyReLU kinks for the new edge rows
        z = case.logits(case.sd)
        near = (z.abs() < 2e-5 * z.abs().max()).any(2).view(B * N, H)
        if not near.any():
            break
        case.sd[:, H:][near] += 1e-4 * z.abs().max().item()
    case.P_aug[:, case.HC:case.HC + 2 * H] = case.sd
    z = case.logits(case.sd)
    assert not (z.abs() < 2e-5 * z.abs().max()).any()
    d = case.desc(PIPELINED)
    vv_g = torch.as_tensor(vv).float().to(DEV).contiguous()
    t0 = torch.arange(B, dtype=torch.int32, device=DEV)
    terms = torch.full((B, H, N, ET_NS), float("nan"), device=DEV)
    wse = C.c_size_t()
    check(cuda_lib.spotv2_edge_terms_from_windows_workspace_bytes(C.byref(d), C.byref(wse)), "edge_terms ws")
    ws_e = torch.empty(max(wse.value, 256), dtype=torch.uint8, device=DEV)
    check(cuda_lib.spotv2_edge_terms_from_windows(C.byref(d), ptr(vv_g), vv_g.shape[0], L, ptr(t0), ptr(case.v), ptr(terms),
                                                  ptr(ws_e), ws_e.numel(), st()), "edge_terms_from_windows")
    torch.cuda.synchronize()
    errs = {"edge terms (windows)": per_graph(terms[..., :N][..., case.off], case.edge_terms()[..., case.off], B)}
    r = case.reference()
    f = case.forward(cuda_lib, terms_in=terms)
    f["terms"] = None                                               # (edge_mode 1: the forward writes no edge terms)
    fe = dict(case.check_forward(dict(f, terms=terms[..., :N]), r))
    errs.update(fe)
    bw = case.backward(cuda_lib, PIPELINED, t36=terms, structured=True)
    dv = torch.full((H, Fe), float("nan"), device=DEV)
    wsz = C.c_size_t()
    check(cuda_lib.spotv2_windows_dv_workspace_bytes(C.byref(d), C.byref(wsz)), "windows_dv ws")
    ws2 = torch.empty(max(wsz.value, 256), dtype=torch.uint8, device=DEV)
    check(cuda_lib.spotv2_windows_dv(C.byref(d), ptr(vv_g), vv_g.shape[0], L, ptr(t0), ptr(bw["d_et36"]), ptr(dv), ptr(ws2),
                                     ws2.numel(), st()), "windows_dv")
    torch.cuda.synchronize()
    bw["dv"] = dv
    errs.update(case.check_backward(bw, r))
    report(f"edge_mode 1, B = {B}", errs)
