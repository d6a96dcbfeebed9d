"""The default pair-format path (p_format 1, gemm_algo 0) stage by stage against float64, with several graphs per CTA.

The projection travels as an fp16 hi | lo pair: proj_fwd_pair writes it, attn_fwd16.cu reads both planes, attn_prep.cu
splits dout into one unit per graph (per (graph, head) for concat layers), the P16 instantiation of attn_bwd2.cu writes dP
back as a padded pair, and proj_bwd_weight / proj_bwd_input read that.  These tests feed the attention kernels operands
built directly as two exact planes, so that P = (hi + lo) * inv is exact in fp64 and in fp32 and the dense fp64 reference
(tests/test_half_precision.py) runs on exactly the P the kernels see:

  hi  fp16, |hi| < 2^15 with the group maximum in [2^14, 2^15); graph b's rows (per head for concat layers) at 2^(k_b - 8)
  lo  fp16, |lo| <= half an ulp of hi, on the grid max(ulp(hi) 2^-12, 2^-24): hi + lo has at most 23 significant bits
  pad columns [C, Cp) zero in both planes; the planes' s|d columns hold the pair of sd at the group-1 scale

dout is plain fp32 with unit u scaled by 2^(m_u), so the prepass's 22-bit split enters the bounds.  Every batch holds
B = G, 2G + 1 or 3G - 5 graphs (G = SM count = the persistent kernels' grid), so CTAs hold one, two, three or four graphs
and some CTAs one more than others.  Errors are taken per graph (max over b of |ours_b - ref_b|_inf / |ref_b|_inf against
the project's 1e-5 bar), and out and dP are also held to elementwise bounds.  With A = 32:

  |out - out64| <= sum_j |a_ij - alpha_ij| |P_j| + A 2^-22 sum_j |alpha_ij| |P_j| + 2^-23 |out64|
  |dP - dP64|   <= sum_i |a_ij - alpha_ij| |dO_i| + A 2^-22 sum_i |alpha_ij| |dO_i| + 2^-23 |dP64| + half an ulp of the stored lo plane * inv
  |ds|dd - ref| <= 1e-5 max_b |ref| + half an ulp of the stored lo plane * inv   (one pair for the whole batch)

a is the kernel's own coefficient tile (held to 1e-5 per graph on its own); its fp32 logits carry the error of the edge
terms' dot products into out and dP through the first term.  The second term gathers the roundings between the exact operands and the fp32 result: the coefficients' hi | lo split at
2^14 (2^-22 relative), dO's split per unit (2^-22 of the element, or 2^-39 of the unit maximum where lo is subnormal),
fp32 accumulation over at most 32 sources, 3 products each, and 8 heads with tensor-core accumulation allowed one ulp
(2^-23) per addition (at most (32 + 8) 2^-23 = 20 * 2^-22), and the fp32 factors 1/H and 1/(1-p) (2^-24 each): 24 * 2^-22
in all, rounded up to A = 32.  The second term covers the final multiply and the bias addition.  The stored pair rounds
the exact dP once more, by at most half an ulp of its lo plane.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import spotv2net_b200 as sv
from spotv2net_b200._lib import GatDesc, check, ptr
from oracle import dense_gat, synth
from test_half_precision import dense_attention, dense_logits, half_ulp_f16, scale_block, workspace

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-5
A_BOUND = 32.0
SEED_LO, SEED_HI = 0x1234567, 0x89ABCDEF          # dropout key: seed_hi != 0 reaches the second key word


def st():
    return torch.cuda.current_stream().cuda_stream


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def graphs(spec):
    """(a, c) -> a G + c graphs."""
    return spec[0] * sm_count() + spec[1]


def per_graph(a, ref, B, scale=None):
    """max over graphs b of |a_b - ref_b|_inf / |ref_b|_inf (rows graph-major; scale: the magnitude to divide by instead of
    |ref|)."""
    a, ref = a.double().reshape(B, -1), ref.double().reshape(B, -1)
    mag = (ref if scale is None else scale.double()).abs().reshape(B, -1).amax(1)
    return ((a - ref).abs().amax(1) / mag.clamp_min(1e-300)).max().item()


def relerr(a, ref):
    a, ref = a.double(), ref.double()
    return ((a - ref).abs().max() / ref.abs().max().clamp_min(1e-300)).item()


# ----------------------------------------------------------------------------------------------- exact operands
def exact_two_planes(shape, e, g):
    """hi | lo fp16 planes of `shape`: hi = fp16(fp16(u 32752) 2^e) with u uniform in (-1, 1) and e <= 0 (broadcast to
    shape); lo = l * max(ulp(hi) 2^-12, 2^-24) with |lo| <= half an ulp of hi.  hi + lo is exact in fp32."""
    base = ((torch.rand(shape, generator=g, device=DEV, dtype=torch.float64) * 2 - 1) * 32752.0).half().double()
    hi = (base * torch.exp2(e.double())).half()
    h = half_ulp_f16(hi)
    unit = torch.clamp(h * 2.0 ** -11, min=2.0 ** -24)
    u = torch.rand(shape, generator=g, device=DEV, dtype=torch.float64) * 2 - 1
    lo64 = torch.round(u * h / unit) * unit
    lo = lo64.half()
    assert torch.equal(lo.double(), lo64) and (lo64.abs() <= h).all()
    assert torch.equal((hi.float() + lo.float()).double(), hi.double() + lo64)       # P = hi + lo: exact in fp32 too
    return hi, lo


def f16_pair_of(t, s):
    """hi = fp16(t s), lo = fp16(t s - hi) (the library's split of an fp32 group at scale s)."""
    hi = (t.double() * s).half()
    return hi, (t.double() * s - hi.double()).half()


def pair_planes(n, H, C_, Cp, ldp16, g0, g1):
    """[2, n, ldp16] planes in the padded layout: group 0 (hi, lo) [n, H, C] at head pitch Cp, group 1 (hi, lo) [n, 2H]."""
    P16 = torch.zeros(2, n, ldp16, device=DEV, dtype=torch.float16)
    for k in range(2):
        P16[k, :, :H * Cp].view(n, H, Cp)[:, :, :C_] = g0[k].reshape(n, H, C_)
        P16[k, :, H * Cp:H * Cp + 2 * H] = g1[k]
    return P16


# --------------------------------------------------------------------------------- the dropout mask, restated
_M0, _M1, _W0, _W1, _MASK = (np.uint64(v) for v in (0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85, 0xFFFFFFFF))


def philox4x32_10(c0, c1, k0, k1):
    """Philox4x32-10 as csrc/attn_common.cuh states it: counter (c0, c1, 0, 0), key (k0, k1); uint64 arithmetic."""
    c0, c1 = c0.astype(np.uint64), c1.astype(np.uint64)
    c2, c3 = np.zeros_like(c0), np.zeros_like(c0)
    k0, k1 = np.uint64(k0), np.uint64(k1)
    for _ in range(10):
        p0, p1 = _M0 * c0, _M1 * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _MASK
        k0, k1 = (k0 + _W0) & _MASK, (k1 + _W1) & _MASK
    return c0, c1, c2, c3


def keep_mask(B, H, N, p, seed_lo, seed_hi):
    """The documented layout (include/spotv2_gat.h, csrc/attn_common.cuh): element e = ((b H + h) N + i) N + j (i target,
    j source) takes lane e & 3 of Philox4x32-10(counter e >> 2, key (seed_lo, seed_hi)); kept iff the draw >= p 2^32.
    Returns keep [B, H, i, j] (bool, on the device)."""
    total = B * H * N * N
    ctr = np.arange((total + 3) // 4, dtype=np.uint64)
    draws = np.stack(philox4x32_10(ctr & _MASK, ctr >> np.uint64(32), seed_lo, seed_hi), axis=1).reshape(-1)[:total]
    t = float(np.float32(p)) * 4294967296.0
    thresh = 0xFFFFFFFF if t >= 4294967295.0 else int(t)
    return torch.from_numpy(draws >= np.uint64(thresh)).view(B, H, N, N).to(DEV)


# --------------------------------------------------------------------------------- one attention case end to end
class Case:
    """Exact two-plane operands, sd off the LeakyReLU kinks, edge rows, dout and the fp64 reference for one geometry."""

    def __init__(self, cuda_lib, B, N, Fe, H, C_, concat, pdrop=0.0, peaked=False, seed=0, edge_mode=0, T=None):
        self.B, self.N, self.Fe, self.H, self.C, self.concat, self.pdrop = B, N, Fe, H, C_, concat, pdrop
        n = self.n = B * N
        self.d = d = GatDesc(B, N, 16, Fe, H, C_, N * (N - 1), int(concat), 0.2, cuda_lib.spotv2_gat_ldp(H, C_), 0, 0, pdrop,
                             edge_mode, SEED_LO, SEED_HI, 1)
        assert cuda_lib.spotv2_gat_pair_format_supported(C.byref(d)) == 1
        self.Cp, self.n_aug = cuda_lib.spotv2_gat_head_pitch(C.byref(d)), cuda_lib.spotv2_gat_n_aug(C.byref(d))
        self.ldp16 = cuda_lib.spotv2_gat_ld16(self.n_aug)
        self.ldo = H * C_ if concat else C_
        U = H if concat else 1
        g = self.g = torch.Generator(device=DEV).manual_seed(1000 * seed + n + C_)
        # per-unit exponents k_b (P) and m_b (dout) in [-8, 8], drawn independently; one unit at 8 puts the group maximum
        # in [2^14, 2^15)
        k = torch.randint(-8, 9, (B, U), generator=g, device=DEV)
        k[0, 0] = 8
        self.m = torch.randint(-8, 9, (B, U), generator=g, device=DEV)
        e = (k - 8).view(B, 1, U, 1).expand(B, N, H, C_)
        hi, lo = exact_two_planes((B, N, H, C_), e, g)
        assert 2.0 ** 14 <= hi.double().abs().max().item() < 2.0 ** 15
        inv0 = 2.0 ** -10
        self.P64 = (hi.double() + lo.double()) * inv0                                       # [B, N, H, C], exact
        # edges and the fp64 edge tile
        if Fe and T is None:
            bt = synth.random_complete_batch(B, N, 1, Fe, seed=5 + seed)
            self.ea = bt.edge_attr.contiguous().to(DEV)
            self.topo = sv.topology_from_edge_index(bt.edge_index.to(DEV), n)
            T = dense_gat.pyg_to_dense_tile(self.ea.double(), bt.edge_index.to(DEV), B, N)
        else:
            self.ea, self.topo = None, None
        self.T = T
        if Fe:
            vs = 0.3 if edge_mode == 0 else 1.0 / (T.abs().max().item() * math.sqrt(Fe))   # edge terms of order 1
            self.v = (torch.randn(H, Fe, device=DEV, generator=g) * vs).contiguous()
        else:
            self.v = None
        sd = torch.randn(n, 2 * H, device=DEV, generator=g) * (4.0 if peaked else 1.0)
        # a logit within fp32 noise of the LeakyReLU kink may fall on either side: move the target term d_i of such a row
        for _ in range(8):
            z = self.logits(sd)
            near = (z.abs() < 1e-4 * z.abs().max()).any(2).view(n, H)
            if not near.any():
                break
            sd[:, H:][near] += 3e-4 * z.abs().max().item()
        self.z = self.logits(sd)
        assert not (self.z.abs() < 1e-4 * self.z.abs().max()).any(), "a logit is left at the LeakyReLU kink"
        self.sd = sd
        s1 = 2.0 ** (15 - math.frexp(sd.abs().max().item())[1])
        self.P16 = pair_planes(n, H, C_, self.Cp, self.ldp16, (hi, lo), f16_pair_of(sd, s1))
        self.pblk = scale_block(self.P64.abs().max().item(), sd.abs().max().item(), inv0, 1.0 / s1)
        self.bias = torch.randn(self.ldo, device=DEV, generator=g)
        dout = torch.randn(n, self.ldo, device=DEV, generator=g).view(B, N, U, C_)
        self.dout = (dout * torch.exp2(self.m.float()).view(B, 1, U, 1)).reshape(n, self.ldo).contiguous()
        etb = C.c_size_t()
        check(cuda_lib.spotv2_gat_edge_terms_bytes(C.byref(d), C.byref(etb)), "edge_terms_bytes")
        self.rec_floats = etb.value // 4
        self.keep = keep_mask(B, H, N, pdrop, SEED_LO, SEED_HI) if pdrop > 0 else None     # [b, h, i, j]

    def logits(self, sd):
        H, B, N = self.H, self.B, self.N
        return dense_logits(sd[:, :H].double().view(B, N, H), sd[:, H:].double().view(B, N, H), self.T,
                            self.v.double() if self.Fe else None)

    def reference(self):
        B, N, H = self.B, self.N, self.H
        mask = self.keep.permute(0, 2, 3, 1) if self.keep is not None else None             # [b, i, j, h]
        return dense_attention(self.P64, self.sd[:, :H].double().view(B, N, H), self.sd[:, H:].double().view(B, N, H), self.T,
                               self.v.double() if self.Fe else None, self.bias.double(), self.dout.double(), H, self.concat,
                               0.2, mask, 1.0 / (1.0 - self.pdrop))

    def edge_terms(self):
        """<e_ij, v_h> in the record's layout [B, H, j, i] (fp64)."""
        return torch.einsum("bijf,hf->bhji", self.T, self.v.double())

    def forward(self, cuda_lib, d=None, P16=None, sd=None, ea=None, rec=None):
        """attn_fwd_pair with NaN-prefilled outputs.  edge_mode 1: rec holds the edge terms and ea is not passed."""
        d = d or self.d
        P16 = self.P16 if P16 is None else P16
        sd = self.sd if sd is None else sd
        ea = self.ea if ea is None else ea
        n = d.B * d.N
        if rec is None and self.Fe:
            rec = torch.full((self.rec_floats // self.B * d.B,), float("nan"), device=DEV)
        out = torch.full((n, self.ldo), float("nan"), device=DEV)
        alpha = torch.full((d.B, self.H, self.N, self.N), float("nan"), device=DEV)
        rows_in = self.Fe and d.edge_mode == 0
        check(cuda_lib.spotv2_gat_attn_fwd_pair(C.byref(d), ptr(P16[0]), ptr(P16[1]), ptr(self.pblk), ptr(sd),
                                                ptr(ea) if rows_in else None, ptr(self.topo.table) if rows_in else None,
                                                ptr(self.v), ptr(self.bias), ptr(out), ptr(alpha), ptr(rec), st()), "attn_fwd_pair")
        torch.cuda.synchronize()
        return dict(out=out, alpha=alpha, rec=rec)

    def backward(self, cuda_lib, rec):
        d, n, H, Fe = self.d, self.n, self.H, self.Fe
        rows_in = Fe and d.edge_mode == 0
        dP16 = torch.full((2, n, self.ldp16), float("nan"), device=DEV, dtype=torch.float16)
        dblk = torch.full((8,), float("nan"), device=DEV)
        dv = torch.full((H, Fe), float("nan"), device=DEV) if rows_in else None
        d_et = torch.full_like(rec, float("nan")) if Fe else None
        dbias = torch.full((self.ldo,), float("nan"), device=DEV)
        ws = workspace(cuda_lib, d)
        check(cuda_lib.spotv2_gat_attn_bwd_pair(C.byref(d), ptr(self.P16[0]), ptr(self.P16[1]), ptr(self.pblk), ptr(self.sd),
                                                ptr(self.ea) if rows_in else None, ptr(rec),
                                                ptr(self.topo.table) if rows_in else None, ptr(self.v), ptr(self.dout),
                                                ptr(dP16[0]), ptr(dP16[1]), ptr(dblk), ptr(dv), ptr(d_et), ptr(dbias), ptr(ws),
                                                ws.numel(), st()), "attn_bwd_pair")
        torch.cuda.synchronize()
        return dict(dP16=dP16, dblk=dblk, dv=dv, d_et=d_et, dbias=dbias)

    # ------------------------------------------------------------------------------------------------ checks
    def alpha_error(self, f, r):
        """|alpha - alpha64| [b, i, j, h] with the kernel's own coefficients (checked on their own against the bar): their
        error reaches out and dP through sum |alpha - alpha64| |P| and sum |alpha - alpha64| |dO|."""
        return (f["alpha"].double() - r["alpha"].permute(0, 3, 2, 1)).abs().permute(0, 3, 2, 1)

    def check_forward(self, f, r):
        B, N, H, Fe = self.B, self.N, self.H, self.Fe
        n = self.n
        errs = {}
        assert torch.isfinite(f["out"]).all() and torch.isfinite(f["alpha"]).all()
        if self.keep is not None:                                    # the zero pattern of alpha is the documented mask
            assert torch.equal(f["alpha"] != 0, self.keep.transpose(2, 3)), "dropout mask differs from its documented layout"
        errs["alpha"] = per_graph(f["alpha"], r["alpha"].permute(0, 3, 2, 1), B)
        errs["out"] = per_graph(f["out"], r["out"], B)
        eP = torch.einsum("bijh,bjhc->bihc", self.alpha_error(f, r), self.P64.abs())
        aP, eP = [t.reshape(n, H * self.C) if self.concat else t.mean(2).reshape(n, self.C) for t in (r["aP"], eP)]
        floor = 2.0 ** -30 * aP.view(B, -1).amax(1).repeat_interleave(N).view(n, 1)
        b_out = eP + A_BOUND * 2.0 ** -22 * aP + 2.0 ** -23 * r["out"].abs() + floor
        e_out = (f["out"].double() - r["out"]).abs()
        errs["out/bound"] = (e_out / b_out).max().item()
        if Fe:
            rec = f["rec"].view(B, H, N, 36)
            assert torch.isfinite(rec).all()                        # every byte of the record is written
            if self.pdrop > 0:                                      # with dropout the record is the edge terms
                off = ~torch.eye(N, dtype=torch.bool, device=DEV)
                errs["record"] = per_graph(rec[..., :N][..., off], self.edge_terms()[..., off], B)
            else:                                                   # |record| = alpha bit for bit, sign = LeakyReLU side
                assert torch.equal(rec[..., :N].abs(), f["alpha"]), "record magnitude differs from alpha"
                assert torch.equal(torch.signbit(rec[..., :N]), self.z.permute(0, 3, 2, 1) <= 0), "record sign"
                assert (rec[..., N:] == 0).all(), "record pad columns"
        return errs

    def check_backward(self, bw, r, f, dv=None):
        """f: the forward's outputs (the backward reads the same coefficients: the record, or the same recomputation)."""
        B, N, H, C_, Cp, n, Fe = self.B, self.N, self.H, self.C, self.Cp, self.n, self.Fe
        HCp = H * Cp
        errs = {}
        dP16, dblk = bw["dP16"], bw["dblk"]
        assert torch.isfinite(dP16[:, :, :self.n_aug].float()).all()
        assert (dP16[:, :, :HCp].reshape(2, n, H, Cp)[..., C_:] == 0).all(), "dP pad columns are not zero"
        hi0, lo0 = dP16[0, :, :HCp].reshape(n, H, Cp)[..., :C_], dP16[1, :, :HCp].reshape(n, H, Cp)[..., :C_]
        inv0, inv1 = dblk[2].item(), dblk[3].item()
        got0 = (hi0.double() + lo0.double()) * inv0
        ref0 = r["dP"].reshape(n, H, C_)
        errs["dP"] = per_graph(got0, ref0, B)
        adO = r["adO"].reshape(n, H, C_)
        edO = torch.einsum("bijh,bihc->bjhc", self.alpha_error(f, r), r["dO"].abs()).reshape(n, H, C_)
        floor = 2.0 ** -30 * adO.reshape(B, -1).amax(1).repeat_interleave(N).view(n, 1, 1)
        b0 = edO + A_BOUND * 2.0 ** -22 * adO + 2.0 ** -23 * ref0.abs() + half_ulp_f16(lo0) * inv0 + floor
        errs["dP/bound"] = ((got0 - ref0).abs() / b0).max().item()
        # ds | dd: fp32 sums (the 1e-5 bar, per graph), then ONE pair for the whole batch at the group's own scale, whose
        # absolute resolution is half an ulp of the stored lo plane (2^-25 / s where lo is subnormal): a graph whose ds | dd
        # lie 2^32 below the batch maximum (k_b = m_b = -8 against 8) keeps 1e-5 of its own maximum only down to that floor
        hi1, lo1 = dP16[0, :, HCp:self.n_aug], dP16[1, :, HCp:self.n_aug]
        got1 = (hi1.double() + lo1.double()) * inv1
        ref1 = torch.cat([r["ds"].reshape(n, H), r["dd"].reshape(n, H)], 1)
        b1 = TOL * ref1.view(B, -1).abs().amax(1).repeat_interleave(N).view(n, 1) + half_ulp_f16(lo1) * inv1
        errs["ds|dd/bound"] = ((got1 - ref1).abs() / b1).max().item()
        errs["dbias"] = relerr(bw["dbias"], r["dbias"])
        if Fe:
            # dz'_ij = dz_ij + dz_ii / (N - 1) in fp32: per graph against the magnitude of its terms (at N = 2 the softmax
            # makes the two cancel exactly wherever both logits share a LeakyReLU side, so |dz'| itself can be 0)
            dz = r["dz"]
            diag = torch.diagonal(dz, dim1=1, dim2=2).permute(0, 2, 1).abs()
            terms = (dz.abs() + diag.unsqueeze(2) / max(N - 1, 1)).permute(0, 3, 2, 1)
            errs["dz'"] = per_graph(bw["d_et"].view(B, H, N, 36)[..., :N], r["dzp"].permute(0, 3, 2, 1), B, scale=terms)
            errs["dv"] = relerr(bw["dv"] if dv is None else dv, r["dv"])
        return errs


def assert_errors(label, errs):
    print(f"{label}: " + ", ".join(f"{k} {e:.2e}" for k, e in errs.items()))
    bad = {k: e for k, e in errs.items() if e > (1.0 if k.endswith("/bound") else TOL)}
    assert not bad, (label, bad)


# ======================================================================================== 1. stages against fp64
STAGE_GEOMS = [
    # (a, c): B = a G + c;  N, Fe, H, C, concat, dropout p, peaked rows
    ((1, 0), 30, 126, 6, 500, False, 0.0, False),     # the default geometry (the kernel's specialised instance)
    ((2, 1), 30, 126, 8, 256, True, 0.0, False),      # config C layer 0
    ((3, -5), 30, 126, 8, 256, False, 0.0, False),    # config C layer 1
    ((3, -5), 30, 126, 7, 20, False, 0.0, False),     # C = 20 -> Cp = 24, odd H
    ((2, 1), 30, 126, 7, 24, True, 0.0, False),       # concat C = 24, odd H
    ((2, 1), 32, 12, 8, 16, False, 0.0, False),       # N = 32
    ((1, 0), 31, 10, 6, 20, False, 0.0, False),       # N = 31
    ((3, -5), 13, 5, 7, 20, False, 0.0, False),       # N = 13
    ((2, 1), 2, 4, 8, 8, True, 0.0, False),           # N = 2
    ((2, 1), 30, 0, 4, 36, False, 0.0, False),        # no edge features
    ((1, 0), 30, 384, 2, 16, False, 0.0, False),      # Fe = 384
    ((1, 0), 30, 126, 2, 1024, False, 0.0, False),    # C = 1024
    ((2, 1), 30, 126, 6, 20, False, 0.3, False),      # attention dropout
    ((2, 1), 30, 126, 6, 20, False, 0.9, True),       # dropout 0.9 on peaked rows
    ((2, 1), 30, 12, 8, 16, False, 0.5, False),       # the dropout mask layout at p = 0.5, H = 8
]


def geom_id(g_):
    (a, c), N, Fe, H, C_, cat, p, peaked = g_
    b = "G" if (a, c) == (1, 0) else f"{a}G{c:+d}"
    return f"B{b}N{N}Fe{Fe}H{H}C{C_}{'cat' if cat else 'mean'}" + (f"_p{p:g}" if p else "") + ("_peaked" if peaked else "")


@pytest.mark.parametrize("geom", STAGE_GEOMS, ids=geom_id)
def test_pair_attention_stages_against_fp64(cuda_lib, geom):
    spec, N, Fe, H, C_, concat, pdrop, peaked = geom
    case = Case(cuda_lib, graphs(spec), N, Fe, H, C_, concat, pdrop, peaked)
    r = case.reference()
    f = case.forward(cuda_lib)
    bw = case.backward(cuda_lib, f["rec"])
    errs = case.check_forward(f, r)
    errs.update(case.check_backward(bw, r, f))
    assert_errors(f"{geom_id(geom)} (B = {case.B})", errs)


# ======================================================================================== 2. cross-graph invariants
@pytest.mark.parametrize("geom", [((2, 1), 30, 126, 6, 500, False), ((2, 1), 30, 126, 8, 256, True)],
                         ids=["default", "configC_l0"])
def test_pair_forward_is_independent_of_batch_position(cuda_lib, geom):
    """With the same scale block and sd, a graph's out, alpha and record are the same bits whether it runs alone or at
    position b of a batch of 2G + 1, and a permutation of the graphs permutes them."""
    spec, N, Fe, H, C_, concat = geom
    case = Case(cuda_lib, graphs(spec), N, Fe, H, C_, concat, seed=1)
    B, G, R = case.B, sm_count(), N * (N - 1)
    full = case.forward(cuda_lib)
    rec = full["rec"].view(B, H, N, 36)
    for b in sorted({0, 1, G - 1, G, 2 * G, B - 1}):
        d1 = GatDesc.from_buffer_copy(case.d)
        d1.B = 1
        rows = slice(b * N, (b + 1) * N)
        one = case.forward(cuda_lib, d=d1, P16=case.P16[:, rows].contiguous(), sd=case.sd[rows].contiguous(),
                           ea=case.ea[b * R:(b + 1) * R].contiguous())
        assert torch.equal(one["out"], full["out"][rows]), ("out", b)
        assert torch.equal(one["alpha"][0], full["alpha"][b]), ("alpha", b)
        assert torch.equal(one["rec"].view(H, N, 36), rec[b]), ("record", b)
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(3)).to(DEV)
    rows = (perm.view(B, 1) * N + torch.arange(N, device=DEV)).reshape(-1)
    erows = (perm.view(B, 1) * R + torch.arange(R, device=DEV)).reshape(-1)
    pm = case.forward(cuda_lib, P16=case.P16[:, rows].contiguous(), sd=case.sd[rows].contiguous(), ea=case.ea[erows].contiguous())
    assert torch.equal(pm["out"], full["out"][rows])
    assert torch.equal(pm["alpha"], full["alpha"][perm])
    assert torch.equal(pm["rec"].view(B, H, N, 36), rec[perm])


# ======================================================================================== 3. the dropout mask layout
def test_host_philox_matches_the_documented_mask_statistics():
    """The host restatement itself: the published Philox4x32-10 answer for counter 0 and key 0 (Random123), the keep rate,
    and lanes 0..3 of one counter are four different draws."""
    kat = philox4x32_10(np.zeros(1, dtype=np.uint64), np.zeros(1, dtype=np.uint64), 0, 0)
    assert [int(w[0]) for w in kat] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    keep = keep_mask(7, 3, 30, 0.5, SEED_LO, SEED_HI).cpu()
    assert abs(keep.double().mean().item() - 0.5) < 0.01
    c = philox4x32_10(np.arange(4, dtype=np.uint64), np.zeros(4, dtype=np.uint64), SEED_LO, SEED_HI)
    assert len({int(x) for x in np.stack(c).reshape(-1)}) == 16


@pytest.mark.parametrize("N", [30, 40], ids=["N30", "N40_large_graph_path"])
def test_fp32_format_dropout_mask_matches_its_documented_layout(cuda_lib, N):
    """attn_fwd (p_format 0; N = 40 takes the several-CTAs-per-graph kernel): the zero pattern of alpha is the host
    Philox mask, element for element, at B = 2G + 1, H = 8, p = 0.5 and a key with seed_hi != 0."""
    B, Fe, H, C_ = graphs((2, 1)), 12, 8, 16
    n = B * N
    d = GatDesc(B, N, 16, Fe, H, C_, N * (N - 1), 0, 0.2, cuda_lib.spotv2_gat_ldp(H, C_), 0, 0, 0.5, 0, SEED_LO, SEED_HI, 0)
    g = torch.Generator(device=DEV).manual_seed(N)
    P_aug = torch.randn(n, d.ldp, device=DEV, generator=g)
    bt = synth.random_complete_batch(B, N, 1, Fe, seed=2)
    ea = bt.edge_attr.contiguous().to(DEV)
    topo = sv.topology_from_edge_index(bt.edge_index.to(DEV), n)
    v = torch.randn(H, Fe, device=DEV, generator=g) * 0.3
    out = torch.full((n, C_), float("nan"), device=DEV)
    alpha = torch.full((B, H, N, N), float("nan"), device=DEV)
    wsb = C.c_size_t()
    check(cuda_lib.spotv2_gat_attn_fwd_workspace_bytes(C.byref(d), C.byref(wsb)), "attn_fwd_workspace_bytes")
    ws = torch.empty(max(wsb.value, 256), dtype=torch.uint8, device=DEV)
    check(cuda_lib.spotv2_gat_attn_fwd(C.byref(d), ptr(P_aug), ptr(ea), ptr(topo.table), ptr(v), None, ptr(out), ptr(alpha),
                                       None, ptr(ws), ws.numel(), st()), "attn_fwd")
    torch.cuda.synchronize()
    keep = keep_mask(B, H, N, 0.5, SEED_LO, SEED_HI)
    assert torch.isfinite(alpha).all()
    assert torch.equal(alpha != 0, keep.transpose(2, 3))


# ======================================================================================== 4. edge_mode 1 on the pair path
def test_structured_edge_source_chain_on_the_pair_path(cuda_lib):
    """edge_terms_from_windows -> attn_fwd_pair (overwrites the edge terms with its record) -> attn_bwd_pair -> windows_dv
    at B = 2G + 1 and the default geometry, against fp64 from the reference's edge rows of the same windows."""
    N, L, H, C_ = 30, 42, 6, 500
    Fe = 3 * L
    B = graphs((2, 1))
    vol, vv = synth.synthetic_matrices(L + B + 2, N, seed=21)
    bt = synth.make_batch(vol, vv, list(range(B)), L)
    T = dense_gat.pyg_to_dense_tile(bt.edge_attr.double().to(DEV), bt.edge_index.to(DEV), B, N)
    case = Case(cuda_lib, B, N, Fe, H, C_, False, seed=2, edge_mode=1, T=T)
    d = case.d
    vv_g = torch.as_tensor(vv).float().to(DEV).contiguous()
    t0 = torch.arange(B, dtype=torch.int32, device=DEV)
    terms = torch.full((case.rec_floats,), float("nan"), device=DEV)
    wse = C.c_size_t()
    check(cuda_lib.spotv2_edge_terms_from_windows_workspace_bytes(C.byref(d), C.byref(wse)), "edge_terms ws")
    ws_e = torch.empty(max(wse.value, 256), dtype=torch.uint8, device=DEV)
    check(cuda_lib.spotv2_edge_terms_from_windows(C.byref(d), ptr(vv_g), vv_g.shape[0], L, ptr(t0), ptr(case.v), ptr(terms),
                                                  ptr(ws_e), ws_e.numel(), st()), "edge_terms_from_windows")
    torch.cuda.synchronize()
    off = ~torch.eye(N, dtype=torch.bool, device=DEV)
    errs = {"edge terms": per_graph(terms.view(B, H, N, 36)[..., :N][..., off], case.edge_terms()[..., off], B)}
    r = case.reference()
    f = case.forward(cuda_lib, rec=terms)                            # the record replaces the edge terms in place
    errs.update(case.check_forward(f, r))
    bw = case.backward(cuda_lib, terms)
    dv = torch.full((H, Fe), float("nan"), device=DEV)
    wsz = C.c_size_t()
    check(cuda_lib.spotv2_windows_dv_workspace_bytes(C.byref(d), C.byref(wsz)), "windows_dv ws")
    ws2 = torch.empty(max(wsz.value, 256), dtype=torch.uint8, device=DEV)
    check(cuda_lib.spotv2_windows_dv(C.byref(d), ptr(vv_g), vv_g.shape[0], L, ptr(t0), ptr(bw["d_et"]), ptr(dv), ptr(ws2),
                                     ws2.numel(), st()), "windows_dv")
    torch.cuda.synchronize()
    errs.update(case.check_backward(bw, r, f, dv=dv))
    assert_errors(f"edge_mode 1, B = {B}", errs)


# ======================================================================================== 5. pair projections at batch scale
PROJ = (4097, 30, 1260, 6, 500)                  # 122 910 rows: 961 row tiles of 128, an odd count, many waves


def per_block(a, ref, rows=128):
    """max over blocks of `rows` rows of |a - ref|_inf / |ref|_inf."""
    n = a.shape[0]
    diff = (a.double() - ref.double()).abs().reshape(n, -1).amax(1)
    mag = ref.double().abs().reshape(n, -1).amax(1)
    pad = (-n) % rows
    diff, mag = F.pad(diff, (0, pad)).view(-1, rows).amax(1), F.pad(mag, (0, pad)).view(-1, rows).amax(1)
    return (diff / mag.clamp_min(1e-300)).max().item()


def projection_operands(cuda_lib):
    B, N, Fin, H, C_ = PROJ
    n = B * N
    d = GatDesc(B, N, Fin, 0, H, C_, 0, 0, 0.2, cuda_lib.spotv2_gat_ldp(H, C_), 0, 0, 0.0, 0, 0, 0, 1)
    Cp, n_aug = cuda_lib.spotv2_gat_head_pitch(C.byref(d)), cuda_lib.spotv2_gat_n_aug(C.byref(d))
    g = torch.Generator(device=DEV).manual_seed(17)
    x = torch.randn(n, Fin, device=DEV, generator=g) * 3.0
    W = torch.randn(H * C_, Fin, device=DEV, generator=g) * 0.05
    a_s, a_d = torch.randn(1, H, C_, device=DEV, generator=g), torch.randn(1, H, C_, device=DEV, generator=g)
    W_aug = torch.empty(n_aug, Fin, device=DEV)
    check(cuda_lib.spotv2_gat_fold(C.byref(d), ptr(W), ptr(a_s), ptr(a_d), None, None, ptr(W_aug), None, st()), "fold")
    ldx = cuda_lib.spotv2_gat_ld16(Fin)
    x16, xblk = torch.empty(2, n, ldx, device=DEV, dtype=torch.float16), torch.empty(8, device=DEV)
    check(cuda_lib.spotv2_split_f16(ptr(x), n, Fin, Fin, 0, 0, ptr(x16[0]), ptr(x16[1]), ldx, ptr(xblk), st()), "split_f16")
    return d, Cp, n_aug, g, x, W_aug, x16, xblk


def test_pair_projection_forward_at_batch_scale(cuda_lib):
    """proj_fwd_pair over 961 row tiles: hi + lo to 1e-5 of every 128-row block's max|P|, pad columns exactly zero, the
    fp32 s | d terms and their copy in the planes' second group to 1e-5 per block, the a-priori bound holds."""
    d, Cp, n_aug, g, x, W_aug, x16, xblk = projection_operands(cuda_lib)
    B, N, Fin, H, C_ = PROJ
    n, HCp = B * N, H * Cp
    ldp16 = cuda_lib.spotv2_gat_ld16(n_aug)
    P16 = torch.full((2, n, ldp16), float("nan"), device=DEV, dtype=torch.float16)
    pblk, sd = torch.full((8,), float("nan"), device=DEV), torch.full((n, 2 * H), float("nan"), device=DEV)
    ws = workspace(cuda_lib, d)
    check(cuda_lib.spotv2_proj_fwd_pair(C.byref(d), ptr(x16[0]), ptr(x16[1]), ptr(xblk), ptr(W_aug), ptr(P16[0]), ptr(P16[1]),
                                        ptr(pblk), ptr(sd), ptr(ws), ws.numel(), st()), "proj_fwd_pair")
    torch.cuda.synchronize()
    ref = x.double() @ W_aug.double().t()
    full = P16[0, :, :n_aug].double() + P16[1, :, :n_aug].double()
    assert torch.isfinite(full).all()
    errs = {"P": per_block(full[:, :HCp] * pblk[2].item(), ref[:, :HCp]),
            "sd": per_block(sd, ref[:, HCp:]),
            "planes s|d": per_block(full[:, HCp:] * pblk[3].item(), ref[:, HCp:])}
    assert (full[:, :HCp].view(n, H, Cp)[:, :, C_:] == 0).all()
    assert ref[:, :HCp].abs().max() <= pblk[0].item() and ref[:, HCp:].abs().max() <= pblk[1].item()
    assert full.abs().max() < 32768.0 and pblk[4].item() * pblk[2].item() == 1.0
    assert_errors(f"proj_fwd_pair at {n} rows, per 128-row block", errs)


def test_pair_projection_backward_at_batch_scale(cuda_lib):
    """proj_bwd_weight / proj_bwd_input from an exact padded dP pair (two planes built as for the attention tests, 128-row
    blocks at 2^(k - 8), pad columns zero) against float64 matmuls on the device: dW over the split-K reduction, dX per
    128-row block."""
    d, Cp, n_aug, g, x, W_aug, x16, xblk = projection_operands(cuda_lib)
    B, N, Fin, H, C_ = PROJ
    n, HCp = B * N, H * Cp
    splits = cuda_lib.spotv2_diag_weight_grad_splits(n, n_aug, Fin)
    assert splits > 1
    k = torch.randint(-8, 9, (-(-n // 128),), generator=g, device=DEV)
    k[0] = 8
    e = (k - 8).repeat_interleave(128)[:n]
    hi0, lo0 = exact_two_planes((n, H, C_), e.view(n, 1, 1).expand(n, H, C_), g)
    hi1, lo1 = exact_two_planes((n, 2 * H), e.view(n, 1).expand(n, 2 * H), g)
    inv0, inv1 = 2.0 ** -15, 2.0 ** -13
    ldp16 = cuda_lib.spotv2_gat_ld16(n_aug)
    dP16 = pair_planes(n, H, C_, Cp, ldp16, (hi0, lo0), (hi1, lo1))
    dblk = scale_block(1.0, 4.0, inv0, inv1)
    dP64 = torch.zeros(n, n_aug, device=DEV, dtype=torch.float64)
    dP64[:, :HCp].view(n, H, Cp)[:, :, :C_] = (hi0.double() + lo0.double()) * inv0
    dP64[:, HCp:] = (hi1.double() + lo1.double()) * inv1
    ws = workspace(cuda_lib, d)
    dW = torch.full((n_aug, Fin), float("nan"), device=DEV)
    check(cuda_lib.spotv2_proj_bwd_weight(C.byref(d), None, ptr(x16[0]), ptr(x16[1]), ptr(xblk), None, ptr(dP16[0]), ptr(dP16[1]),
                                          ptr(dblk), ptr(dW), ptr(ws), ws.numel(), st()), "proj_bwd_weight")
    dX = torch.full((n, Fin), float("nan"), device=DEV)
    check(cuda_lib.spotv2_proj_bwd_input(C.byref(d), None, ptr(dP16[0]), ptr(dP16[1]), ptr(dblk), ptr(W_aug), ptr(dX), ptr(ws),
                                         ws.numel(), st()), "proj_bwd_input")
    torch.cuda.synchronize()
    dW64 = dP64.t() @ x.double()
    dX64 = dP64 @ W_aug.double()
    errs = {"dW": relerr(dW, dW64), "dW (s|d rows)": relerr(dW[HCp:], dW64[HCp:]), "dX": per_block(dX, dX64)}
    assert (dW[:HCp].view(H, Cp, Fin)[:, C_:] == 0).all()                           # the pad rows receive nothing
    assert_errors(f"proj_bwd at {n} rows (weight gradient split-K {splits})", errs)
