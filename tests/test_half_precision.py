"""The half-precision class (gemm_algo 3: layer.precision = "half", GATModel.set_precision("half")) against exact references.

The class issues one fp16 tensor-core product per projection (hi planes only) and, with p_format 1, carries P, alpha,
dout and dP as single fp16 planes.  Its loose end-to-end bars (4e-3 / 2e-2) cannot tell a subtle error from rounding, so
these tests choose operands that are exactly representable in fp16 - small integers times powers of two - where the class
loses nothing at its input roundings.  What is left against float64 then comes from a short list of known roundings:

  A. the 1-CTA single-product GEMM (proj_fwd, proj_fwd_pair, proj_bwd_weight, proj_bwd_input): every partial sum is an
     integer multiple of the product unit below 2^24 units, so fp32 accumulation is exact and the results must equal the
     float64 reference bit for bit - at one row tile, odd multi-wave tile counts, ragged n_aug and F, split-K and both
     config C layers at B = 4096.  The 3-product class on the same operands (lo planes zero) must give the same bits.
  B. the single-plane attention kernels (attn_fwd_pair / attn_bwd_pair with hi planes only) against a dense fp64 forward
     and backward from the GIVEN P: alpha, dv, dz' and dbias to 1e-5; out, dP and ds|dd within elementwise bounds made of
     the alpha -> fp16 rounding and half an fp16 ulp at the dP scale.
  C. GATConv / GATModel in half mode through autograd against an fp64 emulation that rounds to fp16 exactly where the
     kernels round (x and W_aug at their group scales, P and alpha in p_format 1, dP and ds|dd in both formats).
"""
import ctypes as C
import math

import pytest
import torch

import spotv2net_b200 as sv
from spotv2net_b200._lib import GatDesc, check, ptr
from oracle import dense_gat, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def st():
    return torch.cuda.current_stream().cuda_stream


def relerr(a, ref):
    a, ref = torch.as_tensor(a).double().cpu(), torch.as_tensor(ref).double().cpu()
    return ((a - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


def ints(shape, g, lo=-8, hi=8, device=DEV):
    """Integers in [lo, hi] as float32 (exact in fp16 up to 2048)."""
    return torch.randint(lo, hi + 1, shape, generator=g, device=device).float()


def pow2_scale(amax: float) -> float:
    """The library's group-scale rule: the power of two that maps amax into [2^14, 2^15)."""
    if not amax > 0 or not math.isfinite(amax):
        return 1.0
    return 2.0 ** (15 - math.frexp(amax)[1])


def f16_at(t: torch.Tensor, s) -> torch.Tensor:
    """float64 emulation of fp16(t * s) / s: 11 significant bits, round to nearest even, fp16 subnormals below 2^-14."""
    y = t.double() * s
    e = torch.frexp(y.abs().clamp_min(2.0 ** -40))[1]
    ulp = torch.exp2((torch.clamp(e, min=-13) - 11).double())
    return torch.round(y / ulp) * ulp / s


def half_ulp_f16(v: torch.Tensor) -> torch.Tensor:
    """Half an ulp of stored fp16 values (float64)."""
    a = v.double().abs()
    e = torch.frexp(a.clamp_min(2.0 ** -40))[1]
    return torch.exp2((torch.clamp(e, min=-13) - 12).double())


def scale_block(bound0, bound1, inv0, inv1):
    """8-float scale block {bound bits x2, inverse scales x2, scales x2, -, -}."""
    return torch.tensor([bound0, bound1, inv0, inv1, 1.0 / inv0, 1.0 / inv1, 0.0, 0.0], device=DEV, dtype=torch.float32)


# ==================================================================== A. the 1-CTA single-product GEMM
def half_class_splits(rows, m, n, sms):
    """weight_grad_splits(rows, m, n, pair_tiles=false) (csrc/gemm.cuh) restated: the half class runs 128 x 256 tiles over
    the SMs; the 3-product class 256 x 256 pair tiles over the resident CTA pairs."""
    base = min(max((rows + 8191) // 8192, 1), 32)
    if base == 1:
        return 1
    tiles = -(-m // 128) * -(-n // 256)
    best, best_eff = base, 0.0
    s = base
    while s <= base + base // 4 + 1 and s <= 32:
        items = tiles * s
        eff = items / (-(-items // sms) * sms)
        if eff > best_eff + 1e-9:
            best, best_eff = s, eff
        s += 1
    return best


def gemm_desc(cuda_lib, B, N, Fin, H, C_, algo, pf):
    return GatDesc(B, N, Fin, 0, H, C_, 0, 0, 0.2, cuda_lib.spotv2_gat_ldp(H, C_), algo, 0, 0.0, 0, 0, 0, pf)


def exact_gemm_operands(cuda_lib, B, N, Fin, H, C_, pf, seed):
    """x: integers in [-8, 8] * 2^-3; W_aug: integers * 2^-5 on the projection rows, * 2^2 on the s|d rows (their own
    power of two), pad rows of the head pitch zero."""
    d = gemm_desc(cuda_lib, B, N, Fin, H, C_, 3, pf)
    Cp, n_aug = cuda_lib.spotv2_gat_head_pitch(C.byref(d)), cuda_lib.spotv2_gat_n_aug(C.byref(d))
    HC = H * Cp
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = ints((B * N, Fin), g) * 2.0 ** -3
    W_aug = ints((n_aug, Fin), g) * 2.0 ** -5
    W_aug[HC:] *= 2.0 ** 7
    W_aug[:HC].view(H, Cp, Fin)[:, C_:] = 0.0
    return d, Cp, n_aug, HC, x, W_aug


def x_pair(cuda_lib, x):
    n, Fin = x.shape
    ldx = cuda_lib.spotv2_gat_ld16(Fin)
    x16, xblk = torch.zeros(2, n, ldx, device=DEV, dtype=torch.float16), torch.zeros(8, device=DEV)
    check(cuda_lib.spotv2_split_f16(ptr(x), n, Fin, Fin, 0, 0, ptr(x16[0]), ptr(x16[1]), ldx, ptr(xblk), st()), "split_f16")
    return x16, xblk


def workspace(cuda_lib, d):
    a, b, c = C.c_size_t(), C.c_size_t(), C.c_size_t()
    check(cuda_lib.spotv2_gat_workspace_bytes(C.byref(d), C.byref(a), C.byref(b), C.byref(c)), "workspace_bytes")
    return torch.empty(max(a.value, b.value, c.value), dtype=torch.uint8, device=DEV)


def with_algo(d, algo):
    e = GatDesc.from_buffer_copy(d)
    e.gemm_algo = algo
    return e


GEMM_SHAPES = [
    # B, N, F, H, C
    (4, 30, 1260, 8, 256),          # one 128-row tile (120 rows)
    (700, 30, 90, 3, 20),           # 21 000 rows = 165 row tiles: an odd count over several waves; F = 90, Cp = 24
    (5, 7, 33, 5, 12),              # ragged n_aug, F = 33, Cp = 16
    (4096, 30, 1260, 8, 256),       # config C layer 0 at the full batch
    (4096, 30, 2048, 8, 256),       # config C layer 1 at the full batch
]


@pytest.mark.parametrize("shape", GEMM_SHAPES, ids=lambda s: "B%dN%dF%dH%dC%d" % s)
def test_single_product_gemms_are_exact_on_fp16_exact_operands(cuda_lib, shape):
    B, N, Fin, H, C_ = shape
    n = B * N
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    report = {}
    for pf in (0, 1):
        d, Cp, n_aug, HC, x, W_aug = exact_gemm_operands(cuda_lib, B, N, Fin, H, C_, pf, seed=Fin + pf)
        splits = half_class_splits(n, n_aug, Fin, sms)
        report[pf] = (splits, cuda_lib.spotv2_diag_weight_grad_splits(n, n_aug, Fin))
        P64 = x.double() @ W_aug.double().t()                                      # exact: every operand is fp16-exact
        g = torch.Generator(device=DEV).manual_seed(7 + pf)
        # dP: integers * 2^-9 on the projection columns, * 2^-12 on ds|dd (pad columns zero); p_format 1 as a hi plane
        # with inverse scales 2^-20 / 2^-23 (the same values)
        dP_int = ints((n, n_aug), g)
        dP_int[:, :HC].view(n, H, Cp)[:, :, C_:] = 0.0
        if pf == 0:
            dP_val = torch.cat([dP_int[:, :HC] * 2.0 ** -9, dP_int[:, HC:] * 2.0 ** -12], 1)
        else:
            dP_val = torch.cat([dP_int[:, :HC] * 2.0 ** -20, dP_int[:, HC:] * 2.0 ** -23], 1)
        dW64 = dP_val.double().t() @ x.double()
        dX64 = dP_val.double() @ W_aug.double()
        outs = {}
        for algo in (3, 0):                     # the half class, then the 3-product class on the same operands
            da = with_algo(d, algo)
            ws = workspace(cuda_lib, da)
            r = {}
            if pf == 0:
                P = torch.full((n, d.ldp), float("nan"), device=DEV)
                pmax = torch.zeros(8, device=DEV)
                check(cuda_lib.spotv2_proj_fwd(C.byref(da), ptr(x), None, None, None, ptr(W_aug), ptr(P), ptr(pmax), ptr(ws),
                                               ws.numel(), st()), "proj_fwd")
                r["P"] = P[:, :n_aug]
                r["pmax"] = pmax[:1].clone()
                dP32 = torch.zeros(n, d.ldp, device=DEV)
                dP32[:, :n_aug] = dP_val
                dW = torch.full((n_aug, Fin), float("nan"), device=DEV)
                check(cuda_lib.spotv2_proj_bwd_weight(C.byref(da), ptr(x), None, None, None, ptr(dP32), None, None, None, ptr(dW),
                                                      ptr(ws), ws.numel(), st()), "proj_bwd_weight")
                dX = torch.full((n, Fin), float("nan"), device=DEV)
                check(cuda_lib.spotv2_proj_bwd_input(C.byref(da), ptr(dP32), None, None, None, ptr(W_aug), ptr(dX), ptr(ws),
                                                     ws.numel(), st()), "proj_bwd_input")
            else:
                x16, xblk = x_pair(cuda_lib, x)
                assert (x16[1] == 0).all()                                            # exact operands: the lo plane is zero
                ldp16 = cuda_lib.spotv2_gat_ld16(n_aug)
                P16 = torch.full((2, n, ldp16), float("nan"), device=DEV, dtype=torch.float16)
                pblk, sd = torch.zeros(8, device=DEV), torch.full((n, 2 * H), float("nan"), device=DEV)
                check(cuda_lib.spotv2_proj_fwd_pair(C.byref(da), ptr(x16[0]), ptr(x16[1]), ptr(xblk), ptr(W_aug), ptr(P16[0]),
                                                    ptr(P16[1]) if algo != 3 else None, ptr(pblk), ptr(sd), ptr(ws), ws.numel(),
                                                    st()), "proj_fwd_pair")
                r["P_hi"], r["sd"], r["pblk"] = P16[0, :, :n_aug], sd, pblk
                dP16 = torch.zeros(2, n, ldp16, device=DEV, dtype=torch.float16)
                dP16[0, :, :n_aug] = dP_int.half()
                dblk = scale_block(1.0, 1.0, 2.0 ** -20, 2.0 ** -23)
                dW = torch.full((n_aug, Fin), float("nan"), device=DEV)
                check(cuda_lib.spotv2_proj_bwd_weight(C.byref(da), None, ptr(x16[0]), ptr(x16[1]), ptr(xblk), None, ptr(dP16[0]),
                                                      ptr(dP16[1]) if algo != 3 else None, ptr(dblk), ptr(dW), ptr(ws), ws.numel(),
                                                      st()), "proj_bwd_weight")
                dX = torch.full((n, Fin), float("nan"), device=DEV)
                check(cuda_lib.spotv2_proj_bwd_input(C.byref(da), None, ptr(dP16[0]), ptr(dP16[1]) if algo != 3 else None, ptr(dblk),
                                                     ptr(W_aug), ptr(dX), ptr(ws), ws.numel(), st()), "proj_bwd_input")
            torch.cuda.synchronize()
            r["dW"], r["dX"] = dW, dX
            outs[algo] = r
        h = outs[3]
        if pf == 0:
            assert torch.equal(h["P"], P64.float()), ("P", relerr(h["P"], P64))
            assert h["pmax"].view(torch.int32).item() == h["P"][:, :HC].abs().max().reshape(1).view(torch.int32).item()
        else:
            pblk = h["pblk"]
            s0, s1 = pblk[4].item(), pblk[5].item()
            assert s0 == 2.0 ** round(math.log2(s0)) and s1 == 2.0 ** round(math.log2(s1)) and pblk[2].item() * s0 == 1.0
            want = torch.cat([(P64[:, :HC] * s0).float().half(), (P64[:, HC:] * s1).float().half()], 1)
            assert torch.equal(h["P_hi"], want), ("P_hi", relerr(h["P_hi"].double(), want.double()))
            assert torch.equal(h["sd"], P64[:, HC:].float())                         # the s|d logit terms in fp32, exact
            assert (h["P_hi"][:, :HC].reshape(n, H, Cp)[:, :, C_:] == 0).all()       # pad columns
            bound = pblk[:2].double()
            assert P64[:, :HC].abs().max() <= bound[0] and P64[:, HC:].abs().max() <= bound[1]
        assert torch.equal(h["dW"], dW64.float()), ("dW", relerr(h["dW"], dW64))
        assert torch.equal(h["dX"], dX64.float()), ("dX", relerr(h["dX"], dX64))
        for k in h:                                                                   # the 3-product class: same bits
            if k not in ("pblk",):
                assert torch.equal(outs[0][k], h[k]), (k, "3-product class differs")
        assert torch.equal(outs[0]["pblk"], h["pblk"]) if pf == 1 else True
    print(f"{shape}: split-K of the weight gradient, half class (Python rule) / 3-product class: "
          f"p_format 0 {report[0][0]} / {report[0][1]}, p_format 1 {report[1][0]} / {report[1][1]}")
    if (B, Fin) == (4096, 1260) and sms == 148:
        assert report[0] == (19, 18)                          # config C layer 0: the two rules differ


def test_single_product_gemm_error_bound_on_gaussian_operands(cuda_lib):
    """Gaussian operands: |C - C64| <= (2^-10 + 2^-21) (|A| |B|^T)_ij + K 2^-24 (|A| |B|^T)_ij elementwise (both operands
    rounded to 11 bits, fp32 accumulation), and the bound is not vacuous: the largest error / bound ratio is reported."""
    B, N, Fin, H, C_ = 40, 30, 1260, 8, 256
    d = gemm_desc(cuda_lib, B, N, Fin, H, C_, 3, 0)
    n, HC, n_aug = B * N, H * C_, H * C_ + 2 * H
    g = torch.Generator(device=DEV).manual_seed(3)
    x = torch.randn(n, Fin, device=DEV, generator=g)
    W_aug = torch.randn(n_aug, Fin, device=DEV, generator=g) * 0.05
    W_aug[HC:] *= 30.0
    ws = workspace(cuda_lib, d)
    P = torch.zeros(n, d.ldp, device=DEV)
    check(cuda_lib.spotv2_proj_fwd(C.byref(d), ptr(x), None, None, None, ptr(W_aug), ptr(P), None, ptr(ws), ws.numel(), st()),
          "proj_fwd")
    torch.cuda.synchronize()
    ref = x.double() @ W_aug.double().t()
    mag = x.double().abs() @ W_aug.double().abs().t()
    bound = (2.0 ** -10 + 2.0 ** -21 + Fin * 2.0 ** -24) * mag + 2.0 ** -60
    ratio = ((P[:, :n_aug].double() - ref).abs() / bound).max().item()
    print(f"Gaussian operands: max |C - C64| / bound = {ratio:.3f}")
    assert ratio <= 1.0
    assert ratio > 0.02                          # the bound is tight enough to see the 11-bit operand rounding


# ==================================================================== B. single-plane attention stages
def dense_logits(s, d_, T, v):
    """z[b, i, j, h] = s_j + d_i + <e_ij, v_h>, the self loop carrying the mean of the real edges' terms (fp64)."""
    B, N, H = s.shape
    if T is not None:
        gt = torch.einsum("bijf,hf->bijh", T, v)
        eye = torch.eye(N, dtype=torch.bool, device=s.device).view(1, N, N, 1)
        gt = gt.masked_fill(eye, 0.0)
        gt = gt + torch.diag_embed((gt.sum(2) / max(N - 1, 1)).permute(0, 2, 1)).permute(0, 2, 3, 1)
    else:
        gt = s.new_zeros(B, N, N, H)
    return s.unsqueeze(1) + d_.unsqueeze(2) + gt


def dense_attention(P, s, d_, T, v, bias, dout, H, concat, slope, mask=None, keep_scale=1.0):
    """fp64 forward and backward of the attention stage from a GIVEN projection: P [B, N, H, C], s / d [B, N, H], T the
    target-major edge tile [B, N, N, Fe] or None, v [H, Fe]; mask [B, i, j, H] (True = kept) replays attention dropout."""
    B, N, _, C_ = P.shape
    z = dense_logits(s, d_, T, v)
    alpha = torch.softmax(torch.where(z > 0, z, z * slope), dim=2)                  # [b, i, j, h]
    ad = alpha if mask is None else alpha * mask * keep_scale
    O = torch.einsum("bijh,bjhc->bihc", ad, P)
    out = O.reshape(B * N, H * C_) if concat else O.mean(2).reshape(B * N, C_)
    if bias is not None:
        out = out + bias
    dO = dout.view(B, N, H, C_) if concat else (dout.view(B, N, 1, C_) / H).expand(B, N, H, C_)
    dad = torch.einsum("bihc,bjhc->bijh", dO, P)
    dal = dad if mask is None else dad * mask * keep_scale
    dl = alpha * (dal - (alpha * dal).sum(2, keepdim=True))
    dz = dl * torch.where(z > 0, torch.ones_like(z), torch.full_like(z, slope))
    res = dict(alpha=ad, out=out, dP=torch.einsum("bijh,bihc->bjhc", ad, dO), dz=dz, ds=dz.sum(1), dd=dz.sum(2), dbias=dout.sum(0),
               dO=dO, aP=torch.einsum("bijh,bjhc->bihc", ad, P.abs()), adO=torch.einsum("bijh,bihc->bjhc", ad, dO.abs()))
    if T is not None:
        diag = torch.diagonal(dz, dim1=1, dim2=2).permute(0, 2, 1)
        eye = torch.eye(N, dtype=torch.bool, device=P.device).view(1, N, N, 1)
        dzp = (dz + diag.unsqueeze(2) / max(N - 1, 1)).masked_fill(eye, 0.0)
        res.update(dzp=dzp, dv=torch.einsum("bijh,bijf->hf", dzp, T))
    return res


ATTN_GEOMS = [
    # B, N, Fe, H, C, concat, dropout p, peaked
    (6, 30, 126, 6, 20, False, 0.0, False),      # C = 20 -> Cp = 24: odd heads take the shifted dP store
    (4, 30, 126, 6, 500, False, 0.0, False),     # C = 500 -> Cp = 504 (default geometry)
    (5, 13, 5, 7, 20, False, 0.0, False),        # H = 7, N = 13
    (7, 2, 4, 8, 8, True, 0.0, False),           # N = 2, concat
    (300, 31, 10, 8, 32, True, 0.0, False),      # several graphs per CTA, N = 31, concat H = 8
    (301, 32, 12, 7, 24, True, 0.0, False),      # N = 32, odd heads in concat
    (5, 30, 0, 4, 36, False, 0.0, False),        # no edge features
    (3, 30, 384, 2, 16, False, 0.0, False),      # Fe = 384, the pair-format limit
    (3, 30, 126, 2, 1024, False, 0.0, False),    # C = 1024
    (6, 30, 126, 6, 20, False, 0.3, False),      # attention dropout
    (6, 30, 126, 6, 20, False, 0.9, True),       # dropout at 0.9 on peaked rows
]


@pytest.mark.parametrize("geom", ATTN_GEOMS, ids=lambda g_: "B%dN%dFe%dH%dC%d%s_p%g%s" % (
    g_[:5] + ("cat" if g_[5] else "mean", g_[6], "_peaked" if g_[7] else "")))
def test_single_plane_attention_against_dense_fp64(cuda_lib, geom):
    B, N, Fe, H, C_, concat, pdrop, peaked = geom
    n = B * N
    R = N * (N - 1)
    d = GatDesc(B, N, 16, Fe, H, C_, R, int(concat), 0.2, cuda_lib.spotv2_gat_ldp(H, C_), 3, 0, pdrop, 0, 0x1234567, 0x89ab, 1)
    assert cuda_lib.spotv2_gat_pair_format_supported(C.byref(d)) == 1
    Cp, n_aug = cuda_lib.spotv2_gat_head_pitch(C.byref(d)), cuda_lib.spotv2_gat_n_aug(C.byref(d))
    HCp = H * Cp
    ldp16 = cuda_lib.spotv2_gat_ld16(n_aug)
    g = torch.Generator(device=DEV).manual_seed(n + C_)
    # the hi plane: integers in [-1024, 1024] at inverse scale 2^-10 (|P| <= 1), zero pads; the planes' s|d columns copy sd
    P_int = ints((n, H, Cp), g, -1024, 1024)
    P_int[:, :, C_:] = 0.0
    sd = torch.randn(n, 2 * H, device=DEV, generator=g) * (4.0 if peaked else 1.0)
    bt = synth.random_complete_batch(B, N, 1, max(Fe, 1), seed=5)
    topo = sv.topology_from_edge_index(bt.edge_index.to(DEV), n)
    ea = (bt.edge_attr[:, :Fe] if Fe else bt.edge_attr[:, :0]).contiguous().to(DEV)
    v = (torch.randn(H, Fe, device=DEV, generator=g) * 0.3).contiguous()
    T = dense_gat.pyg_to_dense_tile(ea.double(), bt.edge_index.to(DEV), B, N) if Fe else None
    # a logit within fp32 noise of the LeakyReLU kink may fall on either side (dz jumps by the slope there): move the
    # target term d_i of such a row away from it, so that fp32 and fp64 agree on every side
    for _ in range(8):
        z = dense_logits(sd[:, :H].double().view(B, N, H), sd[:, H:].double().view(B, N, H), T, v.double())
        near = (z.abs() < 1e-4 * z.abs().max()).any(2).view(n, H)                    # [b*i, h]
        if not near.any():
            break
        sd[:, H:][near] += 3e-4 * z.abs().max().item()
    assert not near.any()
    P16 = torch.zeros(2, n, ldp16, device=DEV, dtype=torch.float16)
    P16[0, :, :HCp] = P_int.view(n, HCp).half()
    P16[0, :, HCp:n_aug] = (sd * 2.0 ** 10).half()
    pblk = scale_block(1.0, 32.0, 2.0 ** -10, 2.0 ** -10)
    P = (P_int[:, :, :C_] * 2.0 ** -10).double().view(B, N, H, C_)
    bias = torch.randn(H * C_ if concat else C_, device=DEV, generator=g)
    ldo = H * C_ if concat else C_
    dout = ints((n, ldo), g, -1024, 1024) * 2.0 ** -7                          # any power-of-two unit scale keeps it exact
    etb = C.c_size_t()
    check(cuda_lib.spotv2_gat_edge_terms_bytes(C.byref(d), C.byref(etb)), "edge_terms_bytes")
    ws = workspace(cuda_lib, d)

    def run(algo):
        da = with_algo(d, algo)
        rec = torch.zeros(max(etb.value // 4, 4), device=DEV) if Fe else None
        out = torch.full((n, ldo), float("nan"), device=DEV)
        alpha = torch.full((B, H, N, N), float("nan"), device=DEV)
        lo = P16[1] if algo != 3 else None
        check(cuda_lib.spotv2_gat_attn_fwd_pair(C.byref(da), ptr(P16[0]), ptr(lo), ptr(pblk), ptr(sd), ptr(ea) if Fe else None,
                                                ptr(topo.table) if Fe else None, ptr(v) if Fe else None, ptr(bias), ptr(out),
                                                ptr(alpha), ptr(rec), st()), "attn_fwd_pair")
        dP16 = torch.full((2, n, ldp16), float("nan"), device=DEV, dtype=torch.float16)
        dblk = torch.zeros(8, device=DEV)
        dv = torch.full((H, Fe), float("nan"), device=DEV) if Fe else None
        d_et = torch.full_like(rec, float("nan")) if Fe else None
        dbias = torch.full((ldo,), float("nan"), device=DEV)
        check(cuda_lib.spotv2_gat_attn_bwd_pair(C.byref(da), ptr(P16[0]), ptr(lo), ptr(pblk), ptr(sd), ptr(ea) if Fe else None,
                                                ptr(rec), ptr(topo.table) if Fe else None, ptr(v) if Fe else None, ptr(dout),
                                                ptr(dP16[0]), ptr(dP16[1]) if algo != 3 else None, ptr(dblk), ptr(dv), ptr(d_et),
                                                ptr(dbias), ptr(ws), ws.numel(), st()), "attn_bwd_pair")
        torch.cuda.synchronize()
        return dict(out=out, alpha=alpha, dP16=dP16, dblk=dblk, dv=dv, d_et=d_et, dbias=dbias)

    ours = run(3)
    full = run(0)                                 # the fp32 class on the same inputs (its lo plane is zero: P is exact)
    a_ours = ours["alpha"].permute(0, 3, 2, 1).double()                             # [b, i, j, h]
    mask = (a_ours != 0) if pdrop > 0 else None
    if pdrop > 0:
        assert abs(mask.double().mean().item() - (1 - pdrop)) < 0.03
        assert torch.equal(full["alpha"] != 0, ours["alpha"] != 0)                 # same key, same mask
    s64, d64 = sd[:, :H].double().view(B, N, H), sd[:, H:].double().view(B, N, H)
    r = dense_attention(P, s64, d64, T, v.double(), bias.double(), dout.double(), H, concat, 0.2, mask, 1.0 / (1.0 - pdrop))
    def stage_errors(res):
        e = {"alpha": relerr(res["alpha"].permute(0, 3, 2, 1), r["alpha"]), "dbias": relerr(res["dbias"], r["dbias"])}
        if Fe:
            e["dv"] = relerr(res["dv"], r["dv"])
            e["dz'"] = relerr(res["d_et"].view(B, H, N, 36)[..., :N], r["dzp"].permute(0, 3, 2, 1))
        return e
    errs, errs_full = stage_errors(ours), stage_errors(full)
    for k, e in errs.items():
        assert e < 1e-5, (k, e, "fp32 class:", errs_full)
    # out: the only rounding left is alpha -> fp16 in the aggregation
    aP = r["aP"].reshape(n, H * C_) if concat else r["aP"].mean(2).reshape(n, C_)
    e_out = (ours["out"].double() - r["out"]).abs()
    b_out = (2.0 ** -11 + 2.0 ** -19) * aP + 2.0 ** -22 * r["out"].abs() + 1e-7 * r["out"].abs().max()
    assert (e_out <= b_out).all(), (e_out / b_out).max().item()
    e_full = relerr(full["out"], r["out"])
    assert relerr(ours["out"], r["out"]) > 10 * e_full, "the single-plane aggregation did not run"
    # dP group 0: alpha rounding plus half an fp16 ulp at the dP scale; pad columns zero
    dblk, hi = ours["dblk"], ours["dP16"][0]
    assert torch.isfinite(hi[:, :n_aug].float()).all()
    dP0 = hi[:, :HCp].view(n, H, Cp)
    assert (dP0[:, :, C_:] == 0).all()
    got0 = dP0[:, :, :C_].double() * dblk[2].item()
    ref0 = r["dP"].reshape(n, H, C_)
    b0 = (2.0 ** -11 + 2.0 ** -19) * r["adO"].reshape(n, H, C_) + half_ulp_f16(dP0[:, :, :C_]) * dblk[2].item() + 1e-6 * ref0.abs().max()
    assert ((got0 - ref0).abs() <= b0).all(), ((got0 - ref0).abs() / b0).max().item()
    # group 1 (ds | dd): half an ulp at its own scale
    got1 = hi[:, HCp:n_aug].double() * dblk[3].item()
    ref1 = torch.cat([r["ds"].reshape(n, H), r["dd"].reshape(n, H)], 1)
    b1 = half_ulp_f16(hi[:, HCp:n_aug]) * dblk[3].item() + 1e-5 * ref1.abs().max()
    assert ((got1 - ref1).abs() <= b1).all(), ((got1 - ref1).abs() / b1).max().item()
    print(f"{geom}: {({k: f'{e:.1e}' for k, e in errs.items()})}, out {relerr(ours['out'], r['out']):.1e} "
          f"(fp32 class {e_full:.1e}), dP {relerr(got0, ref0):.1e}, ds|dd {relerr(got1, ref1):.1e}")


# ==================================================================== C. GATConv / GATModel in half mode
def emulate_half_layer(x, T, W, a_s, a_d, W_e, a_e, bias, dout, H, C_, concat, slope, pf, alpha_rounded_from=None):
    """fp64 emulation of one half-class layer step.  Rounds to fp16 where the kernels round: x and W_aug at their group
    scales (the single GEMM reads hi planes only), P at its scale and alpha (p_format 1 only), dP and ds|dd at their scales
    (both formats).  alpha_rounded_from: the kernels' own fp32 alpha [b, i, j, h], whose fp16 rounding is emulated (so that
    an fp32-vs-fp64 near-tie cannot flip an alpha by one ulp)."""
    B, N = T.shape[0], T.shape[1]
    HC = H * C_
    x, W, a_s, a_d, bias, dout = [t.double() for t in (x, W, a_s, a_d, bias, dout)]
    W_aug, v = dense_gat.fold_params(W, a_s, a_d, W_e.double() if W_e is not None else None,
                                     a_e.double() if a_e is not None else None, H, C_)
    xq = f16_at(x, pow2_scale(x.abs().max().item()))
    Wq = torch.cat([f16_at(W_aug[:HC], pow2_scale(W_aug[:HC].abs().max().item())),
                    f16_at(W_aug[HC:], pow2_scale(W_aug[HC:].abs().max().item()))])
    P_aug = xq @ Wq.t()
    P = P_aug[:, :HC].reshape(B, N, H, C_)
    if pf == 1:
        bound = x.abs().max().item() * W_aug[:HC].abs().sum(1).max().item()
        P = f16_at(P, pow2_scale(bound))
    s, d_ = P_aug[:, HC:HC + H].reshape(B, N, H), P_aug[:, HC + H:].reshape(B, N, H)
    if v is not None:
        gt = torch.einsum("bijf,hf->bijh", T, v)
        eye = torch.eye(N, dtype=torch.bool, device=x.device).view(1, N, N, 1)
        gt = gt.masked_fill(eye, 0.0)
        gt = gt + torch.diag_embed((gt.sum(2) / max(N - 1, 1)).permute(0, 2, 1)).permute(0, 2, 3, 1)
    else:
        gt = x.new_zeros(B, N, N, H)
    z = s.unsqueeze(1) + d_.unsqueeze(2) + gt
    alpha = torch.softmax(torch.where(z > 0, z, z * slope), dim=2)
    aq = alpha
    if pf == 1:
        aq = f16_at(alpha if alpha_rounded_from is None else alpha_rounded_from.double(), 2.0 ** 14)
    O = torch.einsum("bijh,bjhc->bihc", aq, P)
    out = (O.reshape(B * N, HC) if concat else O.mean(2).reshape(B * N, C_)) + bias
    dO = dout.view(B, N, H, C_) if concat else (dout.view(B, N, 1, C_) / H).expand(B, N, H, C_)
    da = torch.einsum("bihc,bjhc->bijh", dO, P)
    dl = alpha * (da - (alpha * da).sum(2, keepdim=True))
    dz = dl * torch.where(z > 0, torch.ones_like(z), torch.full_like(z, slope))
    dP = torch.einsum("bijh,bihc->bjhc", aq, dO).reshape(B * N, HC)
    dsd = torch.cat([dz.sum(1).reshape(B * N, H), dz.sum(2).reshape(B * N, H)], 1)
    s0 = pow2_scale(dout.abs().max().item() * N * (1.0 if concat else 1.0 / H))
    s1 = pow2_scale(dsd.abs().max().item())
    dPq = torch.cat([f16_at(dP, s0), f16_at(dsd, s1)], 1)
    dW_aug = dPq.t() @ xq
    # dX: W_aug's rows pre-multiplied by dP's inverse group scales, then split with one scale of its own
    g_inv = torch.cat([torch.full((HC,), 1.0 / s0), torch.full((2 * H,), 1.0 / s1)]).to(x.device, torch.float64).view(-1, 1)
    Wd = W_aug * g_inv
    Wd = f16_at(Wd, pow2_scale(Wd.abs().max().item())) / g_inv
    res = dict(out=out, alpha=alpha, g_x=dPq @ Wd, g_bias=dout.sum(0))
    dv = None
    if v is not None:
        diag = torch.diagonal(dz, dim1=1, dim2=2).permute(0, 2, 1)
        eye = torch.eye(N, dtype=torch.bool, device=x.device).view(1, N, N, 1)
        dzp = (dz + diag.unsqueeze(2) / max(N - 1, 1)).masked_fill(eye, 0.0)
        dv = torch.einsum("bijh,bijf->hf", dzp, T)
        res["dzp_tile"] = torch.einsum("bijh,hf->bijf", dzp, v)                     # d edge tile [b, i, j, Fe]
    u = dense_gat.unfold_grads(dW_aug, dv, W, a_s, a_d, W_e.double() if W_e is not None else None,
                               a_e.double() if a_e is not None else None, H, C_)
    res.update({"g_lin_src.weight": u["lin_weight"], "g_att_src": u["att_src"], "g_att_dst": u["att_dst"]})
    if dv is not None:
        res.update({"g_lin_edge.weight": u["lin_edge_weight"], "g_att_edge": u["att_edge"]})
    return res


def exact_layer(Fin, C_, H, concat, Fe, seed):
    """GATConv with fp16-exact parameters: lin_src / lin_edge integers in [-8, 8] times a power of two; att_src / att_dst
    with two entries of +-1/2 per head, so the folded rows u = W_h^T a_h stay small integers (fp16-exact as well)."""
    g = torch.Generator().manual_seed(seed)
    layer = sv.GATConv(Fin, C_, heads=H, concat=concat, edge_dim=Fe)
    wu = 2.0 ** -round(math.log2(8 * math.sqrt(Fin)))
    with torch.no_grad():
        layer.lin_src.weight.copy_(ints((H * C_, Fin), g, device="cpu") * wu)
        for a in (layer.att_src, layer.att_dst):
            a.zero_()
            for h in range(H):
                idx = torch.randperm(C_, generator=g)[:2]
                a[0, h, idx] = (torch.randint(0, 2, (len(idx),), generator=g).float() * 2 - 1) * 0.5
        layer.lin_edge.weight.copy_(ints((H * C_, Fe), g, device="cpu") * 2.0 ** -4)
        layer.att_edge.copy_(ints((1, H, C_), g, device="cpu") * 2.0 ** -round(math.log2(2.2 * math.sqrt(C_ * Fe))))   # |<e, v>| ~ 1
        layer.bias.copy_(ints(layer.bias.shape, g, device="cpu") * 2.0 ** -4)
    layer.precision = "half"
    return layer.to(DEV)


def record_descs(monkeypatch):
    """Every descriptor the layers build (gat_conv._desc), to tell which p_format a call took."""
    from spotv2net_b200 import gat_conv
    seen, orig = [], gat_conv._desc

    def rec(*a, **k):
        d = orig(*a, **k)
        seen.append(d)
        return d
    monkeypatch.setattr(gat_conv, "_desc", rec)
    return seen


def alpha_pyg_to_tile(alpha, B, N, H, edge_index):
    R = N * (N - 1)
    local = edge_index[:, :R]
    tile = alpha.new_zeros(B, N, N, H)
    tile[:, local[1], local[0], :] = alpha[:B * R].view(B, R, H)
    loops = alpha[B * R:].view(B, N, H)
    idx = torch.arange(N, device=alpha.device)
    tile[:, idx, idx, :] = loops
    return tile


# bars from the first B200 run (each case prints its errors against the emulation): out at most 5e-7, gradients at most
# 7e-5 (att_dst of the standardized model's second layer; dX 5e-5).  The residue is fp32-vs-fp64 near-ties before a
# rounding to fp16 and fp32 accumulation order.
HALF_BARS = {"out": 2e-6, "default": 2e-4}

LAYER_CASES = [
    # B, N, F, Fe, H, C, concat, expected p_format, serial backward, edge_attr grad
    (4, 30, 64, 126, 8, 256, True, 1, False, False),     # config C layer 0 geometry (small F)
    (4, 30, 1260, 126, 6, 500, False, 1, False, True),   # default geometry, edge_attr.requires_grad
    (5, 13, 40, 5, 7, 20, False, 1, False, False),
    (3, 40, 24, 9, 4, 12, False, 0, False, False),       # N = 40: the large-graph path
    (3, 30, 40, 390, 2, 16, False, 0, False, True),      # Fe = 390 > 384, edge_attr.requires_grad
    (3, 30, 40, 126, 3, 12, True, 0, False, False),      # concat with C % 8 != 0
    (3, 30, 64, 126, 6, 20, False, 0, True, False),      # the phase-serial backward
]


@pytest.mark.parametrize("case", LAYER_CASES, ids=lambda c: "B%dN%dF%dFe%dH%dC%d%s_pf%d%s%s" % (
    c[:6] + ("cat" if c[6] else "mean", c[7], "_serial" if c[8] else "", "_dea" if c[9] else "")))
def test_half_precision_layer_against_fp64_emulation(cuda_lib, case, monkeypatch):
    from spotv2net_b200 import gat_conv
    B, N, Fin, Fe, H, C_, concat, pf_want, serial, want_dea = case
    if serial:
        monkeypatch.setattr(gat_conv, "ATTN_BWD_ALGO", 1)
    layer = exact_layer(Fin, C_, H, concat, Fe, seed=B * N + Fin)
    ei, topo = sv.batched_topology(B, N, DEV)
    descs = record_descs(monkeypatch)
    g = torch.Generator(device=DEV).manual_seed(11)
    x = (ints((B * N, Fin), g) * 2.0 ** -3).requires_grad_()
    ea = (ints((B * N * (N - 1), Fe), g) * 2.0 ** -2).requires_grad_(want_dea)
    dout = ints((B * N, H * C_ if concat else C_), g, -1024, 1024) * 2.0 ** -7
    out, (_, a_pyg) = layer(x, ei, ea, return_attention_weights=True, topology=topo)
    out.backward(dout)
    torch.cuda.synchronize()
    assert len(descs) == 1 and descs[0].gemm_algo == 3
    d = descs[0]
    assert d.p_format == pf_want, f"expected p_format {pf_want}, the layer took {d.p_format}"
    mine = {"out": out.detach(), "g_x": x.grad}
    mine.update({"g_" + k: p.grad for k, p in layer.named_parameters()})
    T = dense_gat.pyg_to_dense_tile(ea.detach().double(), ei, B, N)
    a_tile = alpha_pyg_to_tile(a_pyg.detach(), B, N, H, ei)
    em = emulate_half_layer(x.detach(), T, layer.lin_src.weight.detach(), layer.att_src.detach(), layer.att_dst.detach(),
                            layer.lin_edge.weight.detach(), layer.att_edge.detach(), layer.bias.detach(), dout, H, C_, concat,
                            0.2, d.p_format, a_tile)
    assert relerr(a_tile, em["alpha"]) < 1e-5
    if want_dea:
        R = N * (N - 1)
        local = ei[:, :R]
        em["g_edge_attr"] = em.pop("dzp_tile")[:, local[1], local[0], :].reshape(B * R, Fe)
        mine["g_edge_attr"] = ea.grad
    errs = {k: relerr(mine[k], em[k]) for k in mine if k in em}
    assert set(errs) >= {"out", "g_x", "g_lin_src.weight", "g_att_src", "g_att_dst", "g_bias", "g_lin_edge.weight", "g_att_edge"}
    print(f"{case}: p_format {d.p_format}, max-norm error against the emulation",
          {k: f"{e:.1e}" for k, e in errs.items()})
    bad = {k: e for k, e in errs.items() if e > HALF_BARS.get(k, HALF_BARS["default"])}
    assert not bad, bad


def test_half_precision_standardized_model_against_fp64_emulation(cuda_lib, monkeypatch):
    """GATModel(standardize=True) in training mode keeps p_format 0 (the edge mean shifts the d columns of an fp32 P_aug);
    x arrives normalised, so its fp16 rounding in the single GEMM is emulated as well.  Each layer is checked at its own
    inputs and upstream gradient (teacher forcing), as the config C model test does."""
    B, N, L = 6, 30, 4
    kw = dict(num_node_features=N * L, num_edge_features=3 * L, num_heads=4, output_node_channels=1,
              dim_hidden_layers=[16, 8], concat_heads=False, standardize=True)
    torch.manual_seed(3)
    model = sv.GATModel(**kw)
    for k, layer in enumerate(model.gat_layers):
        ex = exact_layer(layer.in_channels, layer.out_channels, layer.heads, layer.concat, layer.edge_dim, seed=40 + k)
        layer.load_state_dict(ex.state_dict())
    model.to(DEV).train().set_precision("half")
    bt = synth.random_complete_batch(B, N, N * L, 3 * L, seed=8).to(DEV)
    bt.y = torch.randn(B * N, device=DEV)
    seen = []
    descs = record_descs(monkeypatch)

    def hook(mod, args, kwargs, out):
        out.retain_grad()
        if args[0].requires_grad:
            args[0].retain_grad()
        seen.append((mod, args[0], kwargs, out))

    hs = [layer.register_forward_hook(hook, with_kwargs=True) for layer in model.gat_layers]
    try:
        torch.nn.functional.mse_loss(model(bt), bt.y).backward()
    finally:
        for h_ in hs:
            h_.remove()
    torch.cuda.synchronize()
    assert len(descs) == len(seen) == 2
    for k, (layer, x_in, kwargs, out) in enumerate(seen):
        assert descs[k].gemm_algo == 3 and descs[k].p_format == 0
        e_hat = (bt.edge_attr.double() - kwargs["edge_mean"].double()) * kwargs["edge_scale"].double()
        T = dense_gat.pyg_to_dense_tile(e_hat, bt.edge_index, B, N)
        em = emulate_half_layer(x_in.detach(), T, layer.lin_src.weight.detach(), layer.att_src.detach(), layer.att_dst.detach(),
                                layer.lin_edge.weight.detach(), layer.att_edge.detach(), layer.bias.detach(), out.grad,
                                layer.heads, layer.out_channels, layer.concat, 0.2, 0)
        mine = {"out": out.detach()}
        mine.update({"g_" + n_: p.grad for n_, p in layer.named_parameters()})
        if x_in.grad is not None:
            mine["g_x"] = x_in.grad
        errs = {t: relerr(mine[t], em[t]) for t in mine if t in em}
        print(f"standardized model layer {k}: max-norm error against the emulation", {t: f"{e:.1e}" for t, e in errs.items()})
        bad = {t: e for t, e in errs.items() if e > HALF_BARS.get(t, HALF_BARS["default"])}
        assert not bad, (k, bad)
