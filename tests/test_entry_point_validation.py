"""Argument checks of the four attention entry points, on the CPU.

Every case below breaks one rule (or, for the order cases, two) and must be rejected with its status and message
before anything is launched, so fake device pointers serve: aligned, distinct and never dereferenced.
"""
import ctypes as C

import pytest

from spotv2net_b200 import _lib

INVALID, UNSUPPORTED = 1, 2

# argument order of each entry point (include/spotv2_gat.h), descriptor first
ARGS = {
    "attn_fwd": ["P_aug", "edge_rows", "table", "v", "bias", "out", "alpha", "edge_terms", "ws", "ws_bytes", "stream"],
    "attn_fwd_pair": ["P_hi", "P_lo", "p_scale", "sd", "edge_rows", "table", "v", "bias", "out", "alpha", "edge_terms",
                      "stream"],
    "attn_bwd": ["P_aug", "p_amax", "edge_rows", "edge_terms", "table", "v", "dout", "dP_aug", "dP_hi", "dP_lo",
                 "dp_scale", "dv", "d_edge_terms", "dbias", "ws", "ws_bytes", "stream"],
    "attn_bwd_pair": ["P_hi", "P_lo", "p_scale", "sd", "edge_rows", "edge_terms", "table", "v", "dout", "dP_hi",
                      "dP_lo", "dp_scale", "dv", "d_edge_terms", "dbias", "ws", "ws_bytes", "stream"],
}
# optional arguments left null unless a case sets them (the fp32 backward: dP leaves as fp32 dP_aug by default)
NULL_BY_DEFAULT = {"bias", "alpha", "edge_terms", "ws", "stream", "p_amax", "dP_hi", "dP_lo", "dp_scale", "dv",
                   "d_edge_terms", "dbias"}
PAIR = {"attn_fwd_pair", "attn_bwd_pair"}
BACKWARD = {"attn_bwd", "attn_bwd_pair"}


def fake(i):
    return 0x7f0000000000 + 0x100000 * (i + 1)       # 1 MB apart: 16-byte aligned


def desc(entry, **kw):
    f = dict(B=4, N=30, F=60, Fe=126, H=6, C=500, R=870, concat=0, negative_slope=0.2, gemm_algo=0, attn_bwd_algo=0,
             dropout_p=0.0, edge_mode=0, p_format=1 if entry in PAIR else 0)
    f.update(kw)
    f["ldp"] = _lib.load().spotv2_gat_ldp(f["H"], f["C"])
    return _lib.GatDesc(**f)


def call(entry, d, **ptrs):
    lib = _lib.load()
    args = []
    for i, name in enumerate(ARGS[entry]):
        if name == "ws_bytes":
            args.append(0)
        elif name in ptrs:
            args.append(ptrs[name])
        else:
            args.append(None if name in NULL_BY_DEFAULT else fake(i))
    rc = getattr(lib, "spotv2_gat_" + entry)(C.byref(d) if d is not None else None, *args)
    return rc, lib.spotv2_last_error().decode()


def misaligned(entry, name):
    return fake(ARGS[entry].index(name)) + 4


def shared_cases(entry):
    """The rules all four entry points share: (id, descriptor fields, pointers, status, message)."""
    bwd = entry in BACKWARD
    terms = dict(edge_terms=fake(40), d_edge_terms=fake(41)) if bwd else dict(edge_terms=fake(40))
    mode1 = "edge_mode 1 needs edge_terms and a 16-byte aligned d_edge_terms buffer" if bwd else \
        "edge_mode 1 needs edge_terms (spotv2_edge_terms_from_windows)"
    cases = [
        ("no_edge_rows", {}, dict(edge_rows=None), INVALID, f"{entry}: edge_rows, table and v are required when Fe > 0"),
        ("no_table", {}, dict(table=None), INVALID, f"{entry}: edge_rows, table and v are required when Fe > 0"),
        ("no_v", {}, dict(v=None), INVALID, f"{entry}: edge_rows, table and v are required when Fe > 0"),
        ("mode1_no_terms", dict(edge_mode=1), dict(terms, edge_terms=None), INVALID, f"{entry}: {mode1}"),
        ("H_9", dict(H=9), {}, UNSUPPORTED, "H=9 > 8"),
        ("Fe_513", dict(Fe=513), {}, UNSUPPORTED, "Fe=513 > 512"),
        ("terms_misaligned", {}, dict(edge_terms=fake(40) + 4), INVALID, f"{entry}: edge_terms must be 16-byte aligned"),
        # order: the edge inputs are checked before the size limits, the limits before the edge terms' alignment
        ("order_edges_then_H", dict(H=9), dict(edge_rows=None), INVALID,
         f"{entry}: edge_rows, table and v are required when Fe > 0"),
        ("order_Fe_then_terms", dict(Fe=513), dict(edge_terms=fake(40) + 4), UNSUPPORTED, "Fe=513 > 512"),
    ]
    if bwd:
        cases += [
            ("mode1_no_dterms", dict(edge_mode=1), dict(terms, d_edge_terms=None), INVALID, f"{entry}: {mode1}"),
            ("mode1_dterms_misaligned", dict(edge_mode=1), dict(terms, d_edge_terms=fake(41) + 4), INVALID,
             f"{entry}: {mode1}"),
            ("dterms_misaligned", {}, dict(d_edge_terms=fake(41) + 4), INVALID,
             f"{entry}: d_edge_terms must be 16-byte aligned"),
        ]
    return cases


def own_cases(entry):
    """Each entry point's own pointer, format and alignment rules."""
    m = lambda name: misaligned(entry, name)      # noqa: E731
    if entry == "attn_fwd":
        return [
            ("no_P_aug", {}, dict(P_aug=None), INVALID, "attn_fwd: P_aug and out must be non-null"),
            ("no_out", {}, dict(out=None), INVALID, "attn_fwd: P_aug and out must be non-null"),
            ("P_aug_misaligned", {}, dict(P_aug=m("P_aug")), INVALID, "attn_fwd: P_aug/out must be 16-byte aligned"),
            ("out_misaligned", {}, dict(out=m("out")), INVALID, "attn_fwd: P_aug/out must be 16-byte aligned"),
            ("order_pointers_then_edges", {}, dict(out=None, edge_rows=None), INVALID,
             "attn_fwd: P_aug and out must be non-null"),
            ("order_edges_then_alignment", {}, dict(out=m("out"), v=None), INVALID,
             "attn_fwd: edge_rows, table and v are required when Fe > 0"),
        ]
    if entry == "attn_fwd_pair":
        msg_null = "attn_fwd_pair: P_hi, p_scale, sd and out must be non-null"
        msg_align = "attn_fwd_pair: P planes / out must be 16-byte aligned"
        return [
            ("p_format_0", dict(p_format=0), {}, INVALID, "attn_fwd_pair: the descriptor must say p_format 1"),
            ("no_P_hi", {}, dict(P_hi=None), INVALID, msg_null),
            ("no_p_scale", {}, dict(p_scale=None), INVALID, msg_null),
            ("no_sd", {}, dict(sd=None), INVALID, msg_null),
            ("no_out", {}, dict(out=None), INVALID, msg_null),
            ("no_P_lo", {}, dict(P_lo=None), INVALID, "attn_fwd_pair: the lo plane may be omitted with gemm_algo 3 only"),
            ("P_hi_misaligned", {}, dict(P_hi=m("P_hi")), INVALID, msg_align),
            ("P_lo_misaligned", {}, dict(P_lo=m("P_lo")), INVALID, msg_align),
            ("out_misaligned", {}, dict(out=m("out")), INVALID, msg_align),
            ("order_format_then_pointers", dict(p_format=0), dict(P_hi=None), INVALID,
             "attn_fwd_pair: the descriptor must say p_format 1"),
            ("order_edges_then_alignment", {}, dict(out=m("out"), table=None), INVALID,
             "attn_fwd_pair: edge_rows, table and v are required when Fe > 0"),
        ]
    if entry == "attn_bwd":
        msg_align = "attn_bwd: P_aug/dout/dP must be 16-byte aligned"
        pair = dict(dP_aug=None, dP_hi=fake(50), dP_lo=fake(51), dp_scale=fake(52))
        return [
            ("no_P_aug", {}, dict(P_aug=None), INVALID, "attn_bwd: P_aug and dout must be non-null"),
            ("no_dout", {}, dict(dout=None), INVALID, "attn_bwd: P_aug and dout must be non-null"),
            ("no_dP", {}, dict(dP_aug=None), INVALID, "attn_bwd: give dP_aug (fp32) or dP_hi/dP_lo/dp_scale (fp16 pairs)"),
            ("dP_hi_without_lo", {}, dict(pair, dP_lo=None), INVALID, "attn_bwd: dP_hi needs dP_lo and dp_scale"),
            ("dP_hi_without_scale", {}, dict(pair, dp_scale=None), INVALID, "attn_bwd: dP_hi needs dP_lo and dp_scale"),
            ("mode1_phase_serial", dict(edge_mode=1, attn_bwd_algo=1), dict(edge_terms=fake(40), d_edge_terms=fake(41)),
             UNSUPPORTED, "attn_bwd: for N <= 32, edge_mode 1 runs on the pipelined kernel only"),
            ("P_aug_misaligned", {}, dict(P_aug=m("P_aug")), INVALID, msg_align),
            ("dout_misaligned", {}, dict(dout=m("dout")), INVALID, msg_align),
            ("dP_aug_misaligned", {}, dict(dP_aug=m("dP_aug")), INVALID, msg_align),
            ("dP_hi_misaligned", {}, dict(pair, dP_hi=fake(50) + 4), INVALID, msg_align),
            ("dP_lo_misaligned", {}, dict(pair, dP_lo=fake(51) + 4), INVALID, msg_align),
            ("order_phase_serial_then_alignment", dict(edge_mode=1, attn_bwd_algo=1),
             dict(edge_terms=fake(40), d_edge_terms=fake(41), dout=m("dout")), UNSUPPORTED,
             "attn_bwd: for N <= 32, edge_mode 1 runs on the pipelined kernel only"),
            ("order_pointers_then_edges", {}, dict(dout=None, v=None), INVALID, "attn_bwd: P_aug and dout must be non-null"),
        ]
    msg_null = "attn_bwd_pair: P_hi, p_scale, sd, dout, dP_hi and dp_scale must be non-null"
    msg_lo = "attn_bwd_pair: the lo planes may be omitted with gemm_algo 3 only"
    msg_align = "attn_bwd_pair: P / dout / dP must be 16-byte aligned"
    full = dict(dP_hi=fake(50), dP_lo=fake(51), dp_scale=fake(52))
    return [
        ("p_format_0", dict(p_format=0), full, INVALID, "attn_bwd_pair: the descriptor must say p_format 1"),
        *[(f"no_{n}", {}, dict(full, **{n: None}), INVALID, msg_null)
          for n in ("P_hi", "p_scale", "sd", "dout", "dP_hi", "dp_scale")],
        ("no_P_lo", {}, dict(full, P_lo=None), INVALID, msg_lo),
        ("no_dP_lo", {}, dict(full, dP_lo=None), INVALID, msg_lo),
        *[(f"{n}_misaligned", {}, dict(full, **{n: (full[n] + 4 if n in full else m(n))}), INVALID, msg_align)
          for n in ("P_hi", "P_lo", "dout", "dP_hi", "dP_lo")],
        ("order_lo_then_edges", {}, dict(full, P_lo=None, edge_rows=None), INVALID, msg_lo),
    ]


def with_pair_outputs(entry, ptrs):
    # the pair backward always emits dP as the pair: give it one unless the case is about it
    if entry != "attn_bwd_pair":
        return ptrs
    return {**dict(dP_hi=fake(50), dP_lo=fake(51), dp_scale=fake(52)), **ptrs}


CASES = [pytest.param(entry, *case[1:], id=f"{entry}-{case[0]}")
         for entry in ARGS for case in shared_cases(entry) + own_cases(entry)]


@pytest.mark.parametrize("entry,fields,ptrs,status,message", CASES)
def test_rejected_before_launch(entry, fields, ptrs, status, message):
    rc, err = call(entry, desc(entry, **fields), **with_pair_outputs(entry, ptrs))
    assert rc == status, err
    assert message in err


@pytest.mark.parametrize("entry", list(ARGS))
def test_null_descriptor(entry):
    rc, err = call(entry, None)
    assert rc == INVALID
    assert "descriptor is null" in err
