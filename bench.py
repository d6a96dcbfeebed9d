#!/usr/bin/env python
"""Benchmark of the SpotV2Net GAT hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (one rank per GPU under torchrun)
    python bench.py --impl reference --steps K --warmup W    # reference arm: the CPU oracle port

A step = GATConv forward + backward (fold -> projection GEMM -> fused attention -> fused attention
backward with recompute -> weight-gradient GEMM -> unfold [-> NCCL all-reduce of the flat gradient
arena when N > 1]) over one batch of 4096 synthetic 30-node complete graphs of the standardized H5
shape, default config/GNN_param.yaml hyper-parameters (BASELINE.json configs[1]), fp32.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "SpotV2Net GAT fwd+bwd graphs/sec (30-node, batch 4096)"
UNIT = "graphs/s"
CFG = dict(N=30, L=42, H=6, C=500, slope=0.2, concat=False)
# The bench line is BASELINE configs[1] ("A").  --config D times the 500-node universe (configs[3]) through the
# same code for DESIGN.md; it is a parity-test case, not the headline.
METRIC_BY_CONFIG = {
    "A": METRIC,
    "C": "SpotV2Net wide multi-head variant (8 heads, hidden [256,256], two GAT layers) fwd+bwd graphs/sec (30-node, batch 4096)",
    "D": "SpotV2Net GAT fwd+bwd graphs/sec (500-node universe, batch 32)",
}
CONFIGS = {"C": dict(N=30, batch=4096, name="BASELINE configs[2]: wide multi-head variant (8 heads, hidden [256, 256], concat: layer 0 1260 -> 8x256 "
                                            "concat, layer 1 2048 -> 256 head mean), batch 4096 snapshots per GPU"),
           "A": dict(N=30, batch=4096, name="BASELINE configs[1]: default GNN_param.yaml hyper-parameters, batch 4096 snapshots per GPU"),
           "D": dict(N=500, batch=32, name="BASELINE configs[3]: 500-node complete graph (249,500 edges per snapshot), batch 32 snapshots per GPU, "
                                           "multi-CTA-per-graph attention")}


def attn_bytes():
    """Algorithmic bytes per graph of the attention stage (SURVEY.md §8d): every operand touched once per pass.
    Default geometry: fwd 858 480 B (edge rows 438 480 + P 360 000 + out 60 000), bwd 1 218 480 B (+ dP 360 000)."""
    N, Fin, Fe, H, Cc = cfg_dims()
    edge, P, out = N * (N - 1) * Fe * 4, N * H * Cc * 4, N * Cc * 4
    return edge + P + out, edge + P + out + P


def proj_flop_per_graph():
    N, Fin, Fe, H, Cc = cfg_dims()
    return 2 * (2 * N * Fin * H * Cc)            # P = x W^T and dW = dP^T x  (2 x 226.8 MFLOP at the default geometry)


def cfg_dims():
    N, L = CFG["N"], CFG["L"]
    return N, N * L, 3 * L, CFG["H"], CFG["C"]


# --------------------------------------------------------------------------- --dump-outputs
DUMP_MAX_ELEMS = 1 << 22          # per array; the largest outputs (config A's 246 MB `out`) are sampled down to this
DUMP_MAX_BYTES = 64 << 20         # all arrays together


def sample_rows(t: torch.Tensor, seed: int = 0) -> torch.Tensor:
    """t itself, or - when it holds more than DUMP_MAX_ELEMS elements - a fixed, seeded sample of its rows, in row order."""
    if t.numel() <= DUMP_MAX_ELEMS:
        return t
    keep = max(1, DUMP_MAX_ELEMS // (t.numel() // t.shape[0]))
    idx = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(seed))[:keep].sort().values
    return t[idx.to(t.device)]


def dump_outputs(path: str, arrays: dict) -> None:
    """Writes {name: tensor} as <path>/<name>.npy in float32, rows sampled as by sample_rows."""
    import numpy as np
    host = {k: sample_rows(v.detach()).float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (> {DUMP_MAX_BYTES})")
    os.makedirs(path, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(path, k + ".npy"), a)


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------- CPU oracle arm
def oracle_step_factory(B: int, seed: int = 1234):
    from oracle import pyg_gat, synth
    N, Fin, Fe, H, Cc = cfg_dims()
    vol, vv = synth.synthetic_matrices(CFG["L"] + B + 1, N, seed=seed)
    bt = synth.make_batch(vol, vv, list(range(B)), CFG["L"])
    torch.manual_seed(seed)
    layer = pyg_gat.OracleGATConv(Fin, Cc, heads=H, concat=False, negative_slope=CFG["slope"], edge_dim=Fe)
    dout = torch.randn(B * N, Cc)

    def step():
        layer.zero_grad(set_to_none=True)
        out = layer(bt.x, bt.edge_index, bt.edge_attr)
        out.backward(dout)
        return out
    return step


def time_oracle(B: int, steps: int, warmup: int):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step = oracle_step_factory(B)
    for _ in range(warmup):
        step()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter(); step(); ts.append(time.perf_counter() - t0)
    return B / statistics.median(ts), cores, ts


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B = args.cpu_batch
    gps, cores, ts = time_oracle(B, max(1, args.steps), max(1, min(args.warmup, 2)))
    line = {
        "impl": "reference", "metric": METRIC, "value": gps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * statistics.median(ts), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"default GNN_param.yaml GATConv fwd+bwd; CPU sample of {B} graphs per step "
                               f"(the 4096-graph batch needs >88 GB of PyG intermediates on a CPU)",
                   "nodes": 30, "heads": 6, "hidden": 500, "seq_length": 42},
        "cpu_baseline": {"value": gps, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{B} graphs/step, {args.steps} steps, PyG-2.3.0-order torch eager restatement "
                                   "(PyG itself is not installable here)"},
        "e2e": {"value": gps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- our arm
class HotPath:
    """The hot path through the C ABI on preallocated buffers (what GATConv.forward/backward call)."""

    def __init__(self, B: int, device, seed: int, structured: bool = False, first: int = 0, total: int = 0):
        """B graphs = windows [first, first + B) of a synthetic stack holding `total` (default B) windows; weights, data
        and dout are functions of (seed, total) only, so ranks given the same seed and disjoint window ranges hold
        shards of one global batch (dp_selfcheck)."""
        self.structured = structured
        total = total or B
        import spotv2net_b200 as sv
        from spotv2net_b200 import _lib
        self.sv, self._lib = sv, _lib
        self.lib = sv.load_library()
        self.dev = device
        N, Fin, Fe, H, Cc = cfg_dims()
        self.B, self.N, self.Fin, self.Fe, self.H, self.Cc = B, N, Fin, Fe, H, Cc
        g = torch.Generator(device=device).manual_seed(seed)
        T = total + CFG["L"] + 1
        mats = []
        for _ in range(2):                       # synthetic standardized H5 content: symmetric N(0,1) [T, N, N]
            a = torch.randn(T, N, N, device=device, generator=g)
            mats.append((a + a.transpose(1, 2)) / 2 ** 0.5)
        self.ds = sv.WindowDataset(mats[0], mats[1], seq_length=CFG["L"], device=device, drop_first=0)
        self.batch = self.ds.collate(torch.arange(first, first + B))
        self.win = sv.WindowSource(self.ds.volvol, torch.arange(first, first + B, device=device, dtype=torch.int32), CFG["L"], checked=True)
        torch.manual_seed(seed)
        self.layer = sv.GATConv(Fin, Cc, heads=H, concat=False, negative_slope=CFG["slope"], edge_dim=Fe).to(device)
        n, HC = B * N, H * Cc
        # p_format 1 (the library's default wherever its kernels apply): the projection travels as the fp16 operand pair the
        # GEMM epilogue writes; --p-format 0 keeps the fp32 P_aug of round 1
        pf = getattr(HotPath, "P_FORMAT", None)
        if pf is None:
            pf = 1 if sv.gat_conv.pair_format_applies(N, Fe, Cc, 0, 0) else 0
        self.pair = pf == 1
        self.desc = _lib.GatDesc(B, N, Fin, Fe, H, Cc, N * (N - 1), 0, CFG["slope"], self.lib.spotv2_gat_ldp(H, Cc), 0, 0,
                                 0.0, 1 if structured else 0, 0, 0, pf)
        n_aug = self.lib.spotv2_gat_n_aug(C.byref(self.desc))
        a, b, c = C.c_size_t(), C.c_size_t(), C.c_size_t()
        _lib.check(self.lib.spotv2_gat_workspace_bytes(C.byref(self.desc), C.byref(a), C.byref(b), C.byref(c)), "ws")
        f32 = dict(device=device, dtype=torch.float32)
        f = C.c_size_t()
        _lib.check(self.lib.spotv2_gat_attn_fwd_workspace_bytes(C.byref(self.desc), C.byref(f)), "attn_fwd ws")
        self.ws = torch.empty(max(a.value, b.value, c.value, f.value), device=device, dtype=torch.uint8)
        self.W_aug = torch.empty(n_aug, Fin, **f32)
        self.v = torch.empty(H, Fe, **f32)
        self.P_aug = (torch.empty(2, n, self.lib.spotv2_gat_ld16(n_aug), device=device, dtype=torch.float16) if self.pair
                      else torch.empty(n, self.desc.ldp, **f32))
        self.p_amax = torch.empty(8, **f32)
        self.sd32 = torch.empty(n, 2 * H, **f32) if self.pair else None
        et = C.c_size_t()
        _lib.check(self.lib.spotv2_gat_edge_terms_bytes(C.byref(self.desc), C.byref(et)), "edge_terms_bytes")
        self.edge_terms = torch.empty(et.value // 4, **f32)       # <e_ij, v_h>: written by attn_fwd, read by attn_bwd
        self.d_edge_terms = torch.empty_like(self.edge_terms) if structured else None
        wdv = C.c_size_t()
        _lib.check(self.lib.spotv2_windows_dv_workspace_bytes(C.byref(self.desc), C.byref(wdv)), "windows_dv ws")
        self.ws_dv = torch.empty(wdv.value, device=device, dtype=torch.uint8) if structured else None
        wet = C.c_size_t()
        _lib.check(self.lib.spotv2_edge_terms_from_windows_workspace_bytes(C.byref(self.desc), C.byref(wet)), "edge_terms ws")
        self.ws_w = torch.empty(wet.value, device=device, dtype=torch.uint8) if (structured and wet.value) else None
        self.out = torch.empty(n, Cc, **f32)
        self.dout = torch.randn(total * N, Cc, generator=g, **f32)[first * N:(first + B) * N].contiguous()
        self.tc = bool(self.lib.spotv2_gat_uses_tensor_cores(C.byref(self.desc)))
        # tensor-core operand pairs (scaled fp16 hi/lo + 8-float scale block): x once per step, dP from attn_bwd
        f16 = dict(device=device, dtype=torch.float16)
        self.ldf16, self.ldp16 = self.lib.spotv2_gat_ld16(Fin), self.lib.spotv2_gat_ld16(n_aug)
        self.dP_aug = None if self.tc else torch.empty(n, self.desc.ldp, **f32)
        self.dP16 = torch.empty(2, n, self.ldp16, **f16) if self.tc else None
        # x as the GEMMs' operand pair: emitted by the collation (spotv2_collate_windows_pair; the dataset fixes the scale),
        # as a WindowDataset batch delivers it; --split-x-in-step re-derives it from the fp32 x inside the step (round 1)
        self.x_from_collation = self.tc and not getattr(HotPath, "SPLIT_X_IN_STEP", False) and self.batch.spot_x16 is not None
        if self.x_from_collation:
            self.x16, self.x_blk = self.batch.spot_x16
        else:
            self.x16 = torch.empty(2, n, self.ldf16, **f16) if self.tc else None
            self.x_blk = torch.empty(8, **f32) if self.tc else None
        self.dp_blk = torch.empty(8, **f32) if self.tc else None
        self.dW_aug = torch.empty(n_aug, Fin, **f32)
        self.dv = torch.empty(H, Fe, **f32)
        # flat gradient arena: the one buffer the data-parallel all-reduce moves
        sizes = [HC * Fin, HC, HC, HC * Fe, HC, Cc]
        self.arena = torch.empty(sum(sizes), **f32)
        self.g_W, self.g_as, self.g_ad, self.g_We, self.g_ae, self.g_b = torch.split(self.arena, sizes)
        # counted from the ncu launch list (profiles/r1t_launch_list_summary.txt): fold x2 (W_aug rows, v); amax x5 (x, W_aug x2,
        # dout, ds|dd); split x3 (x, W_aug, ds|dd); GEMM fwd; attn fwd; attn bwd + 2 partial reduces; GEMM bwd + split-K
        # reduce; unfold
        # counted from the ncu launch list (profiles/r2b_launch_list_summary.txt): p_format 1: fold, W_aug statistics + split, GEMM, attention
        # forward, dout prepass, attention backward, partial reduce, ds|dd split, GEMM, split-K reduce, unfold = 12; p_format 0 on the
        # tensor-core GEMM: 17 (amax / split passes over W_aug, dout, ds|dd); CUDA-core GEMM: 10
        self.kernels_per_step = (12 if self.pair else 17) if self.tc else 10
        if N > 32:   # large-universe path (profiles/r1t_config_D_launch_list_summary.txt): attn fwd 3 (logits, softmax, GEMM);
            # attn bwd 11 (+ amax/split of dP on the tensor-core path); fold x2, amax/split of x and W_aug, two projection
            # GEMMs + split-K reduce, unfold
            self.kernels_per_step = 26 if self.tc else 19
        self.ev = {}

    def step(self, timed_events=None, allreduce=None):
        lib, d, p, L = self.lib, C.byref(self.desc), self._lib.ptr, self.layer
        st = torch.cuda.current_stream(self.dev).cuda_stream
        chk = self._lib.check

        def mark(name):
            if timed_events is not None:
                e = torch.cuda.Event(enable_timing=True); e.record(); timed_events.append((name, e))
        mark("start")
        chk(lib.spotv2_gat_fold(d, p(L.lin_src.weight), p(L.att_src), p(L.att_dst), p(L.lin_edge.weight),
                                p(L.att_edge), p(self.W_aug), p(self.v), st), "fold")
        mark("fold")
        xh = self.x16[0] if self.tc else None
        xl = self.x16[1] if self.tc else None
        ph = self.dP16[0] if self.tc else None
        pl = self.dP16[1] if self.tc else None
        if self.tc and not self.x_from_collation:      # x given as fp32 only: one amax + one split pass per step
            chk(lib.spotv2_split_f16(p(self.batch.x), self.B * self.N, self.Fin, self.Fin, 0, 0, p(xh), p(xl), self.ldf16,
                                     p(self.x_blk), st), "split_f16")
        if self.pair:
            chk(lib.spotv2_proj_fwd_pair(d, p(xh), p(xl), p(self.x_blk), p(self.W_aug), p(self.P_aug[0]), p(self.P_aug[1]),
                                         p(self.p_amax), p(self.sd32), p(self.ws), self.ws.numel(), st), "proj_fwd_pair")
        else:
            chk(lib.spotv2_proj_fwd(d, p(self.batch.x), p(xh), p(xl), p(self.x_blk), p(self.W_aug), p(self.P_aug), p(self.p_amax),
                                    p(self.ws), self.ws.numel(), st), "proj_fwd")
        mark("proj_fwd")
        win = self.win
        if self.structured:      # structured edge source: the [L,N,N] windows instead of the materialised edge rows
            chk(lib.spotv2_edge_terms_from_windows(d, p(win.volvol), win.volvol.shape[0], win.L, p(win.t0), p(self.v),
                                                   p(self.edge_terms), p(self.ws_w), self.ws_w.numel() if self.ws_w is not None else 0,
                                                   st), "edge_terms_from_windows")
            mark("edge_terms")
        ea = None if self.structured else self.batch.edge_attr
        tbl = None if self.structured else self.batch.spot_topology.table
        if self.pair:
            chk(lib.spotv2_gat_attn_fwd_pair(d, p(self.P_aug[0]), p(self.P_aug[1]), p(self.p_amax), p(self.sd32), p(ea), p(tbl), p(self.v),
                                             p(L.bias), p(self.out), None, p(self.edge_terms), st), "attn_fwd_pair")
            mark("attn_fwd")
            chk(lib.spotv2_gat_attn_bwd_pair(d, p(self.P_aug[0]), p(self.P_aug[1]), p(self.p_amax), p(self.sd32), p(ea), p(self.edge_terms),
                                             p(tbl), p(self.v), p(self.dout), p(ph), p(pl), p(self.dp_blk),
                                             None if self.structured else p(self.dv), p(self.d_edge_terms),
                                             p(self.g_b), p(self.ws), self.ws.numel(), st), "attn_bwd_pair")
        else:
            chk(lib.spotv2_gat_attn_fwd(d, p(self.P_aug), p(ea), p(tbl), p(self.v), p(L.bias), p(self.out), None,
                                        p(self.edge_terms), p(self.ws), self.ws.numel(), st), "attn_fwd")
            mark("attn_fwd")
            chk(lib.spotv2_gat_attn_bwd(d, p(self.P_aug), p(self.p_amax), p(ea), p(self.edge_terms), p(tbl),
                                        p(self.v), p(self.dout), p(self.dP_aug), p(ph), p(pl), p(self.dp_blk),
                                        None if self.structured else p(self.dv), p(self.d_edge_terms),
                                        p(self.g_b), p(self.ws), self.ws.numel(), st), "attn_bwd")
        mark("attn_bwd")
        if self.structured:
            chk(lib.spotv2_windows_dv(d, p(win.volvol), win.volvol.shape[0], win.L, p(win.t0), p(self.d_edge_terms), p(self.dv),
                                      p(self.ws_dv), self.ws_dv.numel(), st), "windows_dv")
            mark("windows_dv")
        chk(lib.spotv2_proj_bwd_weight(d, p(self.batch.x), p(xh), p(xl), p(self.x_blk), p(self.dP_aug), p(ph), p(pl),
                                       p(self.dp_blk), p(self.dW_aug), p(self.ws), self.ws.numel(), st), "proj_bwd_weight")
        mark("proj_bwd_weight")
        chk(lib.spotv2_gat_unfold(d, p(L.lin_src.weight), p(L.att_src), p(L.att_dst), p(L.lin_edge.weight), p(L.att_edge),
                                  p(self.dW_aug), p(self.dv), p(self.g_W), p(self.g_as), p(self.g_ad), p(self.g_We),
                                  p(self.g_ae), st), "unfold")
        mark("unfold")
        if allreduce is not None:
            allreduce(self.arena)
            mark("allreduce")

    def outputs(self) -> dict:
        """What GATConv forward + backward hands its caller after the last step: the layer output and each parameter's
        gradient, shaped like the parameter."""
        grads = (("lin_src.weight", self.g_W), ("att_src", self.g_as), ("att_dst", self.g_ad),
                 ("lin_edge.weight", self.g_We), ("att_edge", self.g_ae), ("bias", self.g_b))
        res = {"out": self.out}
        res.update({f"{k}.grad": g.view_as(self.layer.get_parameter(k)) for k, g in grads})
        return res


def bind_to_gpu_numa(local: int):
    """Pin this rank's threads to the CPUs NVML lists as local to its GPU, BEFORE any pinned host buffer is allocated (first
    touch then places the staging buffers on the GPU's NUMA node).  Round 1 measured all ranks pinning on node 0 and the
    host -> device rate per GPU falling to 22 - 28 GB/s at N >= 4.  Returns a short description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1]
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return {"bound": True, "cpus": len(allowed), "first": allowed[0], "last": allowed[-1]}
        return {"bound": False, "why": "NVML affinity mask does not intersect this process's CPU set"}
    except Exception as ex:                                  # no NVML / no permission: run unbound, say so
        return {"bound": False, "why": repr(ex)[:120]}


def run_ours(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (our arm) needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    affinity = bind_to_gpu_numa(local) if world > 1 else {"bound": False, "why": "single rank"}
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL prints its version banner on the C stdout while the communicator comes up; stdout carries the ONE JSON
        # line, so file descriptor 1 points at stderr until the first collective is through
        import ctypes
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize()
            ctypes.CDLL(None).fflush(None)
        finally:
            os.dup2(saved, 1)
            os.close(saved)
    B = args.batch
    dp_check = dp_selfcheck(dev, rank, world) if world > 1 else None
    hp = HotPath(B, dev, seed=1234 + rank)

    def allreduce(t):
        dist.all_reduce(t, op=dist.ReduceOp.AVG)         # the 1/world scaling rides inside the collective
    ar = allreduce if world > 1 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, 3)):
        hp.step(allreduce=ar)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    per_step_events = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        evs = []
        hp.step(timed_events=evs, allreduce=ar)
        per_step_events.append(evs)
    e1.record()
    barrier()
    elapsed_ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, hp.outputs())
    if world > 1:
        t = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = t.item()
    ms_per_step = elapsed_ms / args.steps
    value = world * B / (ms_per_step * 1e-3)

    # per-kernel device times (CUDA events on the launching stream, averaged over the timed steps)
    phase_ms = {}
    for evs in per_step_events:
        for (n0, a), (n1, b) in zip(evs[:-1], evs[1:]):
            phase_ms.setdefault(n1, []).append(a.elapsed_time(b))
    phase_ms = {k: sum(v) / len(v) for k, v in phase_ms.items()}

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    ATTN_BYTES_FWD, ATTN_BYTES_BWD = attn_bytes()
    PROJ_FLOP_PER_GRAPH = proj_flop_per_graph()
    t_attn = (phase_ms["attn_fwd"] + phase_ms["attn_bwd"]) * 1e-3
    attn_gbs = (ATTN_BYTES_FWD + ATTN_BYTES_BWD) * B / t_attn / 1e9
    traffic = None
    try:
        if args.config == "A":
            traffic = json.load(open(os.path.join(ROOT, "profiles", "attn_traffic.json")))
    except Exception:
        pass
    traffic_detail = traffic
    if isinstance(traffic, dict):
        traffic = traffic.get("sum")
    roofline = {"bound": "hbm", "kernel": ("gat_attn_fwd16_kernel + dout_pair_kernel + gat_attn_bwd2_kernel (p_format 1: P, dout, dP as fp16 operand pairs)" if hp.pair else "gat_attn_fwd_kernel + gat_attn_bwd2_kernel (p_format 0: fp32 P_aug)") if CFG["N"] <= 32 else
                "attn_large.cu (lg_edge_logit, lg_softmax, bgemm, lg_softmax_bwd, lg_dv kernels)", "achieved": attn_gbs,
                "peak": hbm_peak, "unit": "GB/s", "frac": attn_gbs / hbm_peak, "traffic": traffic,
                "traffic_detail": traffic_detail,
                "algorithmic_bytes_per_launch_pair": (ATTN_BYTES_FWD + ATTN_BYTES_BWD) * B,
                "peak_source": peak_src, "frac_of_8TBs": attn_gbs / 8000.0,
                "fwd": {"ms": phase_ms["attn_fwd"], "GBs": ATTN_BYTES_FWD * B / phase_ms["attn_fwd"] / 1e6},
                "bwd": {"ms": phase_ms["attn_bwd"], "GBs": ATTN_BYTES_BWD * B / phase_ms["attn_bwd"] / 1e6}}
    t_proj = (phase_ms["proj_fwd"] + phase_ms["proj_bwd_weight"]) * 1e-3
    f16_peak = peaks.get("bf16_tflops_sustained", 1400.0)
    proj = {"bound": "tensor", "kernel": "projection GEMMs (P = x W^T, dW = dP^T x)",
            "achieved": PROJ_FLOP_PER_GRAPH * B / t_proj / 1e12, "peak": f16_peak, "unit": "TFLOP/s",
            "frac": PROJ_FLOP_PER_GRAPH * B / t_proj / 1e12 / f16_peak,
            "issued_TFLOPs": 3 * PROJ_FLOP_PER_GRAPH * B / t_proj / 1e12,
            "peak_source": "bf16_tflops_sustained (MEASURED_PEAKS.json; kind::f16 issues at the bf16 rate); 'achieved' counts "
                           "algorithmic fp32 flops, the 3-product fp16-pair scheme issues 3x that ('issued_TFLOPs')",
            "fwd_ms": phase_ms["proj_fwd"], "bwd_ms": phase_ms["proj_bwd_weight"]}

    # `e2e` is the strict reading: the host tensors the reference's `data.to(device)` moves (x, edge_index,
    # edge_attr, y_x) cross PCIe every step.  `e2e_windows` is this library's own input path (the [T,N,N] stacks
    # cross instead, 83x fewer bytes, and the batch is collated on the device); reported beside it, never as `e2e`.
    # Side measurement: the same step captured once into a CUDA graph (every entry point of the library is capture
    # safe) and replayed - what a static-shape training loop would launch.  The bench value above stays on eager
    # launches, where CUDA events can sit between the kernels of the timed region.
    graph_info = None
    if world == 1 and not args.no_graph:
        try:
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                hp.step()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                hp.step()
            g.replay()
            torch.cuda.synchronize(dev)
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(args.steps):
                g.replay()
            g1.record()
            torch.cuda.synchronize(dev)
            gms = g0.elapsed_time(g1) / args.steps
            graph_info = {"ms_per_step": gms, "value": B / (gms * 1e-3), "unit": UNIT,
                          "note": f"one CUDA graph replay per step ({hp.kernels_per_step} kernels), {args.steps} steps"}
            del g
        except Exception as ex:
            graph_info = {"value": None, "error": repr(ex)[:300]}
            torch.cuda.synchronize(dev)
    structured = None
    if not args.no_structured:
        try:
            structured = run_structured(args, dev, world, rank, barrier)
        except Exception as ex:
            structured = {"value": None, "error": repr(ex)[:300]}
    train_step = None
    if not args.no_structured and args.config == "A":
        try:
            train_step = run_train_step(args, dev, world, rank, barrier)
        except Exception as ex:
            train_step = {"value": None, "error": repr(ex)[:300]}
    e2e = e2e_win = None
    if not args.no_e2e:
        try:
            e2e = run_e2e(args, hp, dev, world, rank, barrier)
        except Exception as ex:           # the device-timed line must still print
            e2e = {"value": None, "unit": UNIT, "error": repr(ex)[:300]}
        try:
            e2e_win = run_e2e_windows(args, hp, dev, world, rank, barrier)
        except Exception as ex:
            e2e_win = {"value": None, "unit": UNIT, "error": repr(ex)[:300]}

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.config == "A":
        try:
            gps, cores, ts = time_oracle(args.cpu_batch, 3, 1)
            cpu_baseline = {"value": gps, "unit": UNIT, "cores": cores, "kind": "port",
                            "sample": f"{args.cpu_batch} graphs/step x 3 steps (+1 warm-up), PyG-order torch eager oracle, "
                                      f"median {statistics.median(ts):.2f} s/step"}
        except Exception as ex:
            cpu_baseline = {"value": None, "error": repr(ex)[:300]}

    if rank == 0:
        N, Fin, Fe, H, Cc = cfg_dims()
        line = {
            "metric": METRIC_BY_CONFIG[args.config], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",      # fp32-accurate: every product is a 3-term fp16-pair split with fp32 accumulation
            "config": {"workload": CONFIGS[args.config]["name"] + ", fp32, GATConv fwd+bwd" +
                                   (" + NCCL gradient all-reduce" if world > 1 else ""),
                       "nodes": N, "in_channels": Fin, "edge_dim": Fe, "heads": H, "hidden": Cc, "batch_per_gpu": B,
                       "l2": f"inputs (x {B * N * Fin * 4 / 1e6:.0f} MB, edge_attr {B * N * (N - 1) * Fe * 4 / 1e9:.2f} GB, "
                             f"P {B * N * H * Cc * 4 / 1e6:.0f} MB per step) exceed the 126 MB L2; no flush needed",
                       "parallelism": f"dp{world}", "launch": "eager launches, CUDA events between the entry points"},
            "phase_ms": phase_ms, "roofline": roofline, "roofline_projection": proj, "cpu_baseline": cpu_baseline,
            "dp_gradient_check": dp_check, "cuda_graph_replay": graph_info, "structured_edge_source": structured, "train_step": train_step, "e2e": e2e, "e2e_windows": e2e_win, "gpu_launches": hp.kernels_per_step * args.steps, "clocks": clocks,
            "p_format": 1 if hp.pair else 0, "cpu_affinity": affinity,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dp_selfcheck(dev, rank, world, per_rank: int = 64):
    """N > 1 correctness on the hardware being timed (SURVEY.md:279): every rank runs its shard (64 graphs) of ONE global
    batch through the hot path and the arena is all-reduced exactly as in the timed loop; rank 0 also runs the whole
    concatenated batch on its own GPU.  AVG-all-reduced arena x world must equal the single-GPU gradient to 1e-5
    (max-norm relative, per parameter tensor).  Raises on mismatch: a wrong multi-GPU number is never printed."""
    import torch.distributed as dist
    hp = HotPath(per_rank, dev, seed=4321, first=rank * per_rank, total=world * per_rank)
    hp.step(allreduce=lambda t: dist.all_reduce(t, op=dist.ReduceOp.AVG))
    torch.cuda.synchronize(dev)
    worst = torch.zeros(1, device=dev, dtype=torch.float64)
    if rank == 0:
        full = HotPath(world * per_rank, dev, seed=4321)
        full.step()
        torch.cuda.synchronize(dev)
        for mine, ref in zip((hp.g_W, hp.g_as, hp.g_ad, hp.g_We, hp.g_ae, hp.g_b),
                             (full.g_W, full.g_as, full.g_ad, full.g_We, full.g_ae, full.g_b)):
            err = ((mine.double() * world - ref.double()).abs().max() / ref.double().abs().max()).item()
            worst[0] = max(worst.item(), err)
        del full
    dist.broadcast(worst, 0)
    del hp
    torch.cuda.empty_cache()
    if not worst.item() <= 1e-5:
        raise SystemExit(f"bench.py: all-reduced gradient differs from the single-GPU gradient on the concatenated batch "
                         f"by {worst.item():.2e} (> 1e-5)")
    return {"max_rel_err_vs_single_gpu": worst.item(), "graphs": world * per_rank, "ok": True}


def run_config_c(args):
    """BASELINE configs[2] through the public module API: GATModel(8 heads, hidden [256, 256], concat_heads) forward + MSE +
    autograd backward on one collated 4096-graph batch (utils/models.py:90-104; config/GNN_param.yaml:28-38 widened).  The
    line's value is the reduced-precision mode the config names ("half": one fp16 tensor-core product per MMA step with fp32
    accumulate in the projections AND the attention kernels, P / dP / dout stored as fp16 hi planes - half the attention
    bytes); the fp32-accurate mode is reported beside it.  The attention kernels' share comes from one extra step under torch.profiler (kernel durations by
    name), never from the timed steps."""
    import spotv2net_b200 as sv
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (our arm) needs a CUDA device: the hot path has no CPU fallback")
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    B, N, L, H, Cc = args.batch, 30, CFG["L"], 8, 256
    g = torch.Generator(device=dev).manual_seed(1234)
    mats = []
    for _ in range(2):
        a = torch.randn(B + L + 1, N, N, device=dev, generator=g)
        mats.append((a + a.transpose(1, 2)) / 2 ** 0.5)
    ds = sv.WindowDataset(mats[0], mats[1], seq_length=L, device=dev, drop_first=0)
    bt = ds.collate(torch.arange(B))
    torch.manual_seed(0)
    model = sv.GATModel(N * L, 3 * L, H, 1, dim_hidden_layers=[Cc, Cc], concat_heads=True).to(dev)

    def step():
        model.zero_grad(set_to_none=True)
        loss = torch.nn.functional.mse_loss(model(bt), bt.y_x)
        loss.backward()
        return loss

    sampler = ClockSampler(dev.index or 0)
    res, attn_ms = {}, {}
    for prec in ("fp32", "half"):
        model.set_precision(prec)
        for _ in range(max(args.warmup, 3) + 2):          # (+2: the first mode also pays the caching allocator's growth)
            step()
        torch.cuda.synchronize(dev)
        if prec == "half":
            sampler.start()
        # one event pair per step: the figure is the MEDIAN step (a first-use allocator growth or a lazily loaded module inside
        # one of the timed steps of this eager two-layer model has cost 2x on some boxes; the mean and the slowest step are kept
        # beside it)
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
        evs[0].record()
        for k_ in range(args.steps):
            loss = step()
            evs[k_ + 1].record()
        torch.cuda.synchronize(dev)
        per = sorted(evs[k_].elapsed_time(evs[k_ + 1]) for k_ in range(args.steps))
        ms = per[len(per) // 2] if len(per) % 2 else 0.5 * (per[len(per) // 2 - 1] + per[len(per) // 2])
        res[prec] = {"ms_per_step": ms, "value": B / (ms * 1e-3), "unit": UNIT, "loss": loss.item(),
                     "ms_per_step_mean": evs[0].elapsed_time(evs[-1]) / args.steps, "ms_per_step_max": per[-1],
                     "timing": "median of per-step CUDA-event times"}
        if prec == "half":
            clocks = sampler.stop()
            if args.dump_outputs:
                dump_outputs(args.dump_outputs, {"loss": loss, **{f"{k}.grad": p.grad for k, p in model.named_parameters()}})
        # the attention kernels' share (incl. the backward's operand preparation of dout): one extra step under torch.profiler
        try:
            from torch.profiler import profile, ProfilerActivity
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                step()
                torch.cuda.synchronize(dev)
            attn_ms[prec] = sum(e.device_time_total for e in prof.key_averages() if "gat_attn" in e.key or "dout_pair" in e.key) * 1e-3
        except Exception:
            attn_ms[prec] = None
    # algorithmic attention bytes per graph: layer 0 (concat: out and dout are H*C wide), layer 1 (head mean); eb = bytes per
    # stored element of P and dP: 4 in the fp32-accurate mode (an fp16 hi|lo pair, or fp32), 2 in the half mode (hi plane only)
    edge = N * (N - 1) * 3 * L * 4

    def attn_bytes(eb):
        Pb = N * H * Cc * eb
        l0 = (edge + Pb + N * H * Cc * 4) + (edge + Pb + N * H * Cc * 4 + Pb)
        l1 = (edge + Pb + N * Cc * 4) + (edge + Pb + N * Cc * 4 + Pb)
        return l0 + l1
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = peaks.get("hbm_gbs", 6650.0)

    def roof(prec, eb):
        ms = attn_ms.get(prec)
        ach = attn_bytes(eb) * B / (ms * 1e-3) / 1e9 if ms else None
        return {"bound": "hbm", "kernel": "gat_attn_fwd16_kernel + dout_pair_kernel + gat_attn_bwd2_kernel, both layers",
                "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm if ach else None, "traffic": None,
                "attention_ms_profiled_step": ms, "algorithmic_bytes_per_step": attn_bytes(eb) * B, "bytes_per_P_element": eb,
                "peak_source": "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"}

    res["fp32"]["roofline"] = roof("fp32", 4)
    line = {"metric": METRIC_BY_CONFIG["C"], "value": res["half"]["value"], "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": res["half"]["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None,
            "dtype": "f16 (one tensor-core product per MMA step, fp32 accumulate; P, dP and dout travel as fp16 hi planes: p_format 1 "
                     "with gemm_algo 3 - the config's reduced-precision class; the fp32-accurate mode is under fp32_mode)",
            "data": "synthetic",
            "config": {"workload": CONFIGS["C"]["name"] + ", GATModel forward + MSE + autograd backward", "nodes": N, "heads": H,
                       "hidden": [Cc, Cc], "batch_per_gpu": B, "parallelism": "dp1",
                       "l2": "inputs (x 619 MB, edge_attr 1.80 GB, P 0.5 - 1 GB per layer) exceed the 126 MB L2; no flush needed"},
            "fp32_mode": res["fp32"],
            "roofline": roof("half", 2),
            "cpu_baseline": None, "e2e": None, "gpu_launches": None, "clocks": clocks}
    print(json.dumps(line), flush=True)


def run_train_step(args, dev, world, rank, barrier):
    """Side measurement (SURVEY 8d "full train-step graphs/s"): what one iteration of the reference's loop costs
    (5_train_SpotV2Net.py:150-160) - GATModel forward (GATConv + ReLU + Linear), MSE loss, backward, Adam - on a collated
    4096-graph batch of the default configuration, through the public module API; device time over the timed steps."""
    import spotv2net_b200 as sv
    B, L, N = args.batch, CFG["L"], CFG["N"]
    g = torch.Generator(device=dev).manual_seed(99 + rank)
    mats = []
    for _ in range(2):
        a = torch.randn(B + L + 1, N, N, device=dev, generator=g)
        mats.append((a + a.transpose(1, 2)) / 2 ** 0.5)
    ds = sv.WindowDataset(mats[0], mats[1], seq_length=L, device=dev, drop_first=0)
    bt = ds.collate(torch.arange(B))
    torch.manual_seed(7)
    model = sv.GATModel(N * L, 3 * L, CFG["H"], 1, [CFG["C"]], negative_slope=CFG["slope"]).to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    crit = torch.nn.MSELoss()

    def step():
        opt.zero_grad(set_to_none=True)
        loss = crit(model(bt), bt.y_x)
        loss.backward()
        opt.step()
        return loss

    for _ in range(3):
        step()
    barrier()
    steps = max(2, min(args.steps, 10))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    loss.item()
    barrier()
    ms = e0.elapsed_time(e1) / steps
    del model, opt, bt, ds
    torch.cuda.empty_cache()
    return {"value": world * B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps,
            "what": "spotv2net_b200.GATModel (default config: GATConv 1260 -> 6 x 500 mean, ReLU, Linear 500 -> 1) forward + MSELoss + "
                    "backward + torch.optim.Adam step on one collated batch; per-rank device time, no all-reduce"}


def run_structured(args, dev, world, rank, barrier):
    """Side measurement, NOT the bench value: the same step with the structured edge source (SURVEY.md 8f-2) - the
    attention kernels read the [L,N,N] co-volatility windows the dataset builds edge_attr from (151 KB per graph)
    instead of the materialised edge rows (438 KB).  Model specific, so the generic edge_attr path stays the metric."""
    hp = HotPath(args.batch, dev, seed=1234 + rank, structured=True)
    for _ in range(3):
        hp.step()
    barrier()
    steps = max(2, min(args.steps, 10))
    all_ev = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        ev = []
        hp.step(timed_events=ev)
        all_ev.append(ev)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / steps
    ph = {}
    for evs in all_ev:
        for (n0, a), (n1, b) in zip(evs[:-1], evs[1:]):
            ph.setdefault(n1, []).append(a.elapsed_time(b))
    ph = {k: sum(v) / len(v) for k, v in ph.items()}
    del hp
    torch.cuda.empty_cache()
    return {"value": world * args.batch / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "phase_ms": ph,
            "note": "per-rank device time, no all-reduce; edge terms from the windows (edge_terms), attention forward / backward "
                    "on the terms, dv from the windows (windows_dv)"}


def run_e2e_windows(args, hp, dev, world, rank, barrier):
    """The metric end to end through the repo's public API with HOST inputs: the standardized matrix stacks the
    reference reads from its two H5 files (config/GNN_param.yaml:2-3) sit in pinned host memory; every step
    copies the [T, N, N] stacks its windows need to the device (WindowDataset.vol / .volvol), collates the batch
    on the device (`WindowDataset.collate`, the drop-in for CovarianceLaggedDataset + DataLoader,
    5_train_SpotV2Net.py:90,142-143), runs GATConv forward + backward through autograd and reads the loss back.
    This is the input path a user of this library's WindowDataset takes (reported as `e2e_windows`); the headline
    `e2e` leg (`run_e2e`) ships the already-expanded PyG tensors (x, edge_index, edge_attr: 83x the bytes) the
    way the reference's `data.to(device)` does."""
    # structured=True: the batches carry window references, edge_attr is never materialised in HBM (SURVEY 8f-2)
    layer, dout = hp.layer, hp.dout
    vol_h, vv_h = hp.ds.vol.cpu().pin_memory(), hp.ds.volvol.cpu().pin_memory()
    idx = torch.arange(hp.B)
    h2d = (vol_h.numel() + vv_h.numel()) * 4 + hp.B * 4        # both stacks + the window starts
    steps = max(2, min(args.steps, args.e2e_steps))

    # Two stack copies on the device, filled alternately on a copy stream: the H2D of step i+1 and the host-side launch work
    # of step i+1 run under the kernels of step i.  Every step's loss is still read back inside the timed region - one step
    # late, so that the host never waits on the step it has just launched.
    copy_stream = torch.cuda.Stream(dev)
    main_stream = torch.cuda.current_stream(dev)
    sets = [hp.sv.WindowDataset(hp.ds.vol.clone(), hp.ds.volvol.clone(), seq_length=CFG["L"], device=dev, drop_first=0, structured=True) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]
    for s_ in range(2):
        freed[s_].record(main_stream)

    def issue_copy(s_):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[s_])
            sets[s_].vol.copy_(vol_h, non_blocking=True)
            sets[s_].volvol.copy_(vv_h, non_blocking=True)
            ready[s_].record(copy_stream)

    def launch(s_):
        main_stream.wait_event(ready[s_])
        bt = sets[s_].collate(idx)                           # window starts H2D + device-side gather (x, its operand pair, y)
        layer.zero_grad(set_to_none=True)
        out = layer(bt.x, bt.edge_index, bt.edge_attr, topology=bt.spot_topology, windows=bt.spot_windows)
        loss = (out * dout).sum()
        loss.backward()
        freed[s_].record(main_stream)
        return loss

    for _ in range(3):                                       # warm-up
        issue_copy(0)
        launch(0).item()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    issue_copy(0)
    pending = None
    for i in range(steps):
        if i + 1 < steps:
            issue_copy((i + 1) & 1)
        loss = launch(i & 1)
        if pending is not None:
            pending.item()                                   # D2H read of the previous step's result
        pending = loss
    pending.item()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / steps
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    return {"value": world * hp.B / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
            "ms_per_step": ms, "steps": steps,
            "api": "pinned host [T,N,N] vol / vol-of-vol stacks -> H2D (copy stream, two device copies) -> "
                   "spotv2net_b200.WindowDataset(structured=True).collate (device; edge_attr never materialised; x also as the GEMM "
                   "operand pair) -> GATConv forward + autograd backward on the window references -> loss.item() (read one step "
                   "late, inside the timed region)"}


def run_e2e(args, hp, dev, world, rank, barrier):
    """Same metric through the public module API with HOST buffers.  Every step copies that step's batch
    (x, edge_index, edge_attr, y_x: the tensors the reference's `data.to(device)` moves,
    5_train_SpotV2Net.py:143) from pinned host memory, runs GATConv forward + backward through autograd and
    reads a scalar back.  Like any input pipeline, the copy of step i+1 is issued on a second stream while
    step i computes (two device buffer sets); every copy and every read-back is inside the timed region."""
    bt = hp.batch
    keys = ("x", "edge_index", "edge_attr", "y_x")
    host = {k: getattr(bt, k).cpu().pin_memory() for k in keys}
    h2d = sum(t.numel() * t.element_size() for t in host.values())
    layer, dout = hp.layer, hp.dout
    steps = max(2, min(args.steps, args.e2e_steps))
    copy_stream = torch.cuda.Stream(dev)
    main_stream = torch.cuda.current_stream(dev)
    bufs = [{k: torch.empty_like(getattr(bt, k)) for k in keys} for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]       # copy into set s finished
    freed = [torch.cuda.Event() for _ in range(2)]       # compute on set s finished

    def issue_copy(s):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[s])
            for k in keys:
                bufs[s][k].copy_(host[k], non_blocking=True)
            ready[s].record(copy_stream)

    def compute(s):
        main_stream.wait_event(ready[s])
        d = bufs[s]
        layer.zero_grad(set_to_none=True)
        out = layer(d["x"], d["edge_index"], d["edge_attr"])
        loss = (out * dout).sum()
        loss.backward()
        freed[s].record(main_stream)
        return loss.item()                      # D2H read of the step's result

    for s in range(2):
        freed[s].record(main_stream)
    # the host side's ceiling: the same pinned -> device copies with no compute, all ranks at once
    barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(copy_stream):
        c0.record(copy_stream)
        for _ in range(3):
            for k in keys:
                bufs[0][k].copy_(host[k], non_blocking=True)
        c1.record(copy_stream)
    barrier()
    copy_only = 3 * h2d / (c0.elapsed_time(c1) * 1e-3) / 1e9
    copy_stats = {"h2d_GBs_copy_only": copy_only}
    if world > 1:
        import torch.distributed as dist
        g = [torch.zeros(1, device=dev, dtype=torch.float64) for _ in range(world)]
        dist.all_gather(g, torch.tensor([copy_only], device=dev, dtype=torch.float64))
        per_rank = [t.item() for t in g]
        copy_stats = {"h2d_GBs_copy_only_per_rank": per_rank, "h2d_GBs_copy_only_sum": sum(per_rank),
                      "note": "all ranks copy at once, no compute: what the host (memory + PCIe fabric) delivers"}
    for _ in range(3):                          # warm-up (also validates and caches nothing across steps)
        issue_copy(0); compute(0)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    issue_copy(0)
    for i in range(steps):
        if i + 1 < steps:
            issue_copy((i + 1) & 1)
        compute(i & 1)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / steps
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    return {"value": world * hp.B / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
            "ms_per_step": ms, "steps": steps, "h2d_GBs": h2d / (ms * 1e-3) / 1e9, "host_ceiling": copy_stats,
            "api": "spotv2net_b200.GATConv forward + autograd backward; pinned host inputs, copy of step i+1 overlapped "
                   "with step i on a second stream"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="graphs per GPU (default: 4096 for config A, 32 for config D)")
    ap.add_argument("--config", default="A", choices=sorted(CONFIGS), help="A = the bench line (default); C = wide two-layer variant; D = 500-node universe")
    ap.add_argument("--cpu-batch", type=int, default=128)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (profiling runs)")
    ap.add_argument("--no-structured", action="store_true", help="skip the structured-edge-source side measurement")
    ap.add_argument("--no-graph", action="store_true", help="skip the CUDA-graph replay side measurement")
    ap.add_argument("--p-format", type=int, default=None, choices=[0, 1], help="0: fp32 P_aug between GEMM and attention (round 1); 1: fp16 operand pair (default where it applies)")
    ap.add_argument("--split-x-in-step", action="store_true", help="derive x's operand pair from the fp32 x inside every step (round-1 behaviour)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (config A / D: out and the parameter gradients; "
                         "config C: loss and the parameter gradients of the half-precision mode) as DIR/<name>.npy, float32; arrays "
                         f"above {DUMP_MAX_ELEMS} elements are a fixed, seeded sample of their rows")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's outputs; the reference arm has none")
    CFG["N"] = CONFIGS[args.config]["N"]
    HotPath.SPLIT_X_IN_STEP = args.split_x_in_step
    HotPath.P_FORMAT = args.p_format
    if args.batch <= 0:
        args.batch = CONFIGS[args.config]["batch"]
    if args.impl == "reference":
        run_reference(args)
    elif args.config == "C":
        run_config_c(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
