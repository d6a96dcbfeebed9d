"""Cost of edge_attr.grad at config A (4096 graphs of 30 nodes, Fin 1260, Fe 126, 6 heads x 500, head mean) on one GPU.

  1. the layer backward with and without edge_attr.requires_grad, alternating in one process;
  2. spotv2_gat_edge_rows_grad alone, with its bytes (computed from shapes) and rate against the measured HBM copy peak;
  3. a GATModel training step (forward, MSE, backward) with standardize=True, with and without edge_attr.requires_grad:
     with it, the batch statistics are formed from edge_attr by eager torch ops and carry their own backward.
CUDA events; every arm warmed up; medians of --reps samples.  The card's name and power limit are read (nvidia-smi query,
read-only) and printed with the numbers.

    python tools/edge_grad_bench.py [--reps 30] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes as C
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import spotv2net_b200 as sv                       # noqa: E402
from spotv2net_b200 import _lib, gat_conv         # noqa: E402

B, N, L, H, CC = 4096, 30, 42, 6, 500
FIN, FE, R = N * L, 3 * L, N * (N - 1)
HBM_COPY_PEAK = 6462.0          # GB/s, measured b.copy_(a) on the B200 (BASELINE.md)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi unavailable"
    return f"{torch.cuda.get_device_name(0)} | nvidia-smi: {q}"


def timed(fn, reps):
    """Median and spread of fn's device time (ms) over reps calls, each bracketed by its own event pair."""
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return statistics.median(out), min(out), max(out)


def data(dev):
    g = torch.Generator(device=dev).manual_seed(1)
    T = B + L + 1
    mats = []
    for _ in range(2):
        a = torch.randn(T, N, N, device=dev, generator=g)
        mats.append((a + a.transpose(1, 2)) / 2 ** 0.5 + 1.0)
    ds = sv.WindowDataset(mats[0], mats[1], seq_length=L, device=dev, drop_first=0)
    return ds.collate(torch.arange(B)), g


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures the GPU and has no CPU mode")
    dev = torch.device("cuda:0")
    lines = [f"# edge_attr.grad cost at config A (B={B}, N={N}, Fin={FIN}, Fe={FE}, H={H}, C={CC}, head mean)",
             f"# card: {card()}", f"# medians of {args.reps} samples (CUDA events), arms alternating, [min, max] beside"]
    bt, g = data(dev)
    torch.manual_seed(0)
    layer = sv.GATConv(FIN, CC, heads=H, concat=False, edge_dim=FE).to(dev)
    x = bt.x.detach()
    ea_plain = bt.edge_attr.detach()
    ea_grad = ea_plain.clone().requires_grad_(True)
    dout = torch.randn(B * N, CC, device=dev, generator=g)
    topo = bt.spot_topology

    # ---- 1. layer backward, alternating
    def bwd(ea):
        def run():
            return outs[0].backward(dout)
        outs = []

        def prep():
            layer.zero_grad(set_to_none=True)
            ea.grad = None
            outs[:] = [layer(x, bt.edge_index, ea, topology=topo)]
        return prep, run

    arms = {"without edge grad": bwd(ea_plain), "with edge grad": bwd(ea_grad)}
    samples = {k: [] for k in arms}
    for it in range(args.reps + 3):
        for name, (prep, run) in arms.items():
            prep()
            torch.cuda.synchronize()
            t = timed(run, 1)[0]
            if it >= 3:                                   # first rounds: warm-up
                samples[name].append(t)
    med = {k: statistics.median(v) for k, v in samples.items()}
    lines.append("layer backward (ms):")
    for k, v in samples.items():
        lines.append(f"  {k:<20} {med[k]:.3f}  [{min(v):.3f}, {max(v):.3f}]")
    lines.append(f"  added by edge grad   {med['with edge grad'] - med['without edge grad']:.3f}")

    # ---- 2. the expansion kernel alone
    lib = sv.load_library()
    desc = gat_conv._desc(topo, FIN, FE, H, CC, False, 0.2)
    n_terms = gat_conv._edge_terms_bytes(desc) // 4
    d_et = torch.randn(n_terms, device=dev, generator=g)
    v = torch.randn(H, FE, device=dev, generator=g)
    d_ea = torch.empty(B * R, FE, device=dev)
    st = torch.cuda.current_stream().cuda_stream

    def expand():
        _lib.check(lib.spotv2_gat_edge_rows_grad(C.byref(desc), _lib.ptr(d_et), _lib.ptr(topo.table), _lib.ptr(v),
                                                 _lib.ptr(d_ea), st), "edge_rows_grad")
    for _ in range(5):
        expand()
    t_med, t_min, t_max = timed(expand, args.reps)
    wr, rd = B * R * FE * 4, n_terms * 4 + R * 4 + H * FE * 4
    gbs = (wr + rd) / (t_med * 1e-3) / 1e9
    lines.append("spotv2_gat_edge_rows_grad alone:")
    lines.append(f"  time (ms)            {t_med:.3f}  [{t_min:.3f}, {t_max:.3f}]")
    lines.append(f"  bytes                {wr / 1e9:.3f} GB written + {rd / 1e6:.1f} MB read (from shapes)")
    lines.append(f"  rate                 {gbs:.0f} GB/s = {gbs / HBM_COPY_PEAK:.2f} of the {HBM_COPY_PEAK:.0f} GB/s copy peak")

    # ---- 3. model training step, standardize=True
    torch.manual_seed(0)
    model = sv.GATModel(FIN, FE, H, 1, dim_hidden_layers=[CC], standardize=True).to(dev)
    model.train()
    ea_model = bt.edge_attr

    def step(with_grad):
        def run():
            model.zero_grad(set_to_none=True)
            ea_model.grad = None
            ea_model.requires_grad_(with_grad)
            loss = torch.nn.functional.mse_loss(model(bt), bt.y_x)
            loss.backward()
        return run
    samples = {"without edge grad": [], "with edge grad": []}
    for it in range(args.reps + 3):
        for name, w in (("without edge grad", False), ("with edge grad", True)):
            t = timed(step(w), 1)[0]
            if it >= 3:
                samples[name].append(t)
    ea_model.requires_grad_(False)
    med = {k: statistics.median(v) for k, v in samples.items()}
    lines.append("GATModel train step, standardize=True (forward + MSE + backward, ms):")
    for k, v in samples.items():
        lines.append(f"  {k:<20} {med[k]:.3f}  [{min(v):.3f}, {max(v):.3f}]")
    lines.append(f"  added by edge grad   {med['with edge grad'] - med['without edge grad']:.3f} (statistics from edge_attr "
                 "with their eager backward, copy-out, expansion)")
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
