"""Cost of the gradient through the returned attention coefficients at config A (4096 graphs of 30 nodes, Fin 1260, Fe 126,
6 heads x 500, head mean) on one GPU.

  1. the layer backward when alpha is returned but not in the loss, and when the loss has <alpha, G> (the backward then
     runs spotv2_alpha_to_pyg_grad and the attention backward's d_alpha variant), alternating in one process;
  2. spotv2_alpha_to_pyg_grad alone, with its bytes (computed from shapes) and rate against the measured HBM copy peak.
CUDA events; every arm warmed up; medians of --reps samples.  The card's name and power limit are read (nvidia-smi query,
read-only) and printed with the numbers.

    python tools/alpha_grad_bench.py [--reps 30] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes as C
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import spotv2net_b200 as sv                       # noqa: E402
from spotv2net_b200 import _lib                   # noqa: E402
from spotv2net_b200._lib import GatDesc           # noqa: E402
from edge_grad_bench import B, CC, FE, FIN, H, HBM_COPY_PEAK, N, R, card, data, timed   # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures the GPU and has no CPU mode")
    dev = torch.device("cuda:0")
    lines = [f"# alpha gradient cost at config A (B={B}, N={N}, Fin={FIN}, Fe={FE}, H={H}, C={CC}, head mean)",
             f"# card: {card()}", f"# medians of {args.reps} samples (CUDA events), arms alternating, [min, max] beside"]
    bt, g = data(dev)
    torch.manual_seed(0)
    layer = sv.GATConv(FIN, CC, heads=H, concat=False, edge_dim=FE).to(dev)
    x, ea = bt.x.detach(), bt.edge_attr.detach()
    dout = torch.randn(B * N, CC, device=dev, generator=g)
    G = torch.randn(B * R + B * N, H, device=dev, generator=g)
    topo = bt.spot_topology

    # ---- 1. layer backward, alternating
    def bwd(with_g):
        losses = []

        def prep():
            layer.zero_grad(set_to_none=True)
            out, (_, alpha) = layer(x, bt.edge_index, ea, return_attention_weights=True, topology=topo)
            # the two dot products are formed here, outside the timed window; backward() then runs their (tiny) gradients
            loss = (out * dout).sum()
            losses[:] = [loss + (alpha * G).sum() if with_g else loss]

        def run():
            losses[0].backward()
        return prep, run

    arms = {"alpha unused": bwd(False), "<alpha, G> in loss": bwd(True)}
    samples = {k: [] for k in arms}
    for it in range(args.reps + 3):
        for name, (prep, run) in arms.items():
            prep()
            torch.cuda.synchronize()
            t = timed(run, 1)[0]
            if it >= 3:                                   # first rounds: warm-up
                samples[name].append(t)
    med = {k: statistics.median(v) for k, v in samples.items()}
    lines.append("layer backward (ms, including the eager gradients of the two dot products):")
    for k, v in samples.items():
        lines.append(f"  {k:<20} {med[k]:.3f}  [{min(v):.3f}, {max(v):.3f}]")
    lines.append(f"  added by the G term  {med['<alpha, G> in loss'] - med['alpha unused']:.3f}")

    # ---- 2. the scatter alone
    lib = sv.load_library()
    desc = GatDesc(B, N, FIN, 0, H, CC, R, 0, 0.2, lib.spotv2_gat_ldp(H, CC), 0, 0)
    d_tile = torch.empty(B, H, N, N, device=dev)
    st = torch.cuda.current_stream().cuda_stream

    def scatter():
        _lib.check(lib.spotv2_alpha_to_pyg_grad(C.byref(desc), _lib.ptr(G), _lib.ptr(topo.table), _lib.ptr(d_tile), st),
                   "alpha_to_pyg_grad")
    for _ in range(5):
        scatter()
    t_med, t_min, t_max = timed(scatter, args.reps)
    rd, wr = G.numel() * 4 + R * 4, d_tile.numel() * 4
    gbs = (wr + rd) / (t_med * 1e-3) / 1e9
    lines.append("spotv2_alpha_to_pyg_grad alone:")
    lines.append(f"  time (ms)            {t_med:.3f}  [{t_min:.3f}, {t_max:.3f}]")
    lines.append(f"  bytes                {rd / 1e6:.1f} MB read + {wr / 1e6:.1f} MB written (from shapes)")
    lines.append(f"  rate                 {gbs:.0f} GB/s = {gbs / HBM_COPY_PEAK:.2f} of the {HBM_COPY_PEAK:.0f} GB/s copy peak")
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
