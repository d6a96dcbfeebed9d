"""``GATModel`` — the SpotV2Net model with the reference's constructor and ``forward(data)``
(/root/reference/utils/models.py:61-152), built on the B200 :class:`GATConv`.

Attribute and state-dict names match the reference (``gat_layers.<i>.*``, ``linear.*``,
optional ``bnorm_node`` / ``bnorm_edge``), so ``load_state_dict`` of weights saved by
5_train_SpotV2Net.py:195 works (6_results.ipynb:318).
"""
from __future__ import annotations

import sys
from typing import Sequence

import torch
import torch.distributed as dist
import torch.nn.functional as F
from torch import nn

from ._lib import SpotV2Error
from .gat_conv import GATConv, topology_from_edge_index


def gat_layer_plan(num_node_features: int, num_heads: int, dim_hidden_layers: Sequence[int], concat_heads: bool):
    """(in_channels, out_channels, concat) per layer — the rules of utils/models.py:86-113:
    a single hidden layer never concatenates; otherwise every layer but the last follows
    ``concat_heads`` and the last always averages the heads."""
    dims = list(dim_hidden_layers)
    if len(dims) == 1:
        return [(num_node_features, dims[0], False)]
    wide = bool(concat_heads) and num_heads > 1
    plan = [(num_node_features, dims[0], bool(concat_heads))]
    for i in range(1, len(dims)):
        plan.append((dims[i - 1] * num_heads if wide else dims[i - 1], dims[i],
                     False if i == len(dims) - 1 else bool(concat_heads)))
    return plan


class GATModel(nn.Module):
    def __init__(self, num_node_features, num_edge_features, num_heads, output_node_channels,
                 dim_hidden_layers=[100], dropout_att=0.0, dropout=0.0, activation='relu',
                 concat_heads=False, negative_slope=0.2, standardize=False):
        super().__init__()
        self.dropout = dropout
        self.activation = activation
        # 6_results.ipynb's analysis variant of this class calls every layer with return_attention_weights=True and keeps
        # the result in self.attention_weights; set collect_attention = True for the same behaviour.  Under autograd (training,
        # no torch.no_grad) each alpha is differentiable, so a loss may penalise or supervise the coefficients; each layer's
        # [B, H, N, N] attention tile (88 MB at the default geometry with B = 4096) then stays alive as long as the graph
        # holds that alpha.  spotv2net_b200.attention_weights runs under no_grad and keeps nothing.
        self.collect_attention = False
        self.attention_weights = []
        self.standardize = standardize
        if self.standardize:
            self.bnorm_node = nn.BatchNorm1d(num_node_features, affine=False)
            self.bnorm_edge = nn.BatchNorm1d(num_edge_features, affine=False)
        self.gat_layers = nn.ModuleList(
            GATConv(in_channels=fi, out_channels=fo, heads=num_heads, concat=cc, dropout=dropout_att,
                    edge_dim=num_edge_features, negative_slope=negative_slope)
            for fi, fo, cc in gat_layer_plan(num_node_features, num_heads, dim_hidden_layers, concat_heads))
        self.linear = nn.Linear(list(dim_hidden_layers)[-1], output_node_channels)
        if self.activation == 'relu':
            self.a = F.relu
        elif self.activation == 'tanh':
            self.a = torch.tanh
        elif self.activation == 'sigmoid':
            self.a = torch.sigmoid
        else:
            print('Choose an available activation function')
            sys.exit()

    def set_precision(self, precision: str):
        """"fp32" (default, 1e-5 parity) or "half" (every layer's half-precision class: one fp16 tensor-core product in the
        projections and, where a layer takes the pair format, P, alpha, dout and dP as single fp16 planes; see GATConv)."""
        for layer in self.gat_layers:
            layer.precision = precision
        return self

    def _standardize(self, data, x, edge_attr, win):
        """``bnorm_node(x)`` / ``bnorm_edge(edge_attr)`` of the reference (BatchNorm1d(affine=False), utils/models.py:80-82,
        142-144) without a pass that rewrites the 1.8 GB of edge features: the statistics come from the batch (training) or
        from the running buffers (eval), x is normalised by one fused elementwise pass, and the edge normalisation is handed
        to the layers as a per-feature (mean, scale) pair - the scale rides on the folded edge vector v, the mean becomes a
        per-head constant -<mean, v'> on every logit of the head, inside the LeakyReLU (the backward corrects dv for it).  For batches of a
        WindowDataset the edge statistics are formed from per-matrix sums of the [T, N, N] stack (no pass over edges at all).
        Under torch.distributed the batch statistics are all-reduced (2 (F + Fe) + 2 numbers): every rank normalises with
        the statistics of the GLOBAL batch, as a single process would."""
        bn_x, bn_e = self.bnorm_node, self.bnorm_edge
        if self.training:
            nx = float(x.shape[0])
            sx, qx = x.sum(0, dtype=torch.float64), (x * x).sum(0, dtype=torch.float64)
            src = win if (win is not None and win.mat_stats is not None) else None
            if edge_attr is not None:
                tag = getattr(edge_attr, "_spot_stats_src", None)      # attached by WindowDataset.collate to this very tensor
                src = tag[0] if (tag is not None and tag[1] == edge_attr._version) else None
                # the statistics are functions of edge_attr: when it wants a gradient they are formed from edge_attr itself
                # (the window-stack shortcut has the same value but no autograd graph back to the edge rows)
                if edge_attr.requires_grad:
                    src = None
            if src is not None:
                se, qe, ne = src.edge_stats()                          # [Fe] float64 sums over the batch's real edges
            else:
                if edge_attr is None:
                    raise ValueError("standardize=True needs edge_attr or a WindowDataset batch")
                ne = float(edge_attr.shape[0])
                if edge_attr.requires_grad:          # squares in fp64 as well: the shortcut's accuracy, and its gradient
                    e64 = edge_attr.double()
                    se, qe = e64.sum(0), (e64 * e64).sum(0)
                else:
                    se, qe = edge_attr.sum(0, dtype=torch.float64), (edge_attr * edge_attr).sum(0, dtype=torch.float64)
            if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
                if edge_attr is not None and edge_attr.requires_grad:
                    raise SpotV2Error("standardize=True in training mode with edge_attr.requires_grad under torch.distributed: "
                                      "the all-reduce of the batch statistics is not differentiable")
                buf = torch.cat([sx, qx, se, qe, torch.tensor([nx, ne], device=x.device, dtype=torch.float64)])
                dist.all_reduce(buf)
                F_, Fe_ = sx.numel(), se.numel()
                sx, qx, se, qe = buf[:F_], buf[F_:2 * F_], buf[2 * F_:2 * F_ + Fe_], buf[2 * F_ + Fe_:2 * F_ + 2 * Fe_]
                nx, ne = buf[-2].item(), buf[-1].item()
            mx, me = sx / nx, se / ne
            vx, ve = (qx / nx - mx * mx).clamp_min(0.0), (qe / ne - me * me).clamp_min(0.0)
            with torch.no_grad():                                      # running statistics, as nn.BatchNorm1d keeps them
                for bn, m, v, n in ((bn_x, mx, vx, nx), (bn_e, me, ve, ne)):
                    mom = bn.momentum if bn.momentum is not None else 1.0 / float(bn.num_batches_tracked + 1)
                    bn.running_mean.mul_(1 - mom).add_(mom * m.to(bn.running_mean.dtype))
                    bn.running_var.mul_(1 - mom).add_(mom * (v * (n / max(n - 1.0, 1.0))).to(bn.running_var.dtype))
                    bn.num_batches_tracked += 1
        else:
            mx, vx, me, ve = bn_x.running_mean.double(), bn_x.running_var.double(), bn_e.running_mean.double(), bn_e.running_var.double()
        rx, re = torch.rsqrt(vx + bn_x.eps).float(), torch.rsqrt(ve + bn_e.eps).float()
        x = (x - mx.float()) * rx
        return x, me.float().contiguous(), re.contiguous()

    def forward(self, data):
        x, edge_index, edge_attr = data.x, data.edge_index, data.edge_attr
        # A materialised edge_attr always wins over window references: the caller may have edited it (train() scales it by
        # scale_up, 5_train_SpotV2Net.py:145-147), and the windows would silently ignore that.
        win = None if edge_attr is not None else getattr(data, "spot_windows", None)
        e_mean = e_scale = None
        if self.standardize:
            x, e_mean, e_scale = self._standardize(data, x, edge_attr, win)
        # one topology check per batch, shared by all layers (a batch produced by
        # spotv2net_b200.data carries it already)
        topo = getattr(data, "spot_topology", None)
        if topo is None:
            topo = topology_from_edge_index(edge_index, x.shape[0], getattr(data, "nodes_per_graph", None))
        if self.collect_attention:
            self.attention_weights = []
        for layer in self.gat_layers:
            if self.collect_attention:
                x, att = layer(x, edge_index, edge_attr, return_attention_weights=True, topology=topo, windows=win,
                               edge_scale=e_scale, edge_mean=e_mean)
                self.attention_weights.append(att)
            else:
                x = layer(x, edge_index, edge_attr, topology=topo, windows=win, edge_scale=e_scale, edge_mean=e_mean)
            x = self.a(x)
            if self.dropout:
                x = F.dropout(x, p=self.dropout, training=self.training)
        x = self.linear(x)
        return x.view(-1)
