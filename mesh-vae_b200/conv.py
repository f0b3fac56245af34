"""Drop-in graph-convolution modules backed by the sm_100a kernels.

* `ChebConv_batch`  - same constructor, attributes, static `norm` and `forward` signature as the
  reference class (nn/conv.py:532-581); parameters `weight [K,Fin,Fout]`, `bias [Fout]` keep the
  reference's state-dict names and N(0, 0.1) init (nn/conv.py:536-538, utils.py:34-36).
* `ChebConv`        - the torch-geometric 2.0.4 class used by models/cheb_cls.py:18,76,95
  (`lins.{k}.weight [Fout,Fin]` glorot, `bias` zeros, node_dim=-2, lambda_max=2 'sym').

Module I/O is logically [B, N, F]; physically the returned tensor is a permuted view of a
vertex-major [N, B, F] buffer, so chains of these modules (and F.relu between them, which
preserves strides) never transpose."""
import math
from typing import Optional

import torch
from torch.nn import Parameter

from . import functional as Fn
from . import operators


class ChebConv_batch(torch.nn.Module):
    def __init__(self, in_channels, out_channels, K, normalization=None, bias=True):
        super().__init__()
        assert K > 0
        assert normalization in [None, "sym", "rw"], "Invalid normalization"
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.normalization = normalization
        self.weight = Parameter(torch.empty(K, in_channels, out_channels))
        if bias:
            self.bias = Parameter(torch.empty(out_channels))
        else:
            self.register_parameter("bias", None)
        # set by accelerate()/the model mirror when the caller applies F.relu right after (then
        # idempotent): fuses the activation into the contraction epilogue
        self.fuse_relu = False
        self.reset_parameters()

    def reset_parameters(self):
        torch.nn.init.normal_(self.weight, mean=0, std=0.1)
        if self.bias is not None:
            torch.nn.init.normal_(self.bias, mean=0, std=0.1)

    @staticmethod
    def norm(edge_index, num_nodes, edge_weight=None, dtype=None):
        """(edge_index, norm) with norm_e = -deg^-1/2[row] w_e deg^-1/2[col], self loops removed,
        inf -> 0  (nn/conv.py:541-555).  Init-time host/torch arithmetic, not a hot path."""
        keep = edge_index[0] != edge_index[1]
        edge_index = edge_index[:, keep]
        if edge_weight is None:
            edge_weight = torch.ones((edge_index.size(1),), dtype=dtype, device=edge_index.device)
        else:
            edge_weight = edge_weight[keep]
        return edge_index, _sym_norm_values(edge_index, num_nodes, edge_weight)

    def forward(self, x, edge_index, norm, edge_weight=None):
        """a `norm` that requires grad (computed from learned edge weights) receives its gradient, as in the reference"""
        op, vals = operators.edge_operator(edge_index, norm, x.size(1), x.device)
        y = Fn.cheb_conv(Fn.to_vertex_major(x), self.weight, self.bias, op, self.fuse_relu, norm=vals)
        return Fn.from_vertex_major(y)

    def __repr__(self):
        return "{}({}, {}, K={}, normalization={})".format(self.__class__.__name__, self.in_channels,
                                                           self.out_channels, self.weight.size(0), self.normalization)


class ChebConv(torch.nn.Module):
    """PyG-compatible ChebConv (parity with the third-party class is 'unpinned', see DESIGN.md)."""

    def __init__(self, in_channels, out_channels, K, normalization="sym", bias=True, **kwargs):
        super().__init__()
        assert K > 0
        assert normalization in [None, "sym", "rw"], "Invalid normalization"
        self.in_channels, self.out_channels, self.normalization = in_channels, out_channels, normalization
        self.lins = torch.nn.ModuleList([torch.nn.Linear(in_channels, out_channels, bias=False) for _ in range(K)])
        if bias:
            self.bias = Parameter(torch.empty(out_channels))
        else:
            self.register_parameter("bias", None)
        self.fuse_relu = False
        self.reset_parameters()

    def reset_parameters(self):
        for lin in self.lins:
            a = math.sqrt(6.0 / (lin.weight.size(0) + lin.weight.size(1)))
            torch.nn.init.uniform_(lin.weight, -a, a)
        if self.bias is not None:
            torch.nn.init.zeros_(self.bias)

    def forward(self, x, edge_index, edge_weight: Optional[torch.Tensor] = None, batch=None, lambda_max=None):
        if self.normalization != "sym":
            raise NotImplementedError("only the 'sym' normalisation of models/cheb_cls.py:76 is implemented")
        if batch is not None or (lambda_max is not None and float(lambda_max) != 2.0):
            raise NotImplementedError("ChebConv is only implemented without `batch` and with lambda_max = 2")
        squeeze = x.dim() == 2
        if squeeze:
            x = x.unsqueeze(0)
        n = x.size(-2)
        vals = None
        if edge_weight is None:
            op = self.mesh_operator(edge_index, n, x.device, x.dtype)
        else:
            # the values change with the weights (and carry their gradient): the cached pattern of the self-loop-free
            # edges, their values computed by differentiable torch ops (an index gather: no host synchronisation)
            ei, kept = self._edges(edge_index, n)
            vals = _sym_norm_values(ei, n, edge_weight[kept]).to(device=x.device, dtype=torch.float32)
            op = operators.pattern_from_edges(ei, n, x.device)
        y = Fn.cheb_conv(Fn.to_vertex_major(x), self.stacked_weight(), self.bias, op, self.fuse_relu, norm=vals)
        y = Fn.from_vertex_major(y)
        return y.squeeze(0) if squeeze else y

    @staticmethod
    def _edges(edge_index, n):
        """(edge_index without self loops, positions of the kept edges), cached per index tensor"""
        key = ("pyg_edges", edge_index.data_ptr(), edge_index._version, int(edge_index.shape[1]), n)
        cached = _PYG_NORM.get(key)
        if cached is None:
            kept = (edge_index[0] != edge_index[1]).nonzero().squeeze(1)
            cached = _PYG_NORM[key] = (edge_index[:, kept], kept, edge_index)
        return cached[0], cached[1]

    def mesh_operator(self, edge_index, n, device, dtype=torch.float32):
        """L_hat = 2 L_sym / lambda_max - I = -D^-1/2 A D^-1/2 (PyG's explicit +1/-1 diagonal cancels), cached"""
        key = ("pyg_norm", edge_index.data_ptr(), edge_index._version, int(edge_index.shape[1]), n)
        cached = _PYG_NORM.get(key)
        if cached is None:
            cached = _PYG_NORM[key] = ChebConv_batch.norm(edge_index, n, None, dtype) + (edge_index,)
        return operators.from_edges(cached[0], cached[1], n, device)

    def stacked_weight(self):
        """[K, Fin, Fout] with W_k = lins[k].weight^T (differentiable view of the K Linear weights)"""
        return torch.stack([lin.weight.t() for lin in self.lins], dim=0)

    def __repr__(self):
        return "{}({}, {}, K={}, normalization={})".format(self.__class__.__name__, self.in_channels,
                                                           self.out_channels, len(self.lins), self.normalization)


_PYG_NORM = {}


def _sym_norm_values(edge_index, num_nodes, edge_weight):
    """-deg^-1/2[row] w_e deg^-1/2[col] over self-loop-free edges, deg summed over the row index, inf -> 0
    (nn/conv.py:548-555): plain torch ops, differentiable with respect to edge_weight"""
    row, col = edge_index[0], edge_index[1]
    deg = torch.zeros(num_nodes, dtype=edge_weight.dtype, device=edge_index.device).scatter_add_(0, row, edge_weight)
    dis = deg.pow(-0.5)
    dis[dis == float("inf")] = 0
    return -dis[row] * edge_weight * dis[col]
