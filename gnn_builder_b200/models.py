"""Model description API -- the host-side mirror of ``gnnbuilder/models.py``.

Same class names, constructor arguments, attribute names and parameter names as the
reference (models.py:30-44 GCNConv_GNNB, 70-94 GINConv_GNNB, 209-240 PNAConv_GNNB, 243-262
SAGEConv_GNNB, 326-359 GlobalPooling, 365-450 MLP, 462-634 GNNModel) so that a trained
``state_dict`` and user code written against the reference drop in unchanged.  The reference
wraps PyTorch-Geometric convs; PyG is not a dependency here, so each ``*_GNNB.conv`` is a small
``nn.Module`` that carries PyG's parameter names/shapes (SURVEY appendix B) and a plain-torch
fp32 ``forward`` with PyG's semantics.  That torch forward plays the role it plays in the
reference -- the *golden* model (code_gen.py:279-285) -- and is never used by the CUDA engine.

``p_in/p_out/p_hidden`` (HLS unroll factors) are accepted and stored; on the GPU they are
ignored (they only change the rounding order of the reference's ``linear``, lib:808-905).
"""
from __future__ import annotations

import math
from typing import Callable, Optional

import torch
import torch.nn as nn
from torch import Tensor

TorchModuleArg = Callable[..., torch.nn.Module]
TorchModuleArgOptional = Optional[Callable[..., torch.nn.Module]]


def layer_param_name_combiner(layer_name: str, param_name: str) -> str:
    """utils.py:99-100"""
    return f"{layer_name}_{param_name.replace('.', '_')}"


# ----------------------------------------------------------------------------- torch helpers

def _in_degree(edge_index: Tensor, n: int) -> Tensor:
    return torch.zeros(n, dtype=torch.float32).index_add_(
        0, edge_index[1], torch.ones(edge_index.shape[1], dtype=torch.float32))


def _scatter_sum(src: Tensor, index: Tensor, n: int) -> Tensor:
    return torch.zeros(n, src.shape[1], dtype=src.dtype).index_add_(0, index, src)


def _scatter_minmax(src: Tensor, index: Tensor, n: int, reduce: str) -> Tensor:
    out = torch.zeros(n, src.shape[1], dtype=src.dtype)
    idx = index.view(-1, 1).expand(-1, src.shape[1])
    return out.scatter_reduce(0, idx, src, reduce=reduce, include_self=False)


# ----------------------------------------------------------------------------- conv holders

class _GCNConv(nn.Module):
    """PyG GCNConv parameters: ``bias`` then ``lin.weight`` (bias listed first)."""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        self.bias = nn.Parameter(torch.zeros(out_channels))
        self.lin = nn.Linear(in_channels, out_channels, bias=False)
        nn.init.uniform_(self.bias, -0.1, 0.1)

    def forward(self, x: Tensor, edge_index: Tensor) -> Tensor:
        n = x.shape[0]
        src, dst = edge_index[0], edge_index[1]
        dinv = (_in_degree(edge_index, n) + 1.0).pow(-0.5)
        h = self.lin(x)
        out = _scatter_sum(h[src] * (dinv[src] * dinv[dst]).view(-1, 1), dst, n)
        out = out + h * (dinv * dinv).view(-1, 1)
        return out + self.bias


class _GINConv(nn.Module):
    def __init__(self, mlp: nn.Module, eps: float = 0.0, train_eps: bool = False):
        super().__init__()
        self.nn = mlp
        self.register_buffer("eps", torch.tensor([float(eps)]))

    def forward(self, x: Tensor, edge_index: Tensor) -> Tensor:
        agg = _scatter_sum(x[edge_index[0]], edge_index[1], x.shape[0])
        return self.nn(agg + (1.0 + self.eps) * x)


class _GINEConv(nn.Module):
    """PyG GINEConv with ``edge_dim``: ``lin`` projects the edge features to ``in_channels``."""

    def __init__(self, mlp: nn.Module, eps: float = 0.0, edge_dim: int = 1, in_channels: int = 1):
        super().__init__()
        self.nn = mlp
        self.register_buffer("eps", torch.tensor([float(eps)]))
        self.lin = nn.Linear(edge_dim, in_channels)

    def forward(self, x: Tensor, edge_index: Tensor, edge_attr: Tensor) -> Tensor:
        msg = (x[edge_index[0]] + self.lin(edge_attr)).relu()
        agg = _scatter_sum(msg, edge_index[1], x.shape[0])
        return self.nn(agg + (1.0 + self.eps) * x)


class _GATConv(nn.Module):
    """PyG GATConv with an int ``in_channels``, concatenated heads and self loops, for inference.
    Its own parameters come first in the flat order: ``att_src`` and ``att_dst`` [1][H][C], with
    ``edge_dim`` ``att_edge`` [1][H][C], ``bias`` [H*C], then ``lin.weight`` [H*C][in] (no bias in
    ``lin``) and with ``edge_dim`` ``lin_edge.weight`` [H*C][edge_dim] -- PyG's registration order.
    With edge features each self loop's attribute is the mean of the node's other in-edge
    attributes (PyG's ``fill_value="mean"``), the zero vector for a node without one."""

    def __init__(self, in_channels: int, out_channels: int, heads: int, negative_slope: float,
                 edge_dim: Optional[int] = None):
        super().__init__()
        self.heads = heads
        self.head_channels = out_channels // heads
        self.negative_slope = negative_slope
        self.edge_dim = edge_dim
        self.lin = nn.Linear(in_channels, out_channels, bias=False)
        self.att_src = nn.Parameter(torch.empty(1, heads, self.head_channels))
        self.att_dst = nn.Parameter(torch.empty(1, heads, self.head_channels))
        if edge_dim is not None:
            self.lin_edge = nn.Linear(edge_dim, out_channels, bias=False)
            self.att_edge = nn.Parameter(torch.empty(1, heads, self.head_channels))
            nn.init.xavier_uniform_(self.att_edge)
        self.bias = nn.Parameter(torch.zeros(out_channels))
        nn.init.xavier_uniform_(self.att_src)
        nn.init.xavier_uniform_(self.att_dst)
        nn.init.uniform_(self.bias, -0.1, 0.1)

    def forward(self, x: Tensor, edge_index: Tensor, edge_attr: Optional[Tensor] = None) -> Tensor:
        n, H, C = x.shape[0], self.heads, self.head_channels
        # every self loop of the input is replaced by exactly one per node; duplicates stay
        keep = edge_index[0] != edge_index[1]
        loops = torch.arange(n, dtype=edge_index.dtype)
        src = torch.cat([edge_index[0][keep], loops])
        dst = torch.cat([edge_index[1][keep], loops])
        h = self.lin(x).view(n, H, C)
        a_src = (h * self.att_src).sum(-1)
        a_dst = (h * self.att_dst).sum(-1)
        logit = a_src[src] + a_dst[dst]
        if self.edge_dim is not None:
            ea = edge_attr.reshape(-1, self.edge_dim)[keep]
            cnt = _in_degree(edge_index[:, keep], n).clamp(min=1.0).view(-1, 1)
            ea = torch.cat([ea, _scatter_sum(ea, edge_index[1][keep], n) / cnt])
            logit = logit + (self.lin_edge(ea).view(-1, H, C) * self.att_edge).sum(-1)
        e = torch.nn.functional.leaky_relu(logit, self.negative_slope)
        p = (e - _scatter_minmax(e, dst, n, "amax")[dst]).exp()
        alpha = p / _scatter_sum(p, dst, n)[dst]
        msg = (h[src] * alpha.unsqueeze(-1)).reshape(-1, H * C)
        return _scatter_sum(msg, dst, n) + self.bias


class _GATv2Conv(nn.Module):
    """PyG GATv2Conv with an int ``in_channels``, concatenated heads, self loops and
    ``share_weights=False``, for inference.  Its own parameters come first in the flat order:
    ``att`` [1][H][C], ``bias`` [H*C], then ``lin_l`` and ``lin_r`` (weight [H*C][in] and bias each)
    and with ``edge_dim`` ``lin_edge.weight`` [H*C][edge_dim] (no bias) -- PyG's order.  With edge
    features each self loop's attribute is the mean of the node's other in-edge attributes (PyG's
    ``fill_value="mean"``), the zero vector for a node without one."""

    def __init__(self, in_channels: int, out_channels: int, heads: int, negative_slope: float,
                 edge_dim: Optional[int] = None):
        super().__init__()
        self.heads = heads
        self.head_channels = out_channels // heads
        self.negative_slope = negative_slope
        self.edge_dim = edge_dim
        self.att = nn.Parameter(torch.empty(1, heads, self.head_channels))
        self.bias = nn.Parameter(torch.zeros(out_channels))
        self.lin_l = nn.Linear(in_channels, out_channels, bias=True)
        self.lin_r = nn.Linear(in_channels, out_channels, bias=True)
        if edge_dim is not None:
            self.lin_edge = nn.Linear(edge_dim, out_channels, bias=False)
        nn.init.xavier_uniform_(self.att)
        nn.init.uniform_(self.bias, -0.1, 0.1)
        nn.init.uniform_(self.lin_l.bias, -0.1, 0.1)
        nn.init.uniform_(self.lin_r.bias, -0.1, 0.1)

    def forward(self, x: Tensor, edge_index: Tensor, edge_attr: Optional[Tensor] = None) -> Tensor:
        n, H, C = x.shape[0], self.heads, self.head_channels
        # every self loop of the input is replaced by exactly one per node; duplicates stay
        keep = edge_index[0] != edge_index[1]
        loops = torch.arange(n, dtype=edge_index.dtype)
        src = torch.cat([edge_index[0][keep], loops])
        dst = torch.cat([edge_index[1][keep], loops])
        xl = self.lin_l(x).view(n, H, C)
        xr = self.lin_r(x).view(n, H, C)
        z = xl[src] + xr[dst]
        if self.edge_dim is not None:
            ea = edge_attr.reshape(-1, self.edge_dim)[keep]
            cnt = _in_degree(edge_index[:, keep], n).clamp(min=1.0).view(-1, 1)
            ea = torch.cat([ea, _scatter_sum(ea, edge_index[1][keep], n) / cnt])
            z = z + self.lin_edge(ea).view(-1, H, C)
        e = (torch.nn.functional.leaky_relu(z, self.negative_slope) * self.att).sum(-1)
        p = (e - _scatter_minmax(e, dst, n, "amax")[dst]).exp()
        alpha = p / _scatter_sum(p, dst, n)[dst]
        msg = (xl[src] * alpha.unsqueeze(-1)).reshape(-1, H * C)
        return _scatter_sum(msg, dst, n) + self.bias


class _TransformerConv(nn.Module):
    """PyG TransformerConv with an int ``in_channels``, concatenated heads, ``beta=False`` and
    ``root_weight=True``, for inference.  Parameters in PyG's order: ``lin_key``, ``lin_query``,
    ``lin_value`` (weight [H*C][in] and bias each), with ``edge_dim`` ``lin_edge.weight``
    [H*C][edge_dim] (no bias), then ``lin_skip`` (weight and bias).  No self loops are added: the
    input's self loops and duplicate edges are ordinary edges, and a node without in-edges gets
    ``lin_skip(x)`` alone."""

    def __init__(self, in_channels: int, out_channels: int, heads: int,
                 edge_dim: Optional[int] = None):
        super().__init__()
        self.heads = heads
        self.head_channels = out_channels // heads
        self.edge_dim = edge_dim
        self.lin_key = nn.Linear(in_channels, out_channels, bias=True)
        self.lin_query = nn.Linear(in_channels, out_channels, bias=True)
        self.lin_value = nn.Linear(in_channels, out_channels, bias=True)
        if edge_dim is not None:
            self.lin_edge = nn.Linear(edge_dim, out_channels, bias=False)
        self.lin_skip = nn.Linear(in_channels, out_channels, bias=True)

    def forward(self, x: Tensor, edge_index: Tensor, edge_attr: Optional[Tensor] = None) -> Tensor:
        n, H, C = x.shape[0], self.heads, self.head_channels
        src, dst = edge_index[0], edge_index[1]
        q = self.lin_query(x).view(n, H, C)
        k = self.lin_key(x)[src].view(-1, H, C)
        v = self.lin_value(x)[src].view(-1, H, C)
        if self.edge_dim is not None:
            e = self.lin_edge(edge_attr.reshape(-1, self.edge_dim)).view(-1, H, C)
            k = k + e
            v = v + e
        logit = (q[dst] * k).sum(-1) / math.sqrt(C)
        p = (logit - _scatter_minmax(logit, dst, n, "amax")[dst]).exp()
        alpha = p / _scatter_sum(p, dst, n)[dst]
        msg = (v * alpha.unsqueeze(-1)).reshape(-1, H * C)
        return _scatter_sum(msg, dst, n) + self.lin_skip(x)


class _SAGEConv(nn.Module):
    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        self.lin_l = nn.Linear(in_channels, out_channels, bias=True)
        self.lin_r = nn.Linear(in_channels, out_channels, bias=False)

    def forward(self, x: Tensor, edge_index: Tensor) -> Tensor:
        n = x.shape[0]
        s = _scatter_sum(x[edge_index[0]], edge_index[1], n)
        mean = s / _in_degree(edge_index, n).clamp(min=1.0).view(-1, 1)
        return self.lin_l(mean) + self.lin_r(x)


class _AggrModule(nn.Module):
    def __init__(self):
        super().__init__()
        self.avg_deg_log = torch.Tensor([1.0])


class _PNAConv(nn.Module):
    """PyG PNAConv with towers=1, pre_layers=post_layers=1, aggregators [max,min,mean,std],
    scalers [identity, amplification, attenuation]."""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        F = in_channels
        self.aggr_module = _AggrModule()
        self.pre_nns = nn.ModuleList([nn.Sequential(nn.Linear(2 * F, F))])
        self.post_nns = nn.ModuleList([nn.Sequential(nn.Linear(13 * F, out_channels))])
        self.lin = nn.Linear(out_channels, out_channels)

    def forward(self, x: Tensor, edge_index: Tensor) -> Tensor:
        n = x.shape[0]
        src, dst = edge_index[0], edge_index[1]
        h = self.pre_nns[0](torch.cat([x[dst], x[src]], dim=-1))
        deg = _in_degree(edge_index, n)
        degc = deg.clamp(min=1.0).view(-1, 1)
        mean = _scatter_sum(h, dst, n) / degc
        mean2 = _scatter_sum(h * h, dst, n) / degc
        std = ((mean2 - mean * mean).relu() + 1e-5).sqrt()
        agg = torch.cat([_scatter_minmax(h, dst, n, "amax"), _scatter_minmax(h, dst, n, "amin"),
                         mean, std], dim=-1)
        delta = float(self.aggr_module.avg_deg_log.item())
        amp = torch.log(degc + 1.0) / delta
        att = delta / torch.log(degc + 1.0)
        out = torch.cat([x, agg, agg * amp, agg * att], dim=-1)
        return self.lin(self.post_nns[0](out))


# ----------------------------------------------------------------------------- *_GNNB wrappers

class GCNConv_GNNB(nn.Module):
    """models.py:30-44"""

    def __init__(self, in_channels: int, out_channels: int, p_in: int = 1, p_out: int = 1):
        super().__init__()
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.p_in = p_in
        self.p_out = p_out
        self.conv = _GCNConv(in_channels, out_channels)

    def forward(self, x: Tensor, edge_index: Tensor) -> Tensor:
        return self.conv(x, edge_index)


class GIN_MLP(nn.Module):
    """models.py:47-67"""

    def __init__(self, in_dim: int, out_dim: int, hidden_dim: Optional[int] = None):
        super().__init__()
        self.in_dim = in_dim
        self.out_dim = out_dim
        self.hidden_dim = out_dim if hidden_dim is None else hidden_dim
        self.linear_0 = nn.Linear(self.in_dim, self.hidden_dim)
        self.linear_1 = nn.Linear(self.hidden_dim, self.out_dim)
        self.relu = nn.ReLU()
        self.in_features = self.in_dim

    def forward(self, x):
        return self.linear_1(self.relu(self.linear_0(x)))


class GINConv_GNNB(nn.Module):
    """models.py:70-94.  As in the reference the MLP is always built with hidden = out_channels
    (``GIN_MLP(in, out, None)``, models.py:90) whatever ``hidden_dim`` says."""

    def __init__(self, in_channels: int, out_channels: int, hidden_dim: Optional[int] = None,
                 eps: float = 0.0, p_in: int = 1, p_out: int = 1):
        super().__init__()
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.hidden_dim = hidden_dim
        self.eps = eps
        self.p_in = p_in
        self.p_out = p_out
        self.mlp = GIN_MLP(in_channels, out_channels, None)
        self.conv = _GINConv(self.mlp, eps=eps, train_eps=False)

    def forward(self, x: Tensor, edge_index: Tensor) -> Tensor:
        return self.conv(x, edge_index)


class GINEConv_GNNB(nn.Module):
    """GIN with edge features (PyG ``GINEConv`` with ``edge_dim``; the reference lib's gine_conv,
    lib:1555-1742): y_v = MLP((1 + eps) x_v + sum_{u->v} ReLU(x_u + e_uv W_e^T + b_e)).  Built like
    ``GINConv_GNNB``; each layer has its own edge linear ``conv.lin`` [in_channels][edge_dim] over
    the same raw edge features."""

    def __init__(self, in_channels: int, out_channels: int, edge_dim: int,
                 hidden_dim: Optional[int] = None, eps: float = 0.0, p_in: int = 1, p_out: int = 1):
        super().__init__()
        if not isinstance(edge_dim, int) or isinstance(edge_dim, bool) or edge_dim < 1:
            raise ValueError(f"edge_dim must be a positive int, got {edge_dim!r}")
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.edge_dim = edge_dim
        self.hidden_dim = hidden_dim
        self.eps = eps
        self.p_in = p_in
        self.p_out = p_out
        self.mlp = GIN_MLP(in_channels, out_channels, None)
        self.conv = _GINEConv(self.mlp, eps=eps, edge_dim=edge_dim, in_channels=in_channels)

    def forward(self, x: Tensor, edge_index: Tensor, edge_attr: Tensor) -> Tensor:
        return self.conv(x, edge_index, edge_attr)


class GATConv_GNNB(nn.Module):
    """Graph attention (PyG ``GATConv``, inference): per head, h = x W^T, logits
    e_uv = LeakyReLU(<h_u, att_src> + <h_v, att_dst>) over the in-edges of v plus one self loop,
    y_v = sum softmax_v(e) h_u + bias, heads concatenated.  ``out_channels`` is the concatenated
    width and must be a multiple of ``heads``.  Pass ``heads`` with ``functools.partial``.

    ``edge_dim`` (a positive int, also passed with ``functools.partial``) adds PyG's edge term to
    every logit: + <(e_uv W_e^T)_h, att_edge_h>, where the self loop's e_vv is the mean of v's other
    in-edge attributes.  The model's ``graph_input_edge_dim`` must then equal it."""

    def __init__(self, in_channels: int, out_channels: int, heads: int = 1,
                 negative_slope: float = 0.2, edge_dim: Optional[int] = None, p_in: int = 1,
                 p_out: int = 1):
        super().__init__()
        if not isinstance(heads, int) or isinstance(heads, bool) or heads < 1:
            raise ValueError(f"heads must be a positive int, got {heads!r}")
        if edge_dim is not None and (not isinstance(edge_dim, int) or isinstance(edge_dim, bool)
                                     or edge_dim < 1):
            raise ValueError(f"edge_dim must be None or a positive int, got {edge_dim!r}")
        if out_channels % heads != 0:
            raise ValueError(f"out_channels ({out_channels}) must be a multiple of heads ({heads})")
        if not math.isfinite(negative_slope):
            raise ValueError(f"negative_slope must be finite, got {negative_slope!r}")
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.heads = heads
        self.negative_slope = float(negative_slope)
        self.edge_dim = edge_dim
        self.p_in = p_in
        self.p_out = p_out
        self.conv = _GATConv(in_channels, out_channels, heads, self.negative_slope, edge_dim)

    def forward(self, x: Tensor, edge_index: Tensor, edge_attr: Optional[Tensor] = None) -> Tensor:
        if self.edge_dim is not None and edge_attr is None:
            raise ValueError("a GATConv_GNNB with edge_dim needs edge_attr")
        return self.conv(x, edge_index, edge_attr)


class GATv2Conv_GNNB(nn.Module):
    """Graph attention v2 (PyG ``GATv2Conv``, inference, ``share_weights=False``): per head,
    xl = x W_l^T + b_l, xr = x W_r^T + b_r, logits e_uv = <att, LeakyReLU(xl_u + xr_v)> over the
    in-edges of v plus one self loop, y_v = sum softmax_v(e) xl_u + bias, heads concatenated.
    ``out_channels`` is the concatenated width and must be a multiple of ``heads``.  Pass ``heads``
    with ``functools.partial``.

    ``edge_dim`` (a positive int, also passed with ``functools.partial``) adds ``lin_edge`` (no
    bias) inside the nonlinearity: LeakyReLU(xl_u + xr_v + e_uv W_e^T), where the self loop's e_vv
    is the mean of v's other in-edge attributes.  The model's ``graph_input_edge_dim`` must then
    equal it."""

    def __init__(self, in_channels: int, out_channels: int, heads: int = 1,
                 negative_slope: float = 0.2, edge_dim: Optional[int] = None, p_in: int = 1,
                 p_out: int = 1):
        super().__init__()
        if not isinstance(heads, int) or isinstance(heads, bool) or heads < 1:
            raise ValueError(f"heads must be a positive int, got {heads!r}")
        if edge_dim is not None and (not isinstance(edge_dim, int) or isinstance(edge_dim, bool)
                                     or edge_dim < 1):
            raise ValueError(f"edge_dim must be None or a positive int, got {edge_dim!r}")
        if out_channels % heads != 0:
            raise ValueError(f"out_channels ({out_channels}) must be a multiple of heads ({heads})")
        if not math.isfinite(negative_slope):
            raise ValueError(f"negative_slope must be finite, got {negative_slope!r}")
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.heads = heads
        self.negative_slope = float(negative_slope)
        self.edge_dim = edge_dim
        self.p_in = p_in
        self.p_out = p_out
        self.conv = _GATv2Conv(in_channels, out_channels, heads, self.negative_slope, edge_dim)

    def forward(self, x: Tensor, edge_index: Tensor, edge_attr: Optional[Tensor] = None) -> Tensor:
        if self.edge_dim is not None and edge_attr is None:
            raise ValueError("a GATv2Conv_GNNB with edge_dim needs edge_attr")
        return self.conv(x, edge_index, edge_attr)


class TransformerConv_GNNB(nn.Module):
    """Graph transformer attention (PyG ``TransformerConv``, inference): per head,
    q = x W_q^T + b_q, k = x W_k^T + b_k, v = x W_v^T + b_v, logits a_uv = <q_v, k_u> / sqrt(C) over
    the in-edges of v, y_v = sum softmax_v(a) v_u + x_v W_skip^T + b_skip, heads concatenated.  No
    self loops are added; a node without in-edges gets x_v W_skip^T + b_skip.  ``out_channels`` is
    the concatenated width and must be a multiple of ``heads``.  Pass ``heads`` with
    ``functools.partial``.

    ``edge_dim`` (a positive int, also passed with ``functools.partial``) adds ``lin_edge`` (no
    bias): e_uv W_e^T is added to both k_u and v_u.  The model's ``graph_input_edge_dim`` must then
    equal it.  PyG's ``concat=False``, ``beta=True``, ``root_weight=False``, ``bias=False``,
    ``dropout`` and bipartite ``in_channels`` are not supported."""

    def __init__(self, in_channels: int, out_channels: int, heads: int = 1,
                 edge_dim: Optional[int] = None, concat: bool = True, beta: bool = False,
                 dropout: float = 0.0, bias: bool = True, root_weight: bool = True, p_in: int = 1,
                 p_out: int = 1):
        super().__init__()
        if not isinstance(in_channels, int) or isinstance(in_channels, bool):
            raise ValueError(f"in_channels must be an int (bipartite inputs are not supported), "
                             f"got {in_channels!r}")
        if not isinstance(heads, int) or isinstance(heads, bool) or heads < 1:
            raise ValueError(f"heads must be a positive int, got {heads!r}")
        if edge_dim is not None and (not isinstance(edge_dim, int) or isinstance(edge_dim, bool)
                                     or edge_dim < 1):
            raise ValueError(f"edge_dim must be None or a positive int, got {edge_dim!r}")
        if out_channels % heads != 0:
            raise ValueError(f"out_channels ({out_channels}) must be a multiple of heads ({heads})")
        for name, value, default in (("concat", concat, True), ("beta", beta, False),
                                     ("bias", bias, True), ("root_weight", root_weight, True)):
            if value is not default:
                raise ValueError(f"TransformerConv_GNNB supports only {name}={default}, got {value!r}")
        if dropout != 0.0:
            raise ValueError(f"TransformerConv_GNNB runs inference without dropout, got {dropout!r}")
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.heads = heads
        self.edge_dim = edge_dim
        self.p_in = p_in
        self.p_out = p_out
        self.conv = _TransformerConv(in_channels, out_channels, heads, edge_dim)

    def forward(self, x: Tensor, edge_index: Tensor, edge_attr: Optional[Tensor] = None) -> Tensor:
        if self.edge_dim is not None and edge_attr is None:
            raise ValueError("a TransformerConv_GNNB with edge_dim needs edge_attr")
        return self.conv(x, edge_index, edge_attr)


class PNAConv_GNNB(nn.Module):
    """models.py:209-240"""

    def __init__(self, in_channels: int, out_channels: int, delta: float = 1.0, p_in: int = 1,
                 p_out: int = 1):
        super().__init__()
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.delta = delta
        self.p_in = p_in
        self.p_out = p_out
        self.aggregators = ["max", "min", "mean", "std"]
        self.scalers = ["identity", "amplification", "attenuation"]
        self.conv = _PNAConv(in_channels, out_channels)
        self.conv.aggr_module.avg_deg_log = torch.Tensor([self.delta])
        self.delta_scaler = self.conv.aggr_module.avg_deg_log.item()

    def forward(self, x: Tensor, edge_index: Tensor) -> Tensor:
        return self.conv(x, edge_index)


class SAGEConv_GNNB(nn.Module):
    """models.py:243-262 (mean aggregation: the only SAGE the reference implements)"""

    def __init__(self, in_channels: int, out_channels: int, p_in: int = 1, p_out: int = 1):
        super().__init__()
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.p_in = p_in
        self.p_out = p_out
        self.conv = _SAGEConv(in_channels, out_channels)

    def forward(self, x: Tensor, edge_index: Tensor) -> Tensor:
        return self.conv(x, edge_index)


SUPPORTED_GLOBAL_POOLING_AGGRS = {
    "add": "SumAggregation",
    "max": "MaxAggregation",
    "mean": "MeanAggregation",
}
SUPPORTED_GLOBAL_POOLING_MODE = ["cat"]


class GlobalPooling(nn.Module):
    """models.py:326-359"""

    def __init__(self, aggrs: list, mode: str = "cat"):
        super().__init__()
        self.aggrs = aggrs
        self.mode = mode
        if aggrs == []:
            raise ValueError("Aggregation list is empty.")
        for aggr_str in self.aggrs:
            if aggr_str not in SUPPORTED_GLOBAL_POOLING_AGGRS:
                raise NotImplementedError(
                    f"Aggregation {aggr_str} is not supported. Supported aggregations"
                    f" are {SUPPORTED_GLOBAL_POOLING_AGGRS}.")
        if self.mode not in SUPPORTED_GLOBAL_POOLING_MODE:
            raise NotImplementedError(
                f"Mode {self.mode} is not supported. Supported modes are"
                f" {SUPPORTED_GLOBAL_POOLING_MODE}.")

    def forward(self, x: Tensor, *args, **kwargs) -> Tensor:
        outs = []
        for a in self.aggrs:
            if a == "add":
                outs.append(x.sum(0, keepdim=True))
            elif a == "mean":
                outs.append(x.mean(0, keepdim=True))
            else:
                outs.append(x.max(0, keepdim=True).values)
        return torch.cat(outs, dim=-1)

    @property
    def num_of_aggrs(self) -> int:
        return len(self.aggrs)

    def __repr__(self) -> str:
        return f"{self.__class__.__name__}({self.aggrs}, mode={self.mode})"


SUPPORTED_ACTIVATIONS = [nn.ReLU, nn.GELU, nn.Sigmoid, nn.Tanh]


class MLP(nn.Module):
    """models.py:365-450"""

    def __init__(self, in_dim: int, out_dim: int, hidden_dim: int = 64, hidden_layers: int = 2,
                 activation: TorchModuleArg = nn.ReLU, norm_layer: TorchModuleArgOptional = None,
                 p_in: int = 1, p_hidden: int = 1, p_out: int = 1):
        super().__init__()
        self.in_dim = in_dim
        self.out_dim = out_dim
        self.hidden_dim = hidden_dim
        self.hidden_layers = hidden_layers
        self.activation = activation
        self.norm_layer = norm_layer
        if self.activation not in SUPPORTED_ACTIVATIONS:
            raise ValueError(f"activation {activation} not supported")
        if self.norm_layer is not None:
            raise NotImplementedError("norm not supported yet")
        if hidden_layers < 0:
            raise ValueError("hidden_layers must be >= 0")
        self.p_in = p_in
        self.p_hidden = p_hidden
        self.p_out = p_out

        self.linear_layers = nn.ModuleList()
        self.activations = nn.ModuleList()
        self.norm_layers = nn.ModuleList()
        if hidden_layers == 0:
            self.linear_layers.append(nn.Linear(self.in_dim, self.out_dim))
        else:
            for i in range(hidden_layers):
                self.linear_layers.append(
                    nn.Linear(self.in_dim if i == 0 else self.hidden_dim, self.hidden_dim))
                self.activations.append(self.activation())
            self.linear_layers.append(nn.Linear(self.hidden_dim, self.out_dim))

    def forward(self, x: Tensor) -> Tensor:
        for i, lin in enumerate(self.linear_layers):
            x = lin(x)
            if i < len(self.linear_layers) - 1:
                x = self.activations[i](x)
        return x

    @property
    def p_factors(self):
        if self.hidden_layers == 0:
            return [(self.p_in, self.p_out)]
        f = [(self.p_in, self.p_hidden)]
        f += [(self.p_hidden, self.p_hidden)] * (self.hidden_layers - 1)
        f.append((self.p_hidden, self.p_out))
        return f

    @property
    def num_of_layers(self) -> int:
        return len(self.linear_layers)


SUPPORTED_GNN_CONVS = [GCNConv_GNNB, GINConv_GNNB, PNAConv_GNNB, SAGEConv_GNNB, GINEConv_GNNB,
                       GATConv_GNNB, GATv2Conv_GNNB, TransformerConv_GNNB]

# 6 is not assigned (GNNB_CONV_GATV2 = 7, GNNB_CONV_TRANSFORMER = 8 in include/gnnb_b200.h)
CONV_TYPE_IDS = {"GCNConv_GNNB": 0, "GINConv_GNNB": 1, "SAGEConv_GNNB": 2, "PNAConv_GNNB": 3,
                 "GINEConv_GNNB": 4, "GATConv_GNNB": 5, "GATv2Conv_GNNB": 7,
                 "TransformerConv_GNNB": 8}
# the attention convs: heads, and edge features only when their partial carries edge_dim
_ATTENTION_CONVS = ("GATConv_GNNB", "GATv2Conv_GNNB", "TransformerConv_GNNB")
ACTIVATION_IDS = {None: 0, "ReLU": 1, "GELU": 2, "Sigmoid": 3, "Tanh": 4}
POOL_IDS = {"add": 0, "mean": 1, "max": 2}


class GNNModel(nn.Module):
    """models.py:462-634"""

    def __init__(self, graph_input_feature_dim: int, graph_input_edge_dim: Optional[int],
                 gnn_hidden_dim: int, gnn_num_layers: int, gnn_output_dim: int,
                 gnn_conv: TorchModuleArg, gnn_activation: TorchModuleArg,
                 gnn_skip_connection: bool, global_pooling: GlobalPooling, mlp_head: MLP,
                 output_activation: TorchModuleArgOptional, gnn_p_in: int = 1,
                 gnn_p_hidden: int = 1, gnn_p_out: int = 1) -> None:
        super().__init__()
        self.graph_input_feature_dim = graph_input_feature_dim
        self.graph_input_edge_dim = graph_input_edge_dim
        self.gnn_hidden_dim = gnn_hidden_dim
        self.gnn_num_layers = gnn_num_layers
        self.gnn_output_dim = gnn_output_dim
        self.gnn_conv = gnn_conv
        conv_cls = getattr(gnn_conv, "func", gnn_conv)  # allow functools.partial(delta=..)
        if conv_cls not in SUPPORTED_GNN_CONVS:
            raise ValueError(f"gnn_conv must be one of {SUPPORTED_GNN_CONVS}")
        self._conv_cls = conv_cls
        # the attention convs take edge features only when their partial carries edge_dim
        self._conv_kwargs = dict(getattr(gnn_conv, "keywords", None) or {})
        gat_edge_dim = (self._conv_kwargs.get("edge_dim")
                        if conv_cls.__name__ in _ATTENTION_CONVS else None)
        self.uses_edge_features = conv_cls is GINEConv_GNNB or gat_edge_dim is not None
        conv_kwargs = {}
        if conv_cls is GINEConv_GNNB:
            e = graph_input_edge_dim
            if not isinstance(e, int) or isinstance(e, bool) or e < 1:
                raise ValueError("GINEConv_GNNB needs graph_input_edge_dim to be a positive int, "
                                 f"got {e!r}")
            conv_kwargs["edge_dim"] = e
        elif gat_edge_dim is not None:
            e = graph_input_edge_dim
            for v in (gat_edge_dim, e):
                if not isinstance(v, int) or isinstance(v, bool) or v < 1 or v != gat_edge_dim:
                    raise ValueError(f"{conv_cls.__name__} with edge_dim={gat_edge_dim!r} needs a "
                                     "positive int edge_dim and graph_input_edge_dim equal to it, "
                                     f"got {e!r}")
        self.gnn_activation = gnn_activation
        if self.gnn_activation not in SUPPORTED_ACTIVATIONS:
            raise ValueError(f"gnn_activation must be one of {SUPPORTED_ACTIVATIONS}")
        self.gnn_skip_connection = gnn_skip_connection
        self.global_pooling = global_pooling
        self.mlp_head = mlp_head
        self.output_activation = output_activation
        if self.output_activation is not None:
            # The reference template only knows ReLU/GELU/Sigmoid/Tanh here and every
            # reference caller passes None (SURVEY appendix); same restriction.
            if self.output_activation not in SUPPORTED_ACTIVATIONS:
                raise ValueError(f"output_activation must be None or one of {SUPPORTED_ACTIVATIONS}")
        self.gnn_p_in = gnn_p_in
        self.gnn_p_hidden = gnn_p_hidden
        self.gnn_p_out = gnn_p_out

        self.gnn_convs = nn.ModuleList()
        self.gnn_activations = nn.ModuleList()
        if self.gnn_num_layers == 0:
            if self.graph_input_feature_dim != self.gnn_output_dim:
                raise ValueError(
                    "You specified gnn_num_layers=0, but"
                    f" (gnn_output_dim={self.gnn_output_dim}) !="
                    f" (graph_input_feature_dim={self.graph_input_feature_dim}).")
        L = self.gnn_num_layers
        for i in range(L):
            in_dim = self.graph_input_feature_dim if i == 0 else self.gnn_hidden_dim
            out_dim = self.gnn_output_dim if i == L - 1 else self.gnn_hidden_dim
            p_in = self.gnn_p_in if i == 0 else self.gnn_p_hidden
            p_out = self.gnn_p_out if i == L - 1 else self.gnn_p_hidden
            self.gnn_convs.append(self.gnn_conv(in_dim, out_dim, p_in=p_in, p_out=p_out,
                                                **conv_kwargs))
            self.gnn_activations.append(self.gnn_activation())
        if self.gnn_skip_connection:
            for i in range(1, L - 1):
                c = self.gnn_convs[i]
                if c.in_channels != c.out_channels:
                    raise ValueError("skip connections need in_channels == out_channels")

    def forward(self, x: Tensor, edge_index: Tensor, batch: Optional[Tensor] = None,
                edge_attr: Optional[Tensor] = None) -> Tensor:
        if self.uses_edge_features and self.gnn_num_layers > 0 and edge_attr is None:
            raise ValueError(f"a {self._conv_cls.__name__} model with edge features needs edge_attr")
        x_gnn = x
        for i, (conv, act) in enumerate(zip(self.gnn_convs, self.gnn_activations)):
            x_in = x_gnn
            if self.uses_edge_features:
                x_gnn = conv(x_gnn, edge_index, edge_attr)
            else:
                x_gnn = conv(x_gnn, edge_index)
            if self.gnn_skip_connection and i != 0 and i != self.gnn_num_layers - 1:
                x_gnn = x_gnn + x_in
            x_gnn = act(x_gnn)
        out = self.mlp_head(self.global_pooling(x_gnn))
        if self.output_activation is not None:
            out = self.output_activation()(out)
        return out

    # ---- introspection used by the drop-in boundary (same names as the reference)
    @property
    def input_node_features_dim(self):
        return self.graph_input_feature_dim

    @property
    def input_edge_features_dim(self):
        return self.graph_input_edge_dim

    @property
    def output_features_dim(self):
        return self.mlp_head.out_dim

    @property
    def gnn_layer_sizes(self):
        return [(c.in_channels, c.out_channels) for c in self.gnn_convs]

    @property
    def layers(self):
        return dict(self.named_children())

    @property
    def layer_names(self):
        return {k: f"{k}" for k in self.layers}

    @property
    def layer_parameters(self):
        return {k: list(v.named_parameters()) for k, v in self.layers.items()}

    @property
    def layer_parameters_flat(self):
        return [p for l in self.layer_parameters.values() for p in l]

    @property
    def layer_parameter_names(self):
        return {k: [layer_param_name_combiner(self.layer_names[k], p[0]) for p in v]
                for k, v in self.layer_parameters.items()}

    @property
    def layer_parameter_names_flat(self):
        return [p for l in self.layer_parameter_names.values() for p in l]

    @property
    def layer_parameter_shapes(self):
        return {k: [list(p[1].size()) for p in v] for k, v in self.layer_parameters.items()}

    @property
    def layer_parameter_shapes_flat(self):
        return [p for l in self.layer_parameter_shapes.values() for p in l]

    def named_parameter_arrays(self):
        """{flat reference name: contiguous fp32 numpy array}, in the reference's flat order."""
        out = {}
        for name, (_, p) in zip(self.layer_parameter_names_flat, self.layer_parameters_flat):
            out[name] = p.detach().cpu().to(torch.float32).contiguous().numpy()
        return out

    def describe(self) -> dict:
        """Plain description consumed by the C-ABI (gnnb_model_desc, include/gnnb_b200.h)."""
        conv0 = self.gnn_convs[0] if self.gnn_num_layers > 0 else None
        conv_name = conv0.__class__.__name__ if conv0 is not None else "GCNConv_GNNB"
        if self.uses_edge_features:
            conv_name = self._conv_cls.__name__
        d = dict(
            conv_type=CONV_TYPE_IDS[conv_name],
            num_layers=self.gnn_num_layers,
            in_dim=self.graph_input_feature_dim,
            hidden_dim=self.gnn_hidden_dim,
            out_dim=self.gnn_output_dim,
            skip=int(bool(self.gnn_skip_connection)),
            gnn_act=ACTIVATION_IDS[self.gnn_activation.__name__],
            gin_eps=float(getattr(conv0, "eps", 0.0) or 0.0),
            pna_delta=float(getattr(conv0, "delta_scaler", 1.0)),
            pools=[POOL_IDS[a] for a in self.global_pooling.aggrs],
            mlp_num_linear=self.mlp_head.num_of_layers,
            mlp_hidden=self.mlp_head.hidden_dim,
            mlp_out=self.mlp_head.out_dim,
            mlp_act=ACTIVATION_IDS[self.mlp_head.activation.__name__],
            out_act=ACTIVATION_IDS[self.output_activation.__name__
                                   if self.output_activation is not None else None],
        )
        if self.uses_edge_features:
            d["edge_dim"] = int(self.graph_input_edge_dim)
        if conv_name in _ATTENTION_CONVS:
            kw = self._conv_kwargs   # a model without layers has no conv to ask
            d["gat_heads"] = int(conv0.heads if conv0 is not None else kw.get("heads", 1))
        if conv_name in ("GATConv_GNNB", "GATv2Conv_GNNB"):   # TransformerConv has no slope
            d["gat_negative_slope"] = float(conv0.negative_slope if conv0 is not None
                                            else kw.get("negative_slope", 0.2))
        return d


def build_model(workload, pna_delta: float = 1.0, seed: int = 0) -> GNNModel:
    """GNNModel for one of ``configs.WORKLOADS`` with torch default-initialised weights
    (``torch.manual_seed(seed)``; there is no network for trained checkpoints)."""
    import functools

    torch.manual_seed(seed)
    conv = {"gcn": GCNConv_GNNB, "gin": GINConv_GNNB, "sage": SAGEConv_GNNB,
            "pna": PNAConv_GNNB}[workload.conv]
    if workload.conv == "pna":
        conv = functools.partial(PNAConv_GNNB, delta=pna_delta)
    elif workload.conv == "gin" and workload.gin_eps:
        conv = functools.partial(GINConv_GNNB, eps=workload.gin_eps)
    act = {"relu": nn.ReLU, "gelu": nn.GELU, "sigmoid": nn.Sigmoid, "tanh": nn.Tanh}[
        workload.activation]
    head = MLP(workload.gnn_output_dim * len(workload.pools), workload.out_dim,
               hidden_dim=workload.mlp_hidden_dim, hidden_layers=workload.mlp_hidden_layers,
               activation=nn.ReLU)
    return GNNModel(workload.in_dim, None, workload.hidden_dim, workload.num_layers,
                    workload.gnn_output_dim, conv, act, workload.skip,
                    GlobalPooling(list(workload.pools)), head, None)
