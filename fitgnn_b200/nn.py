"""Drop-in operator and model classes: same names, constructor arguments, forward signatures and
state_dict keys as the reference (/root/reference/network.py:8-204 and the Net1/Net2 duplicates in
inference.py:72-116), computing on the sm_100a kernels of libfitgnn_b200.so.

`GCNConv` stands where `getattr(pyg_nn, args.layer_name)` resolves (network.py:13): ctor
`GCNConv(in_channels, out_channels)`, parameters `lin.weight [out,in]` (glorot) and `bias [out]` (zeros),
`__call__(x[n,in] fp32, edge_index[2,E] int64) -> [n,out]`.

Autograd: when gradients are enabled and a parameter (or x) requires grad, the conv runs through
`fitgnn_b200.autograd.GCNConvFn`, whose backward uses the same kernels (SpMM with the reversed CSR; the dX = gz·W and
dW = gzᵀ·x products on the bf16x3 tensor cores, or on the exact-fp32 GEMM after `set_precision("fp32")`), so
the reference's training loops (run.py:26-37, :177-215) work unchanged; `.train()` mode applies F.dropout like
network.py:33.  Under torch.no_grad() the lean inference path is taken.  CUDA tensors only — there is no CPU path.
"""
from __future__ import annotations

import torch

from . import ops
from .autograd import CsrPair, SageCsr, gcn_conv, sage_conv, sage_weight_cat
from .engine import PackedForward
from .pack import Pack

# Arithmetic of the dense transforms on the inference (no-grad) path of the drop-in classes: 'bf16x3' = tcgen05 tensor
# cores on a bf16 hi/lo split of both operands with fp32 accumulation (default), 'fp32' = exact-fp32 CUDA-core GEMM
# (explicit opt-in: the numerics anchor).  The autograd path (training) follows the same setting: its forward GEMMs and the
# dX / dW products of the backward (fitgnn_gemm_tn) run on the bf16x3 tensor cores unless 'fp32' is selected.
_PRECISION = "bf16x3"


def set_precision(precision: str) -> str:
    """Select the GEMM arithmetic of GCNConv / the model classes' no-grad forward; returns the previous setting."""
    global _PRECISION
    if precision not in ("bf16x3", "fp32"):
        raise ValueError(f"precision={precision!r}")
    old, _PRECISION = _PRECISION, precision
    return old


_CSR_CACHE: dict = {}  # (kind, id(edge_index)) -> (weakref to the tensor, version, n, CsrPair | SageCsr)
_CSR_CACHE_MAX = 64


def _csr_for(edge_index, n, kind=CsrPair):
    """gcn_norm structure, cached per edge_index TENSOR OBJECT (PyG recomputes it on every call; cached=False).
    The entry is valid only while that very tensor is alive and unmodified: the weak reference must still resolve to
    the same object (an address or id reused by a new tensor can never alias a stale entry) and `_version` must match
    (in-place edits invalidate).  kind: CsrPair (gcn_norm structure) or SageCsr (the edges as given); the two never share an
    entry."""
    import weakref
    key = (kind, id(edge_index))
    hit = _CSR_CACHE.get(key)
    if hit is not None:
        ref, version, n_hit, csr = hit
        if ref() is edge_index and version == edge_index._version and n_hit == n:
            return csr
    if len(_CSR_CACHE) >= _CSR_CACHE_MAX:
        for k in [k for k, v in _CSR_CACHE.items() if v[0]() is None]:
            del _CSR_CACHE[k]
        if len(_CSR_CACHE) >= _CSR_CACHE_MAX:
            _CSR_CACHE.clear()
    csr = kind.from_edge_index(edge_index, n)
    _CSR_CACHE[key] = (weakref.ref(edge_index), edge_index._version, n, csr)
    return csr


def _as_f32_padded(x, align=4):
    """fp32, contiguous, row pitch a multiple of `align` floats (16-byte vector loads; 8 for the bf16 planes' pitch)."""
    if x.dtype != torch.float32:
        x = x.float()
    f = x.shape[1]
    if f % align != 0:
        xp = torch.zeros(x.shape[0], (f + align - 1) // align * align, dtype=torch.float32, device=x.device)
        xp[:, :f] = x
        return xp
    return x.contiguous()


def _pad_weight(w):
    w = w.detach()
    if w.shape[1] % 4 != 0:
        w = torch.nn.functional.pad(w, (0, ops.pad4(w.shape[1]) - w.shape[1]))
    return w.contiguous()


def _require_cuda(x):
    if not x.is_cuda:
        raise RuntimeError("fitgnn_b200 computes on CUDA tensors only (no CPU fallback); got a CPU tensor")


class GCNConv(torch.nn.Module):
    """Replacement for torch_geometric.nn.GCNConv as the reference uses it (add_self_loops=True,
    normalize=True, cached=False, bias=True)."""

    def __init__(self, in_channels: int, out_channels: int, **kwargs):
        super().__init__()
        if kwargs:
            raise TypeError(f"unsupported GCNConv options: {sorted(kwargs)}")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.lin = torch.nn.Linear(in_channels, out_channels, bias=False)
        self.bias = torch.nn.Parameter(torch.zeros(out_channels))
        self.reset_parameters()

    def reset_parameters(self):
        torch.nn.init.xavier_uniform_(self.lin.weight)  # PyG: glorot
        torch.nn.init.zeros_(self.bias)

    def forward(self, x, edge_index, act: int = ops.ACT_NONE, dropout_p: float = 0.0):
        """act / dropout_p: the F.elu / F.dropout that follow the conv in every reference model (network.py:32-33), fused
        into the operator (epilogue; Philox mask regenerated in the backward).  Defaults = the plain PyG operator."""
        _require_cuda(x)
        if self.out_channels % 4 != 0:
            raise RuntimeError("fitgnn_b200.GCNConv needs out_channels % 4 == 0")
        n = x.shape[0]
        csr = _csr_for(edge_index, n)
        if torch.is_grad_enabled() and (x.requires_grad or self.lin.weight.requires_grad or self.bias.requires_grad):
            return gcn_conv(x, self.lin.weight, self.bias, csr, act, dropout_p)
        if dropout_p > 0.0:  # train mode without gradients (the reference's loops never do this, but F.dropout would)
            y = self.forward(x, edge_index, act)
            return ops.dropout(y, dropout_p, int(torch.randint(0, 2 ** 62, (1,)).item()))
        rowptr, col, dinv = csr.rowptr, csr.col, csr.dinv
        b = self.bias.detach().contiguous()
        if _PRECISION == "bf16x3":  # tensor cores (network.py:31 call pattern, one conv per call)
            xp = _as_f32_padded(x.detach(), 8)
            if self.in_channels > self.out_channels:  # transform, then aggregate the narrower rows
                z = ops.linear_tc(xp, self.lin.weight)
                return ops.spmm_symnorm(rowptr, col, dinv, z, bias=b, act=act)
            # aggregate-first: Â(XW^T) = (ÂX)W^T; the SpMM emits the transform's bf16 hi/lo operand planes directly
            a = ops.spmm_symnorm(rowptr, col, dinv, xp, split=True)
            return ops.linear_tc(None, self.lin.weight, b, act, x_planes=a)
        xp = _as_f32_padded(x.detach())
        w = _pad_weight(self.lin.weight)
        if self.in_channels > self.out_channels:
            z = ops.gemm_bias_act(xp, w, None, ops.ACT_NONE, K=xp.shape[1])
            return ops.spmm_symnorm(rowptr, col, dinv, z, bias=b, act=act)
        a = ops.spmm_symnorm(rowptr, col, dinv, xp)
        return ops.gemm_bias_act(a, w, b, act, K=xp.shape[1])

    def extra_repr(self):
        return f"{self.in_channels}, {self.out_channels}"


class SAGEConv(torch.nn.Module):
    """Replacement for torch_geometric.nn.SAGEConv as `SAGEConv(in_channels, out_channels)` builds it (aggr='mean',
    normalize=False, root_weight=True, project=False, bias=True):  out_i = lin_l(mean_{j->i} x_j) + lin_r(x_i).
    Parameters lin_l.weight [out,in], lin_l.bias [out], lin_r.weight [out,in] (no bias).  Messages flow from
    edge_index[0] to edge_index[1]; no self loop is added, one in edge_index is an ordinary neighbour; duplicate edges count
    once per occurrence; a node without in-edges gets mean 0."""

    _DEFAULTS = dict(aggr="mean", normalize=False, root_weight=True, project=False, bias=True)

    def __init__(self, in_channels: int, out_channels: int, **kwargs):
        super().__init__()
        bad = sorted(k for k, v in kwargs.items() if k not in self._DEFAULTS or v != self._DEFAULTS[k])
        if bad:
            raise TypeError(f"unsupported SAGEConv options: {bad}")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.lin_l = torch.nn.Linear(in_channels, out_channels, bias=True)
        self.lin_r = torch.nn.Linear(in_channels, out_channels, bias=False)
        self.reset_parameters()

    def reset_parameters(self):
        self.lin_l.reset_parameters()  # PyG Linear: kaiming_uniform(a=sqrt(5)) weight, uniform bias — torch.nn.Linear's
        self.lin_r.reset_parameters()

    def forward(self, x, edge_index, act: int = ops.ACT_NONE, dropout_p: float = 0.0):
        """act / dropout_p: the F.elu / F.dropout that follow the conv in every reference model, fused as in GCNConv."""
        _require_cuda(x)
        if self.out_channels % 4 != 0:
            raise RuntimeError("fitgnn_b200.SAGEConv needs out_channels % 4 == 0")
        n = x.shape[0]
        csr = _csr_for(edge_index, n, SageCsr)
        wl, bl, wr = self.lin_l.weight, self.lin_l.bias, self.lin_r.weight
        if torch.is_grad_enabled() and (x.requires_grad or wl.requires_grad or bl.requires_grad or wr.requires_grad):
            return sage_conv(x, wl, bl, wr, csr, act, dropout_p)
        if dropout_p > 0.0:
            y = self.forward(x, edge_index, act)
            return ops.dropout(y, dropout_p, int(torch.randint(0, 2 ** 62, (1,)).item()))
        b = bl.detach().contiguous()
        align = 8 if _PRECISION == "bf16x3" else 4
        xp = _as_f32_padded(x.detach(), align)
        if self.in_channels > self.out_channels:  # Z = x [W_l ; W_r]^T on the wide rows, then mean + root + bias + act
            w = torch.cat([wl.detach(), wr.detach()], 0)
            if _PRECISION == "bf16x3":
                z = ops.linear_tc(xp, w)
            else:
                z = ops.gemm_bias_act(xp, _pad_weight(w), None, ops.ACT_NONE, K=xp.shape[1])
            return ops.spmm_mean_root(csr.rowptr, csr.col, z, self.out_channels, bias=b, act=act)
        # aggregate-first: [mean x | x] as ONE operand, one GEMM against [W_l | W_r]
        kh = xp.shape[1]
        w = sage_weight_cat(wl, wr, kh)
        if _PRECISION == "bf16x3":
            a = ops.spmm_mean_concat(csr.rowptr, csr.col, xp, kh, kh, split=True)
            return ops.linear_tc(None, w, b, act, x_planes=a)
        a = ops.spmm_mean_concat(csr.rowptr, csr.col, xp, kh, kh)
        return ops.gemm_bias_act(a, w, b, act, K=2 * kh)

    def extra_repr(self):
        return f"{self.in_channels}, {self.out_channels}, aggr=mean"


_LAYERS = {"GCNConv": GCNConv, "SAGEConv": SAGEConv}


def _layer_class(args):
    name = getattr(args, "layer_name", "GCNConv")
    if name not in _LAYERS:
        raise NotImplementedError(f"layer_name={name!r}: only {sorted(_LAYERS)} are on the B200 hot path (SURVEY §2 row 15)")
    return _LAYERS[name]


class _ConvStack(torch.nn.Module):
    """Shared body of the six reference model classes (network.py:9-27 etc.)."""
    _out_dim_from_args = True

    def __init__(self, args):
        super().__init__()
        self.num_layers = args.num_layers1
        Layer = _layer_class(args)
        self.conv = torch.nn.ModuleList()
        self.conv.append(Layer(args.num_features, args.hidden))
        for _ in range(self.num_layers - 1):
            self.conv.append(Layer(args.hidden, args.hidden))
        self.lt1 = torch.nn.Linear(args.hidden, args.num_classes if self._out_dim_from_args else 1)

    def reset_parameters(self):
        for module in self.conv:
            module.reset_parameters()
        self.lt1.reset_parameters()

    def _convs(self, x, edge_index):
        # network.py:30-33: conv -> F.elu -> F.dropout(training=self.training); ELU is fused into the conv epilogue
        for i in range(self.num_layers):
            x = self.conv[i](x, edge_index, act=ops.ACT_ELU, dropout_p=0.5 if self.training else 0.0)  # F.dropout default p
        return x

    def _lt1(self, x, head):
        if torch.is_grad_enabled() and (x.requires_grad or self.lt1.weight.requires_grad or self.lt1.bias.requires_grad):
            y = self.lt1(x)  # differentiable tail (F.linear + softmax family), network.py:34-35
            if head == ops.HEAD_LOG_SOFTMAX:
                return torch.nn.functional.log_softmax(y, dim=1)
            return torch.nn.functional.softmax(y, dim=1) if head == ops.HEAD_SOFTMAX else y
        w = self.lt1.weight.detach().contiguous()
        if _PRECISION == "bf16x3" and x.shape[1] % 8 == 0:
            return ops.linear_tc(x.contiguous(), w, self.lt1.bias.detach().contiguous(), ops.ACT_NONE, head)
        return ops.gemm_bias_act(x, w, self.lt1.bias.detach().contiguous(), ops.ACT_NONE, head)

    def packed(self, pack: Pack, head=None, rows=None, precision=None) -> PackedForward:
        """Fast path: the prepared whole-pack forward with this module's current parameters."""
        return PackedForward(pack, self.state_dict(), head=head if head is not None else self._head,
                             rows=rows if rows is not None else self._rows, precision=precision or _PRECISION)


class Classify_node(_ConvStack):
    """network.py:8-35."""
    _head, _rows = "log_softmax", "core"

    def forward(self, x, edge_index):
        return self._lt1(self._convs(x, edge_index), ops.HEAD_LOG_SOFTMAX)


class Regress_node(_ConvStack):
    """network.py:37-64."""
    _out_dim_from_args = False
    _head, _rows = "identity", "core"

    def forward(self, x, edge_index):
        return self._lt1(self._convs(x, edge_index), ops.HEAD_IDENTITY)


class GraphBatch:
    """A collated batch of graphs, each given as its list of subgraphs (the `set_gs` argument of the
    reference's *_gs models, built by colater utils.py:893-908): one block-diagonal CSR for all subgraphs of
    all graphs, the masked rows in order, and the pooling segments of batch_tensor."""

    def __init__(self, set_gs, batch_tensor, device):
        xs, eis, masks, off = [], [], [], 0
        for gs in set_gs:
            for g in gs:
                xs.append(g.x.float())
                eis.append(g.edge_index + off)
                masks.append(g.mask)
                off += g.x.shape[0]
        self.x = torch.cat(xs, 0).to(device)
        self.edge_index = torch.cat(eis, 1).to(device).contiguous()
        mask = torch.cat(masks, 0).to(device)
        self.rows = torch.nonzero(mask).view(-1).to(torch.int32)
        bt = batch_tensor.to(device).to(torch.int64)  # network.py:131: batch_tensor.type(torch.int64)
        n_graphs = int(bt.max().item()) + 1 if bt.numel() else 0
        assert bt.numel() == self.rows.numel(), "batch_tensor must have one entry per masked row"
        assert bool((bt[1:] >= bt[:-1]).all()), "batch_tensor must be sorted (colater builds it that way)"
        counts = torch.bincount(bt, minlength=n_graphs)
        self.seg_ptr = torch.zeros(n_graphs + 1, dtype=torch.int32, device=device)
        self.seg_ptr[1:] = torch.cumsum(counts, 0).to(torch.int32)


class _GraphGs(_ConvStack):
    def _forward_gs(self, set_gs, batch_tensor, pool, head):
        dev = self.lt1.weight.device
        gb = set_gs if isinstance(set_gs, GraphBatch) else GraphBatch(set_gs, batch_tensor, dev)
        x = self._convs(gb.x, gb.edge_index)
        pooled = ops.segment_pool(x, gb.rows, gb.seg_ptr, pool)
        return self._lt1(pooled, head)


class _GraphGc(_ConvStack):
    def _forward_gc(self, gc, pool, head):
        x, edge_index, batch = gc.x, gc.edge_index, gc.batch
        _require_cuda(x)
        n_graphs = int(batch.max().item()) + 1
        assert bool((batch[1:] >= batch[:-1]).all()), "gc.batch must be sorted (PyG Batch builds it that way)"
        seg_ptr = torch.zeros(n_graphs + 1, dtype=torch.int32, device=x.device)
        seg_ptr[1:] = torch.cumsum(torch.bincount(batch, minlength=n_graphs), 0).to(torch.int32)
        h = self._convs(x.float(), edge_index.contiguous())
        return self._lt1(ops.segment_pool(h, None, seg_ptr, pool), head)


class Classify_graph_gc(_GraphGc):
    """network.py:66-95: conv stack -> global_max_pool -> lt1 -> softmax."""
    _head, _rows = "softmax", "all"

    def forward(self, gc):
        return self._forward_gc(gc, ops.POOL_MAX, ops.HEAD_SOFTMAX)


class Classify_graph_gs(_GraphGs):
    """network.py:97-135: per-subgraph conv stack -> x[mask] -> global_max_pool -> lt1 -> softmax."""
    _head, _rows = "softmax", "mask"

    def forward(self, set_gs, batch_tensor=None):
        return self._forward_gs(set_gs, batch_tensor, ops.POOL_MAX, ops.HEAD_SOFTMAX)


class Regress_graph_gc(_GraphGc):
    """network.py:137-166: conv stack -> global_mean_pool -> lt1."""
    _out_dim_from_args = False
    _head, _rows = "identity", "all"

    def forward(self, gc):
        return self._forward_gc(gc, ops.POOL_MEAN, ops.HEAD_IDENTITY)


class Regress_graph_gs(_GraphGs):
    """network.py:168-204: per-subgraph conv stack -> x[mask] -> global_mean_pool -> lt1."""
    _out_dim_from_args = False
    _head, _rows = "identity", "mask"

    def forward(self, set_gs, batch_tensor=None):
        return self._forward_gs(set_gs, batch_tensor, ops.POOL_MEAN, ops.HEAD_IDENTITY)


def _ns(num_features, hidden, num_layers, num_classes, layer_name="GCNConv"):
    import argparse
    return argparse.Namespace(num_features=num_features, hidden=hidden, num_layers1=num_layers,
                              num_classes=num_classes, layer_name=layer_name)


class Net1(Classify_node):
    """inference.py:72-93 `Net1(num_features, hidden, num_layers, num_classes)` — same state_dict keys.  layer_name: the
    conv class, as args.layer_name of the network.py models."""

    def __init__(self, num_features, hidden, num_layers, num_classes, layer_name="GCNConv"):
        super().__init__(_ns(num_features, hidden, num_layers, num_classes, layer_name))


class Net2(Regress_node):
    """inference.py:95-116 `Net2(num_features, hidden, num_layers)`."""

    def __init__(self, num_features, hidden, num_layers, num_classes=1, layer_name="GCNConv"):
        super().__init__(_ns(num_features, hidden, num_layers, 1, layer_name))


def install():
    """Route the reference's layer lookup to this module: after `fitgnn_b200.nn.install()`,
    `getattr(torch_geometric.nn, 'GCNConv')` / `'SAGEConv'` (network.py:13) and `from torch_geometric.nn import GCNConv`
    (network.py:5, inference.py) resolve to the B200 operators.  Call before importing network.py."""
    import importlib
    pyg_nn = importlib.import_module("torch_geometric.nn")
    pyg_nn.GCNConv = GCNConv
    pyg_nn.SAGEConv = SAGEConv
    return pyg_nn
