"""Backward of the GCN operator on the same kernels (the first "next" row of the scope table, SURVEY §8f rank 1).

The reference trains through PyG autograd (node_train_Gc run.py:26-37, node_train_Gs_GD run.py:177-215).  Here
x' = dropout(act(conv(x))) (network.py:31-33) is ONE torch.autograd.Function whose forward AND backward run on
libfitgnn_b200:

    out = act(Â · (x Wᵀ) + b);  y = out ⊙ mask / (1 - p)        mask = Philox(seed): regenerated in the backward, not stored
    gz  = g ⊙ mask / (1 - p) ⊙ act'(out)                        one kernel (fitgnn_elu_dropout_backward)
    db  = Σ_rows gz
    aggregate-first (in <= out):  A = Â x (saved);  dW = gzᵀ A;  dx = Âᵀ (gz W)
    transform-first (in >  out):  dZ = Âᵀ gz;       dW = dZᵀ x;  dx = dZ W

dW is the TN product over the rows: fitgnn_gemm_tn (transposing bf16 hi/lo split + batched split-K tcgen05 GEMM +
deterministic reduction); gz W and the forward transforms are NT products on the same tensor-core kernel.  Âᵀ is applied
with the CSR of the reversed edges and the ORIGINAL deg^-1/2 vector (for the undirected graphs of every reference
dataset Âᵀ = Â).  `nn.set_precision('fp32')` switches every GEMM here to the exact-fp32 CUDA-core kernel.
"""
from __future__ import annotations

import torch

from . import ops


class CsrPair:
    """Forward CSR (rows = targets) + CSR of the reversed graph (rows = sources), both with the forward dinv."""

    def __init__(self, rowptr, col, dinv, rowptr_t=None, col_t=None):
        self.rowptr, self.col, self.dinv = rowptr, col, dinv
        self.rowptr_t, self.col_t = rowptr_t, col_t

    @staticmethod
    def from_edge_index(edge_index, n):
        rowptr, col, dinv = ops.csr_from_coo(edge_index, n)
        return CsrPair(rowptr, col, dinv)

    def transposed(self):
        if self.rowptr_t is None:
            n = self.rowptr.numel() - 1
            deg = (self.rowptr[1:] - self.rowptr[:-1]).long()
            tgt = torch.repeat_interleave(torch.arange(n, device=self.col.device), deg)
            rev = torch.stack([tgt, self.col.long()])  # reversed edges: source := old target
            self.rowptr_t, self.col_t, _ = ops.csr_from_coo(rev.contiguous(), n)
        return self.rowptr_t, self.col_t


def _pad4(t):
    f = t.shape[1]
    if f % 4 == 0:
        return t.contiguous()
    out = torch.zeros(t.shape[0], ops.pad4(f), dtype=t.dtype, device=t.device)
    out[:, :f] = t
    return out


def _tc():
    from . import nn
    return nn._PRECISION == "bf16x3"


def _linear(x, w, bias=None, act=ops.ACT_NONE):
    """act(x · wᵀ + bias) with w [N, K]: tensor cores (bf16x3) or the exact-fp32 kernel (nn.set_precision)."""
    if _tc():
        return ops.linear_tc(x.contiguous(), w, bias, act)
    xp, wp = _pad4(x), _pad4(w)
    return ops.gemm_bias_act(xp, wp, bias, act, K=xp.shape[1])


def _grad_weight(g, a):
    """gᵀ · a  [out, in] — the contraction runs over the rows."""
    if _tc():
        return ops.gemm_tn(g, a)
    return ops.gemm_bias_act(g.t().contiguous(), a.t().contiguous())


class GCNConvFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, csr: CsrPair, act: int, dropout_p: float = 0.0, seed: int = 0):
        xin = _pad4(x.detach().float())
        w = _pad4(weight.detach())
        b = bias.detach().contiguous() if bias is not None else None
        fin, fout = weight.shape[1], weight.shape[0]
        ctx.csr, ctx.act, ctx.fin = csr, act, fin
        ctx.p, ctx.seed = float(dropout_p), int(seed)
        ctx.transform_first = fin > fout
        if ctx.transform_first:
            z = _linear(xin, w)
            out = ops.spmm_symnorm(csr.rowptr, csr.col, csr.dinv, z, bias=b, act=act)
            saved_in = xin
        else:
            a = ops.spmm_symnorm(csr.rowptr, csr.col, csr.dinv, xin)
            out = _linear(a, w, b, act)
            saved_in = a
        ctx.save_for_backward(saved_in, w, out)
        ctx.has_bias = bias is not None
        if ctx.p > 0.0:
            return ops.dropout(out, ctx.p, ctx.seed)
        return out

    @staticmethod
    def backward(ctx, g):
        saved_in, w, out = ctx.saved_tensors
        csr = ctx.csr
        g = g.contiguous().float()
        gz = ops.elu_dropout_backward(g, out, ctx.act, ctx.p, ctx.seed)
        db = gz.sum(0) if ctx.has_bias else None
        rp_t, col_t = csr.transposed()
        fin = ctx.fin
        wt = w.t().contiguous()  # [in_p, out]: the "weight" of the NT product gz · W
        if ctx.transform_first:
            dz = ops.spmm_symnorm(rp_t, col_t, csr.dinv, gz)               # Âᵀ gz   [n, out]
            dw = _grad_weight(dz, saved_in)                                 # dZᵀ x   [out, in_p]
            dx = _linear(dz, wt) if ctx.needs_input_grad[0] else None       # dZ W    [n, in_p]
        else:
            dw = _grad_weight(gz, saved_in)                                 # gzᵀ A   [out, in_p]
            dx = None
            if ctx.needs_input_grad[0]:
                da = _linear(gz, wt)                                        # gz W    [n, in_p]
                dx = ops.spmm_symnorm(rp_t, col_t, csr.dinv, da)            # Âᵀ dA
        if dx is not None:
            dx = dx[:, :fin]
        return dx, dw[:, :fin], db, None, None, None, None


def gcn_conv(x, weight, bias, csr: CsrPair, act: int = ops.ACT_NONE, dropout_p: float = 0.0, seed: int | None = None):
    """act(conv(x)) followed by dropout(p) (network.py:31-33).  seed None: drawn from torch's CPU generator, so
    torch.manual_seed makes a training run reproducible."""
    if dropout_p > 0.0 and seed is None:
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    return GCNConvFn.apply(x, weight, bias, csr, act, float(dropout_p), int(seed or 0))


# ----------------------------------------------------------------------------------------- SAGEConv
#   out = act(lin_l(M x) + lin_r(x)),  M = mean over the in-edges (a row without in-edges: 0);  y = dropout(out)
#   aggregate-first (in <= out):  A = [M x | x] (saved);  [dW_l | dW_r] = gzᵀ A;  dx = Mᵀ (gz W_l) + gz W_r
#   transform-first (in >  out):  dZ = [Mᵀ gz | gz];     [dW_l ; dW_r] = dZᵀ x;  dx = dZ [W_l ; W_r]
# Mᵀ runs on the CSR of the reversed edges with the per-entry weight 1 / count[original target] (the kernels' src_scale).
class SageCsr:
    """Raw CSR of an edge_index (ops.csr_raw_from_coo) + the reversed CSR and 1/in-degree for the backward."""

    def __init__(self, rowptr, col):
        self.rowptr, self.col = rowptr, col
        self.rowptr_t = self.col_t = self.inv_cnt = None

    @staticmethod
    def from_edge_index(edge_index, n):
        return SageCsr(*ops.csr_raw_from_coo(edge_index, n))

    def transposed(self):
        if self.rowptr_t is None:
            n = self.rowptr.numel() - 1
            deg = (self.rowptr[1:] - self.rowptr[:-1]).long()
            tgt = torch.repeat_interleave(torch.arange(n, device=self.col.device), deg)
            self.rowptr_t, self.col_t = ops.csr_raw_from_coo(torch.stack([tgt, self.col.long()]).contiguous(), n)
            self.inv_cnt = torch.where(deg > 0, 1.0 / deg.clamp(min=1).float(), torch.zeros((), device=deg.device)).contiguous()
        return self.rowptr_t, self.col_t, self.inv_cnt


def sage_weight_cat(w_l, w_r, half):
    """[W_l | W_r] with each half zero-padded to `half` columns: the weight of the concatenated operand [M x | x]."""
    f = w_l.shape[1]
    pad = (0, half - f)
    return torch.cat([torch.nn.functional.pad(w_l.detach().float(), pad), torch.nn.functional.pad(w_r.detach().float(), pad)],
                     1).contiguous()


class SAGEConvFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w_l, b_l, w_r, csr: SageCsr, act: int, dropout_p: float = 0.0, seed: int = 0):
        xin = _pad4(x.detach().float())
        fin, fout = w_l.shape[1], w_l.shape[0]
        b = b_l.detach().contiguous() if b_l is not None else None
        ctx.csr, ctx.act, ctx.fin, ctx.fout = csr, act, fin, fout
        ctx.p, ctx.seed = float(dropout_p), int(seed)
        ctx.transform_first = fin > fout
        if ctx.transform_first:
            w = _pad4(torch.cat([w_l.detach(), w_r.detach()], 0))        # [2 out, in_p]
            z = _linear(xin, w)
            out = ops.spmm_mean_root(csr.rowptr, csr.col, z, fout, bias=b, act=act)
            saved_in = xin
        else:
            kh = xin.shape[1]
            w = sage_weight_cat(w_l, w_r, kh)                              # [out, 2 kh]
            a = ops.spmm_mean_concat(csr.rowptr, csr.col, xin, kh, kh)
            out = _linear(a, w, b, act)
            saved_in = a
        ctx.save_for_backward(saved_in, w, out)
        ctx.has_bias = b_l is not None
        if ctx.p > 0.0:
            return ops.dropout(out, ctx.p, ctx.seed)
        return out

    @staticmethod
    def backward(ctx, g):
        saved_in, w, out = ctx.saved_tensors
        g = g.contiguous().float()
        gz = ops.elu_dropout_backward(g, out, ctx.act, ctx.p, ctx.seed)
        db = gz.sum(0) if ctx.has_bias else None
        rp_t, col_t, inv_cnt = ctx.csr.transposed()
        fin, fout = ctx.fin, ctx.fout
        dx = None
        if ctx.transform_first:
            dz = ops.spmm_mean_concat(rp_t, col_t, gz, fout, fout, src_scale=inv_cnt)  # [Mᵀ gz | gz]  [n, 2 out]
            dw = _grad_weight(dz, saved_in)                                             # [2 out, in_p]
            dw_l, dw_r = dw[:fout, :fin], dw[fout:, :fin]
            if ctx.needs_input_grad[0]:
                dx = _linear(dz, w.t().contiguous())[:, :fin]                           # dZ [W_l ; W_r]
        else:
            kh = w.shape[1] // 2
            dw = _grad_weight(gz, saved_in)                                             # [out, 2 kh]
            dw_l, dw_r = dw[:, :fin], dw[:, kh:kh + fin]
            if ctx.needs_input_grad[0]:
                da = _linear(gz, w.t().contiguous())                                    # [gz W_l | gz W_r]  [n, 2 kh]
                dx = ops.spmm_mean_root(rp_t, col_t, da, kh, kh, src_scale=inv_cnt)[:, :fin]
        return dx, dw_l.contiguous(), db, dw_r.contiguous(), None, None, None, None


def sage_conv(x, w_l, b_l, w_r, csr: SageCsr, act: int = ops.ACT_NONE, dropout_p: float = 0.0, seed: int | None = None):
    """dropout(act(SAGEConv(x))) (network.py:31-33 with layer_name='SAGEConv'); seed as gcn_conv."""
    if dropout_p > 0.0 and seed is None:
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    return SAGEConvFn.apply(x, w_l, b_l, w_r, csr, act, float(dropout_p), int(seed or 0))
