"""Thin torch-tensor wrappers over the C ABI (include/fitgnn.h).  torch is used for device memory and
streams only; every computation happens inside libfitgnn_b200.so on the current CUDA stream."""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import check, lib, ptr, stream_ptr

ACT_NONE, ACT_ELU = 0, 1
HEAD_IDENTITY, HEAD_LOG_SOFTMAX, HEAD_SOFTMAX = 0, 1, 2
MODE_NONE, MODE_EXTRA, MODE_CLUSTER = 0, 1, 2
POOL_MAX, POOL_MEAN = 0, 1
GEMM_FP32, GEMM_BF16X3 = 0, 1
MODES = {"none": MODE_NONE, "extra": MODE_EXTRA, "cluster": MODE_CLUSTER}


def _ws(nbytes, device):
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


def pad4(n):
    return (int(n) + 3) // 4 * 4


# ----------------------------------------------------------------------------------------- primitives
def sort_u64(keys, vals=None, key_bits=64):
    """In-place ascending radix sort of int64 keys interpreted as unsigned (low key_bits bits)."""
    assert keys.dtype == torch.int64 and (vals is None or vals.dtype == torch.int32)
    ws = _ws(lib().fitgnn_sort_workspace_bytes(keys.numel()), keys.device)
    check(lib().fitgnn_sort_u64(ptr(keys), ptr(vals), keys.numel(), key_bits, ptr(ws), ws.numel(), stream_ptr()))
    return keys, vals


def scan_i32(x, with_total=True):
    assert x.dtype == torch.int32
    out = torch.empty(x.numel() + (1 if with_total else 0), dtype=torch.int32, device=x.device)
    ws = _ws(lib().fitgnn_scan_workspace_bytes(x.numel()), x.device)
    check(lib().fitgnn_scan_i32(ptr(x), ptr(out), x.numel(), int(with_total), ptr(ws), ws.numel(), stream_ptr()))
    return out


# ----------------------------------------------------------------------------------------- CSR / SpMM
def csr_from_coo(edge_index, n):
    """gcn_norm structure for the drop-in GCNConv: (rowptr, col, dinv) with self loops re-added."""
    assert edge_index.dtype == torch.int64 and edge_index.dim() == 2 and edge_index.shape[0] == 2
    ei = edge_index.contiguous()
    E = ei.shape[1]
    ws = _ws(lib().fitgnn_csr_workspace_bytes(E, n), ei.device)
    nnz = C.c_int64(0)
    check(lib().fitgnn_csr_plan(ptr(ei), E, n, ptr(ws), ws.numel(), C.byref(nnz), stream_ptr()))
    rowptr = torch.empty(n + 1, dtype=torch.int32, device=ei.device)
    col = torch.empty(max(nnz.value, 1), dtype=torch.int32, device=ei.device)[: nnz.value]
    dinv = torch.empty(n, dtype=torch.float32, device=ei.device)
    check(lib().fitgnn_csr_fill(n, ptr(ws), ws.numel(), ptr(rowptr), ptr(col), ptr(dinv), stream_ptr()))
    return rowptr, col, dinv


def csr_raw_from_coo(edge_index, n):
    """CSR of the edges exactly as given (drop-in SAGEConv): (rowptr, col), rows = targets, self loops and duplicate
    edges kept as ordinary entries, none added; columns ascending inside a row."""
    assert edge_index.dtype == torch.int64 and edge_index.dim() == 2 and edge_index.shape[0] == 2
    ei = edge_index.contiguous()
    E = ei.shape[1]
    ws = _ws(lib().fitgnn_csr_workspace_bytes(E, n), ei.device)
    nnz = C.c_int64(0)
    check(lib().fitgnn_csr_raw_plan(ptr(ei), E, n, ptr(ws), ws.numel(), C.byref(nnz), stream_ptr()))
    rowptr = torch.empty(n + 1, dtype=torch.int32, device=ei.device)
    col = torch.empty(max(nnz.value, 1), dtype=torch.int32, device=ei.device)[: nnz.value]
    check(lib().fitgnn_csr_raw_fill(n, ptr(ws), ws.numel(), ptr(rowptr), ptr(col), stream_ptr()))
    return rowptr, col


def _mean_out(n_out, ncols, split, out, device):
    if split:
        if out is None:
            out = (torch.empty(n_out, ncols, dtype=torch.bfloat16, device=device),
                   torch.empty(n_out, ncols, dtype=torch.bfloat16, device=device))
        return out, out[0], out[1], out[0].stride(0)
    if out is None:
        out = torch.empty(n_out, ncols, dtype=torch.float32, device=device)
    return out, out, None, out.stride(0)


def spmm_mean_concat(rowptr, col, X, width=None, half=None, src_index=None, src_scale=None, skip_self=False, out_rows=None,
                     out=None, split=False):
    """SAGEConv operand: Y[i] = [mean_j X[src(j)] | X[src(r_i)]], halves `half` columns apart (default width), pad columns
    zero (fitgnn_spmm_mean_concat).  split=True returns bf16 (hi, lo) planes [n_out, 2*half] for the tensor-core GEMM.
    skip_self: the entry col == row is not a neighbour (pack CSRs); src_scale: weighted sum instead of the mean."""
    assert X.dtype == torch.float32 and X.dim() == 2
    width = X.shape[1] if width is None else width
    half = width if half is None else half
    n_out = out_rows.numel() if out_rows is not None else rowptr.numel() - 1
    out, y, ylo, ldy = _mean_out(n_out, 2 * half, split, out, X.device)
    check(lib().fitgnn_spmm_mean_concat(ptr(rowptr), ptr(col), ptr(X), X.stride(0), width, half, ptr(src_index),
                                        ptr(src_scale), int(bool(skip_self)), ptr(out_rows), n_out, ptr(y), ptr(ylo), ldy,
                                        stream_ptr()))
    return out


def spmm_mean_root(rowptr, col, Z, width, root_off=None, src_index=None, src_scale=None, skip_self=False, bias=None,
                   act=ACT_NONE, out_rows=None, out=None, split=False):
    """Transform-first SAGEConv: Y[i] = act(mean_j Z[src(j), :width] + Z[src(r_i), root_off:root_off+width] + bias) with
    Z = X·[W_l ; W_r]^T (root_off defaults to width) (fitgnn_spmm_mean_root)."""
    assert Z.dtype == torch.float32 and Z.dim() == 2
    root_off = width if root_off is None else root_off
    n_out = out_rows.numel() if out_rows is not None else rowptr.numel() - 1
    out, y, ylo, ldy = _mean_out(n_out, width, split, out, Z.device)
    check(lib().fitgnn_spmm_mean_root(ptr(rowptr), ptr(col), ptr(Z), Z.stride(0), width, root_off, ptr(src_index),
                                      ptr(src_scale), int(bool(skip_self)), ptr(bias), act, ptr(out_rows), n_out, ptr(y),
                                      ptr(ylo), ldy, stream_ptr()))
    return out


def spmm_mean_f16(rowptr, col, X, width=None, half=None, src_index=None, skip_self=False, out_rows=None, concat=False,
                  out=None):
    """spmm_mean_concat on fp16 planes (fitgnn_spmm_mean_f16): X one fp16 plane, the result one fp16 plane [n_out, half]
    (the mean alone) or, concat=True, [n_out, 2*half] = [mean | root]; fp32 sums, one saturating rounding."""
    assert X.dtype == torch.float16 and X.dim() == 2
    width = X.shape[1] if width is None else width
    half = width if half is None else half
    n_out = out_rows.numel() if out_rows is not None else rowptr.numel() - 1
    if out is None:
        out = torch.empty(n_out, 2 * half if concat else half, dtype=torch.float16, device=X.device)
    check(lib().fitgnn_spmm_mean_f16(ptr(rowptr), ptr(col), ptr(X), X.stride(0), width, half, ptr(src_index),
                                     int(bool(skip_self)), int(bool(concat)), ptr(out_rows), n_out, ptr(out), out.stride(0),
                                     stream_ptr()))
    return out


def spmm_mean_root_f16(rowptr, col, Z, width, root_off=None, src_index=None, skip_self=False, bias=None, act=ACT_NONE,
                       out_rows=None, out=None):
    """spmm_mean_root whose result is ONE fp16 plane [n_out, width] (fitgnn_spmm_mean_root_f16); Z stays fp32."""
    assert Z.dtype == torch.float32 and Z.dim() == 2
    root_off = width if root_off is None else root_off
    n_out = out_rows.numel() if out_rows is not None else rowptr.numel() - 1
    if out is None:
        out = torch.empty(n_out, width, dtype=torch.float16, device=Z.device)
    check(lib().fitgnn_spmm_mean_root_f16(ptr(rowptr), ptr(col), ptr(Z), Z.stride(0), width, root_off, ptr(src_index),
                                          int(bool(skip_self)), ptr(bias), act, ptr(out_rows), n_out, ptr(out), out.stride(0),
                                          stream_ptr()))
    return out


def spmm_symnorm(rowptr, col, dinv, X, width=None, src_index=None, bias=None, act=ACT_NONE, out_rows=None,
                 out=None, split=False, hubs=None):
    """Y = act(Â·X[src_index] + bias) on the rows `out_rows` (all rows when None).
    split=True returns bf16 (hi, lo) planes for the tensor-core GEMM instead of fp32."""
    assert X.dtype == torch.float32 and X.dim() == 2
    ldx = X.stride(0)
    width = X.shape[1] if width is None else width
    n_out = out_rows.numel() if out_rows is not None else rowptr.numel() - 1
    if split:
        if out is None:
            out = (torch.empty(n_out, width, dtype=torch.bfloat16, device=X.device),
                   torch.empty(n_out, width, dtype=torch.bfloat16, device=X.device))
        y, ylo, ldy = out[0], out[1], out[0].stride(0)
    else:
        if out is None:
            out = torch.empty(n_out, width, dtype=torch.float32, device=X.device)
        y, ylo, ldy = out, None, out.stride(0)
    if hubs is not None and hubs[1] > 0:
        hub_list, n_hub, hub_deg = hubs
        check(lib().fitgnn_spmm_symnorm_hub(ptr(rowptr), ptr(col), ptr(dinv), ptr(X), ldx, width, ptr(src_index),
                                            ptr(bias), act, ptr(out_rows), n_out, ptr(y), ptr(ylo), ldy,
                                            ptr(hub_list), n_hub, hub_deg, stream_ptr()))
    else:
        check(lib().fitgnn_spmm_symnorm(ptr(rowptr), ptr(col), ptr(dinv), ptr(X), ldx, width, ptr(src_index),
                                        ptr(bias), act, ptr(out_rows), n_out, ptr(y), ptr(ylo), ldy, stream_ptr()))
    return out


def spmm_symnorm_f16(rowptr, col, dinv, X, width=None, src_index=None, bias=None, act=ACT_NONE, out_rows=None, out=None,
                     hubs=None):
    """spmm_symnorm on ONE fp16 plane in and out (FITGNN_GEMM_FP16X2's hidden state): fp32 sums, half the gathered bytes."""
    assert X.dtype == torch.float16 and X.dim() == 2
    width = X.shape[1] if width is None else width
    n_out = out_rows.numel() if out_rows is not None else rowptr.numel() - 1
    if out is None:
        out = torch.empty(n_out, width, dtype=torch.float16, device=X.device)
    hub_list, n_hub, hub_deg = hubs if (hubs is not None and hubs[1] > 0) else (None, 0, 0)
    check(lib().fitgnn_spmm_symnorm_f16(ptr(rowptr), ptr(col), ptr(dinv), ptr(X), X.stride(0), width, ptr(src_index), ptr(bias),
                                        act, ptr(out_rows), n_out, ptr(out), out.stride(0), ptr(hub_list), None, n_hub, hub_deg,
                                        stream_ptr()))
    return out


def spmm_symnorm_grouped(rowptr, col, dinv, X, width=None, src_index=None, out=None, split=False, group=32,
                         pad_value=None):
    """Y = Â·X[src_index] on a group-aligned pack (Pack.aligned): fitgnn_spmm_symnorm_grouped, bit-identical to
    spmm_symnorm without bias / activation / row selection.  Raises FitgnnError(EUNSUP) for width > 128.
    pad_value (split planes with pitch width + 4 only): also write the pad columns, hi[:, width] = pad_value, rest 0."""
    assert X.dtype == torch.float32 and X.dim() == 2
    width = X.shape[1] if width is None else width
    n = rowptr.numel() - 1
    if split:
        if out is None:
            out = (torch.empty(n, width, dtype=torch.bfloat16, device=X.device),
                   torch.empty(n, width, dtype=torch.bfloat16, device=X.device))
        y, ylo, ldy = out[0], out[1], out[0].stride(0)
    else:
        if out is None:
            out = torch.empty(n, width, dtype=torch.float32, device=X.device)
        y, ylo, ldy = out, None, out.stride(0)
    check(lib().fitgnn_spmm_symnorm_grouped(ptr(rowptr), ptr(col), ptr(dinv), ptr(X), X.stride(0), width, ptr(src_index),
                                            n, group, ptr(y), ptr(ylo), ldy, int(pad_value is not None),
                                            float(pad_value or 0.0), stream_ptr()))
    return out


def spmm_symnorm_grouped_f16(rowptr, col, dinv, X, width=None, src_index=None, out=None, pad_value=None):
    """spmm_symnorm_grouped written as ONE fp16 plane (fitgnn_spmm_symnorm_grouped_f16): fp32 sums, one rounding.  `out`:
    fp16 [n_rows, ldy]; pad_value (pitch width + 4 only): out[:, width] = pad_value, the other pad elements 0."""
    assert X.dtype == torch.float32 and X.dim() == 2
    width = X.shape[1] if width is None else width
    n = rowptr.numel() - 1
    if out is None:
        out = torch.empty(n, width, dtype=torch.float16, device=X.device)
    assert out.dtype == torch.float16 and out.shape[0] == n
    check(lib().fitgnn_spmm_symnorm_grouped_f16(ptr(rowptr), ptr(col), ptr(dinv), ptr(X), X.stride(0), width, ptr(src_index), n,
                                                32, ptr(out), out.stride(0), int(pad_value is not None), float(pad_value or 0.0),
                                                stream_ptr()))
    return out


def row_blocks(sub_ptr, n_rows, window=64, compact=False):
    """blk_ptr for spmm_symnorm_blocked: block b = the subgraphs whose first row lies in [b*window, (b+1)*window) — unions
    of whole subgraphs, so closed under adjacency; a block has fewer than window + (largest subgraph) rows, empty blocks
    (inside a subgraph that spans several windows) are skipped by the kernel.  sub_ptr must be non-decreasing."""
    sp = sub_ptr.long()
    nb = (int(n_rows) + window - 1) // window
    first = torch.searchsorted(sp[:-1].contiguous(), torch.arange(nb, device=sp.device) * window)
    blk = torch.cat([sp[first.clamp(max=sp.numel() - 1)], sp[-1:]])
    if compact:  # drop the empty blocks (windows inside a subgraph that spans several): the kernels skip them, but each costs
        blk = torch.unique_consecutive(blk)  # a CTA two dependent loads; boundaries stay whole-subgraph boundaries
        if blk.numel() < 2:
            blk = torch.stack([sp[0], sp[-1]])
    return blk.to(torch.int32).contiguous()


def block_row_order(rowptr, blk_ptr):
    """row_order for spmm_symnorm_blocked: the rows of every block sorted by row length (descending, stable), blocks in
    place.  int32 [n_rows]."""
    n = rowptr.numel() - 1
    deg = (rowptr[1:] - rowptr[:-1]).long()
    rows = torch.arange(n, device=rowptr.device)
    blk = torch.searchsorted(blk_ptr[1:].long().contiguous(), rows, right=True)
    key = blk * (int(deg.max()) + 1 if n else 1) + (int(deg.max()) - deg if n else deg)
    return torch.sort(key, stable=True).indices.to(torch.int32).contiguous()


def spmm_symnorm_blocked(rowptr, col, dinv, X, blk_ptr, width=None, src_index=None, bias=None, act=ACT_NONE, out=None,
                         split=False, row_order=None):
    """Y = act(Â·X[src_index] + bias) for every row, sources staged block by block in shared memory
    (fitgnn_spmm_symnorm_blocked; blk_ptr from row_blocks).  Bit-identical to spmm_symnorm."""
    assert X.dtype == torch.float32 and X.dim() == 2 and blk_ptr.dtype == torch.int32
    width = X.shape[1] if width is None else width
    n = rowptr.numel() - 1
    if split:
        if out is None:
            out = (torch.empty(n, width, dtype=torch.bfloat16, device=X.device),
                   torch.empty(n, width, dtype=torch.bfloat16, device=X.device))
        y, ylo, ldy = out[0], out[1], out[0].stride(0)
    else:
        if out is None:
            out = torch.empty(n, width, dtype=torch.float32, device=X.device)
        y, ylo, ldy = out, None, out.stride(0)
    check(lib().fitgnn_spmm_symnorm_blocked(ptr(rowptr), ptr(col), ptr(dinv), ptr(X), X.stride(0), width, ptr(src_index),
                                            ptr(blk_ptr), blk_ptr.numel() - 1, ptr(row_order), ptr(bias), act, ptr(y),
                                            ptr(ylo), ldy, stream_ptr()))
    return out


def spmm_symnorm_mma(rowptr, col, dinv, X, blk_ptr, width=None, src_index=None, bias=None, act=ACT_NONE, out=None, split=False):
    """Y = act(Â·X[src_index] + bias) for every row with the block-dense tensor-core kernel (fitgnn_spmm_symnorm_mma):
    per 128 x 128 piece of a block's 0/1 adjacency one small MMA.  ~1e-6 relative to spmm_symnorm."""
    assert X.dtype == torch.float32 and X.dim() == 2 and blk_ptr.dtype == torch.int32
    width = X.shape[1] if width is None else width
    n = rowptr.numel() - 1
    if split:
        if out is None:
            out = (torch.empty(n, width, dtype=torch.bfloat16, device=X.device),
                   torch.empty(n, width, dtype=torch.bfloat16, device=X.device))
        y, ylo, ldy = out[0], out[1], out[0].stride(0)
    else:
        if out is None:
            out = torch.empty(n, width, dtype=torch.float32, device=X.device)
        y, ylo, ldy = out, None, out.stride(0)
    check(lib().fitgnn_spmm_symnorm_mma(ptr(rowptr), ptr(col), ptr(dinv), ptr(X), X.stride(0), width, ptr(src_index),
                                        ptr(blk_ptr), blk_ptr.numel() - 1, ptr(bias), act, ptr(y), ptr(ylo), ldy, stream_ptr()))
    return out


def find_hubs(rowptr, out_rows, n_out, hub_deg=256, cap=None):
    """Output rows with >= hub_deg entries -> (hub_list, n_hub, hub_deg).  Synchronises once (build time)."""
    cap = int(cap if cap is not None else max(1024, n_out // 64))
    hub_list = torch.empty(cap, dtype=torch.int32, device=rowptr.device)
    cnt = torch.zeros(1, dtype=torch.int32, device=rowptr.device)
    check(lib().fitgnn_spmm_hubs(ptr(rowptr), ptr(out_rows), n_out, hub_deg, ptr(hub_list), ptr(cnt), cap,
                                 stream_ptr()))
    n = int(cnt.item())
    if n > cap:
        return find_hubs(rowptr, out_rows, n_out, hub_deg, n)
    hub_list = torch.sort(hub_list[:n]).values.contiguous() if n > 0 else hub_list[:0]
    return hub_list, n, hub_deg


# ----------------------------------------------------------------------------------------- dense
def gemm_bias_act(A, W, bias=None, act=ACT_NONE, head=HEAD_IDENTITY, out=None, K=None, N=None, precision=GEMM_FP32,
                  split_out=False, row_scale=None):
    """Y = head(act(row_scale[:, None] * (A·W^T) + bias)).  FP32: A [M,K] fp32, W [N,K] fp32.  BF16X3: A=(hi,lo),
    W=(hi,lo) bf16 planes.  split_out=True (BF16X3 only) returns the result as bf16 (hi, lo) planes for the next
    tensor-core GEMM.  row_scale ([M] fp32, BF16X3 only) is folded into the bias add."""
    if precision == GEMM_FP32:
        a_hi, a_lo, w_hi, w_lo = A, None, W, None
        assert A.dtype == torch.float32 and W.dtype == torch.float32
    else:
        (a_hi, a_lo), (w_hi, w_lo) = A, W
        assert a_hi.dtype == torch.bfloat16 and w_hi.dtype == torch.bfloat16
    M = a_hi.shape[0]
    K = a_hi.shape[1] if K is None else K
    N = w_hi.shape[0] if N is None else N
    if split_out:
        if out is None:
            out = (torch.empty(M, N, dtype=torch.bfloat16, device=a_hi.device),
                   torch.empty(M, N, dtype=torch.bfloat16, device=a_hi.device))
        check(lib().fitgnn_gemm_rowscale_bias_act_split(precision, ptr(a_hi), ptr(a_lo), a_hi.stride(0), ptr(w_hi),
                                                        ptr(w_lo), w_hi.stride(0), ptr(row_scale), ptr(bias), M, K, N, act,
                                                        head, ptr(out[0]), ptr(out[1]), out[0].stride(0), stream_ptr()))
        return out
    if out is None:
        out = torch.empty(M, N, dtype=torch.float32, device=a_hi.device)
    check(lib().fitgnn_gemm_rowscale_bias_act_split(precision, ptr(a_hi), ptr(a_lo), a_hi.stride(0), ptr(w_hi), ptr(w_lo),
                                                    w_hi.stride(0), ptr(row_scale), ptr(bias), M, K, N, act, head, ptr(out),
                                                    None, out.stride(0), stream_ptr()))
    return out


def pad8(n):
    return (int(n) + 7) // 8 * 8


def linear_tc(x, weight, bias=None, act=ACT_NONE, head=HEAD_IDENTITY, x_planes=None):
    """head(act(x · weight^T + bias)) on the tensor cores from fp32 operands: both are split into bf16 hi/lo planes
    (K padded to 8) and run through FITGNN_GEMM_BF16X3.  x: [M, K] fp32 (ignored when x_planes — already split, pitch
    pad8(K) — is given); weight: [N, K] fp32 as lin.weight."""
    N, K = weight.shape
    Kp = pad8(K)
    w_pl = split_bf16(weight.detach().contiguous(), ldo=Kp)
    a_pl = x_planes if x_planes is not None else split_bf16(x, cols=K, ldo=Kp)
    return gemm_bias_act(a_pl, w_pl, bias, act, head, K=Kp, N=N, precision=GEMM_BF16X3)


def gcn_layer_fused(rowptr, col, dinv, X, width, W, bias=None, act=ACT_NONE, src_index=None, out_rows=None, N=None,
                    split_out=False):
    """One fused GCN layer (aggregate-first, feature width <= 128): act((Â·X[src_index])[out_rows]·W^T + bias) with
    the A operand gathered in-kernel.  W = bf16 (hi, lo) planes.  Raises FitgnnError (EUNSUP) for ineligible shapes."""
    w_hi, w_lo = W
    N = w_hi.shape[0] if N is None else N
    n_out = out_rows.numel() if out_rows is not None else rowptr.numel() - 1
    if split_out:
        out = (torch.empty(n_out, N, dtype=torch.bfloat16, device=X.device),
               torch.empty(n_out, N, dtype=torch.bfloat16, device=X.device))
        y, ylo, ldy = out[0], out[1], N
    else:
        out = torch.empty(n_out, N, dtype=torch.float32, device=X.device)
        y, ylo, ldy = out, None, N
    check(lib().fitgnn_gcn_layer_fused(ptr(rowptr), ptr(col), ptr(dinv), ptr(X), X.stride(0), width, ptr(src_index),
                                       ptr(out_rows), n_out, ptr(w_hi), ptr(w_lo), w_hi.stride(0), ptr(bias), N, act,
                                       ptr(y), ptr(ylo), ldy, stream_ptr()))
    return out


def gcn_transform_aggregate(A, W, bias, act, agg_desc, dinv, K=None, N=None, split_out=True, defer_row_scale=False):
    """G = Â_local·act(A·W^T + bias) on a group-aligned pack: the next layer's propagate fused into the tensor-core
    transform's epilogue.  A, W = bf16 (hi, lo) planes; agg_desc / dinv come from Pack.aligned()."""
    (a_hi, a_lo), (w_hi, w_lo) = A, W
    assert a_hi.dtype == torch.bfloat16 and w_hi.dtype == torch.bfloat16 and agg_desc.dtype == torch.int64
    M = a_hi.shape[0]
    K = a_hi.shape[1] if K is None else K
    N = w_hi.shape[0] if N is None else N
    assert agg_desc.numel() == M and dinv.numel() == M
    if split_out:
        out = (torch.empty(M, N, dtype=torch.bfloat16, device=a_hi.device),
               torch.empty(M, N, dtype=torch.bfloat16, device=a_hi.device))
        y, ylo, ldy = out[0], out[1], N
    else:
        out = torch.empty(M, N, dtype=torch.float32, device=a_hi.device)
        y, ylo, ldy = out, None, N
    check(lib().fitgnn_gcn_transform_aggregate(ptr(a_hi), ptr(a_lo), a_hi.stride(0), ptr(w_hi), ptr(w_lo), w_hi.stride(0),
                                               ptr(bias), M, K, N, act, ptr(agg_desc), ptr(dinv), int(defer_row_scale),
                                               ptr(y), ptr(ylo), ldy, stream_ptr()))
    return out


def gemm_head_rows(A, W, bias, act, head, row_map, out, K=None, N=None):
    """head(act(A·W^T + bias)) with output row m written to out[row_map[m]] (skipped when row_map[m] < 0)."""
    (a_hi, a_lo), (w_hi, w_lo) = A, W
    M = a_hi.shape[0]
    K = a_hi.shape[1] if K is None else K
    N = w_hi.shape[0] if N is None else N
    assert row_map.dtype == torch.int32 and row_map.numel() == M and out.dtype == torch.float32
    check(lib().fitgnn_gemm_head_rows(ptr(a_hi), ptr(a_lo), a_hi.stride(0), ptr(w_hi), ptr(w_lo), w_hi.stride(0), ptr(bias),
                                      M, K, N, act, head, ptr(row_map), ptr(out), out.stride(0), stream_ptr()))
    return out


def gemm_head_rows_peers(A, W, bias, act, head, row_map, peer_ptrs, ldy, K=None, N=None):
    """gemm_head_rows with every output row stored to peer_ptrs[p] + row_map[m]*ldy floats for each p (raw device
    addresses of the same slot in every rank's gather buffer, see dist.PeerGather): the all-gather fused into the head."""
    (a_hi, a_lo), (w_hi, w_lo) = A, W
    M = a_hi.shape[0]
    K = a_hi.shape[1] if K is None else K
    N = w_hi.shape[0] if N is None else N
    assert row_map.dtype == torch.int32 and row_map.numel() == M
    bases = (C.c_void_p * len(peer_ptrs))(*[C.c_void_p(int(p)) for p in peer_ptrs])
    check(lib().fitgnn_gemm_head_rows_peers(ptr(a_hi), ptr(a_lo), a_hi.stride(0), ptr(w_hi), ptr(w_lo), w_hi.stride(0),
                                            ptr(bias), M, K, N, act, head, ptr(row_map), bases, len(peer_ptrs), ldy,
                                            stream_ptr()))


def gcn_forward(pack, X, state_dict, head=HEAD_LOG_SOFTMAX, precision=GEMM_BF16X3, out=None):
    """The whole forward over one pack in ONE C call (include/fitgnn.h fitgnn_gcn_forward): conv stack + lt1 + head on the
    core rows, classic schedule.  pack: fitgnn_b200.pack.Pack; X: [n_src, F] fp32 feature table; state_dict: the
    reference's keys (conv.{i}.lin.weight, conv.{i}.bias, lt1.weight, lt1.bias).  Returns [n_core, C]."""
    from ._lib import WeightsStruct
    if "conv.0.lin_l.weight" in state_dict:
        raise NotImplementedError("fitgnn_gcn_forward runs GCNConv models only; run a SAGEConv model with PackedForward")
    dev = X.device
    L = len({k.split(".")[1] for k in state_dict if k.startswith("conv.")})
    f32 = dict(dtype=torch.float32, device=dev)
    cw = [state_dict[f"conv.{i}.lin.weight"].detach().to(**f32).contiguous() for i in range(L)]
    cb = [state_dict[f"conv.{i}.bias"].detach().to(**f32).contiguous() for i in range(L)]
    lw = state_dict["lt1.weight"].detach().to(**f32).contiguous()
    lb = state_dict["lt1.bias"].detach().to(**f32).contiguous()
    F_, H, Cn = cw[0].shape[1], cw[0].shape[0], lw.shape[0]
    assert X.dtype == torch.float32 and X.shape[0] == pack.n_src and X.shape[1] >= F_
    if X.shape[1] % 4 != 0 or not X.is_contiguous():
        Xp = torch.zeros(X.shape[0], pad4(X.shape[1]), **f32)
        Xp[:, : X.shape[1]].copy_(X)
        X = Xp
    wptr = (C.c_void_p * L)(*[C.c_void_p(t.data_ptr()) for t in cw])
    bptr = (C.c_void_p * L)(*[C.c_void_p(t.data_ptr()) for t in cb])
    ws_ = WeightsStruct(L, F_, H, Cn, wptr, bptr, lw.data_ptr(), lb.data_ptr())
    st = pack.struct()
    nbytes = lib().fitgnn_gcn_forward_workspace_bytes(C.byref(st), C.byref(ws_), precision)
    if nbytes == 0:
        raise _lib.FitgnnError(f"fitgnn_gcn_forward_workspace_bytes: {_lib.last_error()}")
    ws = _ws(nbytes, dev)
    if out is None:
        out = torch.empty(pack.n_core, pad4(Cn), **f32)
    check(lib().fitgnn_gcn_forward(C.byref(st), ptr(X), X.stride(0), C.byref(ws_), head, precision, ptr(out), out.stride(0),
                                   ptr(ws), ws.numel(), stream_ptr()))
    return out[:, :Cn]


# ----------------------------------------------------------------------------------------- training path
def gemm_tn(G, A):
    """dW [out, in] = G[R, out]^T · A[R, in] on the tensor cores (fitgnn_gemm_tn): the weight gradient of a linear layer."""
    assert G.dtype == torch.float32 and A.dtype == torch.float32 and G.shape[0] == A.shape[0] and G.dim() == 2 and A.dim() == 2
    if G.stride(1) != 1:
        G = G.contiguous()
    if A.stride(1) != 1:
        A = A.contiguous()
    R, out, inn = G.shape[0], G.shape[1], A.shape[1]
    dW = torch.empty(out, inn, dtype=torch.float32, device=G.device)
    if R == 0:
        return dW.zero_()
    ws = _ws(lib().fitgnn_gemm_tn_workspace_bytes(R, out, inn), G.device)
    # row-strided operands (column slices of wider matrices) are fine: the kernel takes the row pitch
    check(lib().fitgnn_gemm_tn(C.c_void_p(G.data_ptr()), G.stride(0), C.c_void_p(A.data_ptr()), A.stride(0), R, out, inn,
                               ptr(dW), dW.stride(0), ptr(ws), ws.numel(), stream_ptr()))
    return dW


def dropout(X, p, seed, offset=0, out=None):
    """X * mask / (1 - p) with the Philox mask of (seed, offset) (fitgnn_dropout; F.dropout of network.py:33)."""
    assert X.dtype == torch.float32 and X.dim() == 2 and X.stride(1) == 1
    if out is None:
        out = torch.empty(X.shape, dtype=torch.float32, device=X.device)
    check(lib().fitgnn_dropout(C.c_void_p(X.data_ptr()), X.stride(0), X.shape[0], X.shape[1], float(p), int(seed), int(offset),
                               ptr(out), out.stride(0), stream_ptr()))
    return out


def elu_dropout_backward(G, H, act=ACT_ELU, p=0.0, seed=0, offset=0):
    """G * mask/(1-p) * act'(H): gradient w.r.t. the pre-activation of x = dropout(act(z)) given H = act(z)."""
    assert G.dtype == torch.float32 and H.dtype == torch.float32 and G.shape == H.shape and G.dim() == 2
    G = G if G.stride(1) == 1 else G.contiguous()
    H = H if H.stride(1) == 1 else H.contiguous()
    out = torch.empty(G.shape, dtype=torch.float32, device=G.device)
    check(lib().fitgnn_elu_dropout_backward(C.c_void_p(G.data_ptr()), G.stride(0), C.c_void_p(H.data_ptr()), H.stride(0),
                                            G.shape[0], G.shape[1], act, float(p),
                                            int(seed), int(offset), ptr(out), out.stride(0), stream_ptr()))
    return out


def adam_step(param, grad, exp_avg, exp_avg_sq, step, lr=0.01, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
    """One fused Adam step over flat fp32 buffers (fitgnn_adam_step, torch.optim.Adam semantics)."""
    n = param.numel()
    assert all(t.dtype == torch.float32 and t.is_contiguous() and t.numel() == n for t in (param, grad, exp_avg, exp_avg_sq))
    check(lib().fitgnn_adam_step(ptr(param), ptr(grad), ptr(exp_avg), ptr(exp_avg_sq), n, float(lr), float(betas[0]),
                                 float(betas[1]), float(eps), float(weight_decay), int(step), stream_ptr()))


def raw_tensor(ptr_value, shape, device, owner=None):
    """fp32 torch view of a raw device address (library-allocated or peer-mapped memory); `owner` is kept alive by it."""
    class _Raw:
        pass

    raw = _Raw()
    raw.__cuda_array_interface__ = {"shape": tuple(int(d) for d in shape), "typestr": "<f4", "data": (int(ptr_value), False),
                                    "version": 2, "strides": None}
    t = torch.as_tensor(raw, device=torch.device(device))
    t._fitgnn_owner = owner
    return t


class PeerBuffer:
    """A zero-filled device buffer allocated by the library (cudaMalloc) and exportable as a CUDA IPC handle.
    `.tensor(shape)` views it as a torch fp32 tensor; `.handle` is the 64-byte blob the other ranks `open`."""

    def __init__(self, nbytes, device):
        self.nbytes, self.device = int(nbytes), torch.device(device)
        p, h = C.c_void_p(), C.create_string_buffer(64)
        with torch.cuda.device(self.device):
            check(lib().fitgnn_peer_alloc(self.nbytes, C.byref(p), h))
        self.ptr, self.handle, self.opened = p.value, h.raw, {}

    def tensor(self, shape, dtype=torch.float32):
        n = 1
        for d in shape:
            n *= int(d)
        assert n * torch.empty(0, dtype=dtype).element_size() <= self.nbytes

        return raw_tensor(self.ptr, shape, self.device, owner=self)  # the tensor must not outlive the allocation

    def open_peer(self, rank, handle):
        """Map another rank's buffer into this process; returns its device address here."""
        p = C.c_void_p()
        with torch.cuda.device(self.device):
            check(lib().fitgnn_peer_open(handle, C.byref(p)))
        self.opened[rank] = p.value
        return p.value

    def close(self):
        for p in self.opened.values():
            lib().fitgnn_peer_close(C.c_void_p(p))
        self.opened = {}
        if self.ptr:
            lib().fitgnn_peer_free(C.c_void_p(self.ptr))
            self.ptr = None


def split_bf16(X, cols=None, ldo=None):
    """fp32 [rows, cols] -> bf16 (hi, lo) planes [rows, ldo] with zero-filled padding columns."""
    rows = X.shape[0]
    cols = X.shape[1] if cols is None else cols
    ldo = cols if ldo is None else ldo
    hi = torch.empty(rows, ldo, dtype=torch.bfloat16, device=X.device)
    lo = torch.empty(rows, ldo, dtype=torch.bfloat16, device=X.device)
    check(lib().fitgnn_split_bf16(ptr(X), X.stride(0), rows, cols, ptr(hi), ptr(lo), ldo, stream_ptr()))
    return hi, lo


def _segment_pool_raw(X, rows, seg_ptr, pool, width=None):
    width = X.shape[1] if width is None else width
    n_seg = seg_ptr.numel() - 1
    out = torch.empty(n_seg, width, dtype=torch.float32, device=X.device)
    check(lib().fitgnn_segment_pool(ptr(X), X.stride(0), width, ptr(rows), ptr(seg_ptr), n_seg, pool, ptr(out),
                                    out.stride(0), stream_ptr()))
    return out


class _SegmentPoolFn(torch.autograd.Function):
    """global_max_pool / global_mean_pool (network.py:93,131,164,202) with their gradients: mean spreads g / count over the
    segment's rows, max routes g to the first row attaining the maximum (index plumbing in torch)."""

    @staticmethod
    def forward(ctx, X, rows, seg_ptr, pool):
        Xc = X.detach().contiguous()
        out = _segment_pool_raw(Xc, rows, seg_ptr, pool)
        ctx.pool, ctx.n_rows = pool, X.shape[0]
        ctx.save_for_backward(Xc, rows if rows is not None else torch.empty(0, dtype=torch.int32, device=X.device), seg_ptr, out)
        ctx.has_rows = rows is not None
        return out

    @staticmethod
    def backward(ctx, g):
        X, rows, seg_ptr, out = ctx.saved_tensors
        n_seg = seg_ptr.numel() - 1
        counts = (seg_ptr[1:] - seg_ptr[:-1]).long()
        R = int(seg_ptr[-1])
        sel = rows.long() if ctx.has_rows else torch.arange(R, device=X.device)
        seg_of = torch.repeat_interleave(torch.arange(n_seg, device=X.device), counts)
        g = g.contiguous()
        if ctx.pool == POOL_MEAN:
            gr = g[seg_of] / counts[seg_of].clamp(min=1).to(g.dtype)[:, None]
        else:
            xr = X[sel]
            idx = torch.arange(R, device=X.device)[:, None].expand(R, X.shape[1])
            cand = torch.where(xr == out[seg_of], idx, torch.full_like(idx, R))
            first = torch.full((n_seg, X.shape[1]), R, dtype=torch.long, device=X.device)
            first.scatter_reduce_(0, seg_of[:, None].expand(R, X.shape[1]), cand, reduce="amin")
            gr = torch.where(idx == first[seg_of], g[seg_of], torch.zeros((), dtype=g.dtype, device=g.device))
        gx = torch.zeros(ctx.n_rows, X.shape[1], dtype=g.dtype, device=g.device)
        gx.index_add_(0, sel, gr)
        return gx, None, None, None


# ----------------------------------------------------------------------------------------- fp16 hidden state (opt-in)
def split_f16(X, cols=None, ldo=None, lo=True):
    """fp32 [rows, cols] -> fp16 (hi, lo) planes [rows, ldo] (lo=False: (hi, None)); padding columns zero."""
    rows = X.shape[0]
    cols = X.shape[1] if cols is None else cols
    ldo = cols if ldo is None else ldo
    hi = torch.empty(rows, ldo, dtype=torch.float16, device=X.device)
    lo_t = torch.empty(rows, ldo, dtype=torch.float16, device=X.device) if lo else None
    check(lib().fitgnn_split_f16(ptr(X), X.stride(0), rows, cols, ptr(hi), ptr(lo_t), ldo, stream_ptr()))
    return hi, lo_t


def gemm_f16(A, W, bias=None, act=ACT_NONE, head=HEAD_IDENTITY, row_scale=None, out_f16=False, row_map=None, out=None,
             K=None, N=None):
    """head(act(row_scale * (A·W^T) + bias)) with A ONE fp16 plane [M, K] and W = fp16 (hi, lo) planes (FITGNN_GEMM_FP16X2);
    W = (hi, None): ONE fp16 weight plane, one MMA per product.
    out_f16: the result as one fp16 plane (the next product's A); row_map: rows scattered into `out` (fp32, required then)."""
    w_hi, w_lo = W
    assert A.dtype == torch.float16 and w_hi.dtype == torch.float16
    M = A.shape[0]
    K = A.shape[1] if K is None else K
    N = w_hi.shape[0] if N is None else N
    if out is None:
        assert row_map is None
        out = torch.empty(M, N if (out_f16 or N % 4 == 0) else pad4(N), dtype=torch.float16 if out_f16 else torch.float32,
                          device=A.device)
    check(lib().fitgnn_gemm_f16(ptr(A), A.stride(0), ptr(w_hi), ptr(w_lo), w_hi.stride(0), ptr(row_scale), ptr(bias), M, K, N,
                                act, head, ptr(out), out.stride(0), int(out_f16), ptr(row_map), stream_ptr()))
    return out


def gemm_f16_2seg(A0, A1, W, K0, bias=None, act=ACT_NONE, out_f16=False, a0_cols=None, K=None, N=None):
    """act(A·W^T + bias) with A = [A0 | 0 | A1]: k-blocks [0, K0) read the fp16 plane A0 (a0_cols columns, zero beyond), the
    rest the fp16 plane A1 (K - K0 columns; K defaults to K0 + A1's width) (fitgnn_gemm_f16_2seg).  W = fp16 (hi, lo) planes or
    (hi, None).  out_f16: the result as one fp16 plane."""
    w_hi, w_lo = W
    assert A0.dtype == torch.float16 and A1.dtype == torch.float16 and w_hi.dtype == torch.float16
    M = A0.shape[0]
    assert A1.shape[0] == M
    a0_cols = A0.shape[1] if a0_cols is None else a0_cols
    K = K0 + A1.shape[1] if K is None else K
    N = w_hi.shape[0] if N is None else N
    out = torch.empty(M, N if (out_f16 or N % 4 == 0) else pad4(N), dtype=torch.float16 if out_f16 else torch.float32,
                      device=A0.device)
    check(lib().fitgnn_gemm_f16_2seg(ptr(A0), A0.stride(0), a0_cols, K0, ptr(A1), A1.stride(0), ptr(w_hi), ptr(w_lo),
                                     w_hi.stride(0), ptr(bias), M, K, N, act, ptr(out), out.stride(0), int(out_f16), stream_ptr()))
    return out


def gemm_f16_head_rows_peers(A, W, bias, act, head, row_map, peer_ptrs, ldy, K=None, N=None):
    """gemm_head_rows_peers with A one fp16 plane and W = fp16 (hi, lo) planes."""
    w_hi, w_lo = W
    M = A.shape[0]
    K = A.shape[1] if K is None else K
    N = w_hi.shape[0] if N is None else N
    assert A.dtype == torch.float16 and row_map.dtype == torch.int32 and row_map.numel() == M
    bases = (C.c_void_p * len(peer_ptrs))(*[C.c_void_p(int(p)) for p in peer_ptrs])
    check(lib().fitgnn_gemm_f16_head_rows_peers(ptr(A), A.stride(0), ptr(w_hi), ptr(w_lo), w_hi.stride(0), ptr(bias), M, K, N, act,
                                                head, ptr(row_map), bases, len(peer_ptrs), ldy, stream_ptr()))


def gcn_transform_aggregate_f16(A, W, bias, act, agg_desc, dinv, K=None, N=None, defer_row_scale=False):
    """gcn_transform_aggregate whose result is ONE fp16 plane.  A = bf16 (hi, lo) planes with W = bf16 planes, or A = one
    fp16 plane with W = fp16 (hi, lo) planes.  agg_desc = None: the plain transform into an fp16 plane."""
    w_hi, w_lo = W
    in_f16 = not isinstance(A, tuple)
    a_hi, a_lo = (A, None) if in_f16 else A
    M = a_hi.shape[0]
    K = a_hi.shape[1] if K is None else K
    N = w_hi.shape[0] if N is None else N
    out = torch.empty(M, N, dtype=torch.float16, device=a_hi.device)
    check(lib().fitgnn_gcn_transform_aggregate_f16(int(in_f16), ptr(a_hi), ptr(a_lo), a_hi.stride(0), ptr(w_hi), ptr(w_lo),
                                                   w_hi.stride(0), ptr(bias), M, K, N, act, ptr(agg_desc), ptr(dinv),
                                                   int(defer_row_scale), ptr(out), out.stride(0), stream_ptr()))
    return out


def gcn_conv_aligned_f16(A, W, bias, act, agg_desc, dinv, K=None, N=None):
    """act(Â·(A·W^T) + bias) on a group-aligned pack in one kernel (fitgnn_gcn_conv_aligned_f16): A one fp16 plane, W fp16
    (hi, lo) planes or (hi, None); the result is one fp16 plane."""
    w_hi, w_lo = W
    assert A.dtype == torch.float16 and w_hi.dtype == torch.float16
    M = A.shape[0]
    K = A.shape[1] if K is None else K
    N = w_hi.shape[0] if N is None else N
    out = torch.empty(M, N, dtype=torch.float16, device=A.device)
    check(lib().fitgnn_gcn_conv_aligned_f16(ptr(A), A.stride(0), ptr(w_hi), ptr(w_lo), w_hi.stride(0), ptr(bias), M, K, N, act,
                                            ptr(agg_desc), ptr(dinv), ptr(out), out.stride(0), stream_ptr()))
    return out


def segment_pool(X, rows, seg_ptr, pool, width=None):
    """Segment max / mean over the selected rows (fitgnn_segment_pool); differentiable w.r.t. X when X requires grad."""
    if torch.is_grad_enabled() and X.requires_grad:
        assert width is None or width == X.shape[1]
        return _SegmentPoolFn.apply(X, rows, seg_ptr, pool)
    return _segment_pool_raw(X, rows, seg_ptr, pool, width)


# ----------------------------------------------------------------------------------------- projection
def group_by_part(part, k):
    assert part.dtype == torch.int32
    N = part.numel()
    members = torch.empty(N, dtype=torch.int32, device=part.device)
    member_ptr = torch.empty(k + 1, dtype=torch.int32, device=part.device)
    ws = _ws(lib().fitgnn_group_workspace_bytes(N, k), part.device)
    check(lib().fitgnn_group_by_part(ptr(part), N, k, ptr(members), ptr(member_ptr), ptr(ws), ws.numel(),
                                     stream_ptr()))
    return members, member_ptr


def project_features(members, member_ptr, cweight, X):
    """Xc = C·X with C given as (part -> members/member_ptr, cweight[N] float64)."""
    assert cweight.dtype == torch.float64 and X.dtype == torch.float32
    k = member_ptr.numel() - 1
    F = X.shape[1]
    Xc = torch.empty(k, F, dtype=torch.float32, device=X.device)
    check(lib().fitgnn_project_features(ptr(members), ptr(member_ptr), k, ptr(cweight), ptr(X), X.stride(0), F,
                                        ptr(Xc), Xc.stride(0), stream_ptr()))
    return Xc


def project_adj(edge_index, part, k, want_rowptr=True):
    """Pattern of P_bin·A·P_bin^T minus its diagonal: (row int64, col int64, cnt int32, rowptr int32)."""
    ei = edge_index.contiguous()
    E = ei.shape[1]
    N = part.numel()
    ws = _ws(lib().fitgnn_project_adj_workspace_bytes(E), ei.device)
    nnz = C.c_int64(0)
    check(lib().fitgnn_project_adj_plan(ptr(ei), E, N, ptr(part), k, ptr(ws), ws.numel(), C.byref(nnz), stream_ptr()))
    n = nnz.value
    row = torch.empty(max(n, 1), dtype=torch.int64, device=ei.device)[:n]
    col = torch.empty(max(n, 1), dtype=torch.int64, device=ei.device)[:n]
    cnt = torch.empty(max(n, 1), dtype=torch.int32, device=ei.device)[:n]
    rowptr = torch.empty(k + 1, dtype=torch.int32, device=ei.device) if want_rowptr else None
    check(lib().fitgnn_project_adj_fill(ptr(ws), ws.numel(), k, ptr(row), ptr(col), ptr(cnt), ptr(rowptr),
                                        stream_ptr()))
    return row, col, cnt, rowptr
