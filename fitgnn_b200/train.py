"""Training steps on the pack (SURVEY §8f rank 1): the reference's GD semantics — one forward over ALL subgraphs, one loss
over all selected nodes, one backward, one optimiser step (node_train_Gs_GD run.py:177-215; node_train_Gc run.py:26-37
is the same call on the coarsened graph) — with the conv forward/backward on libfitgnn_b200 (autograd.GCNConvFn), and
the gradient all-reduce the multi-GPU path needs (one flat buffer per step)."""
from __future__ import annotations

import torch

from .autograd import CsrPair, SageCsr
from .pack import Pack


def pack_csr(pack: Pack) -> CsrPair:
    return CsrPair(pack.rowptr, pack.col, pack.dinv)


def pack_sage_csr(pack: Pack) -> SageCsr:
    """The pack's CSR without its self entries (the SAGEConv root, not a neighbour; as PackedForward's skip_self).  Built
    with a sort: pass it to forward_on_pack / train_step_Gs as `csr` to reuse it across steps."""
    rp = pack.rowptr.long()
    row = torch.repeat_interleave(torch.arange(pack.n_rows, device=rp.device), rp[1:] - rp[:-1])
    col = pack.col.long()
    keep = col != row
    return SageCsr.from_edge_index(torch.stack([col[keep], row[keep]]).contiguous(), pack.n_rows)


def forward_on_pack(model, pack: Pack, X, csr: CsrPair | SageCsr | None = None):
    """Differentiable forward of a node model (fitgnn_b200.nn.Classify_node / Regress_node, GCNConv or SAGEConv layers)
    over every row of the pack; X is the de-duplicated feature table ([N (+k), F]).  Returns [n_rows, C] with grad_fn."""
    from . import ops
    from .autograd import gcn_conv, sage_conv
    sage = hasattr(model.conv[0], "lin_l")
    csr = csr or (pack_sage_csr(pack) if sage else pack_csr(pack))
    x = X[pack.gid.long()]
    for i in range(model.num_layers):  # conv -> ELU -> dropout (network.py:31-33, p = 0.5 in train mode), one fused operator
        c, p = model.conv[i], 0.5 if model.training else 0.0
        if sage:
            x = sage_conv(x, c.lin_l.weight, c.lin_l.bias, c.lin_r.weight, csr, ops.ACT_ELU, p)
        else:
            x = gcn_conv(x, c.lin.weight, c.bias, csr, ops.ACT_ELU, p)
    y = model.lt1(x)
    return torch.nn.functional.log_softmax(y, dim=1) if model._head == "log_softmax" else y


def allreduce_gradients(model, world_size: int, group=None, local_count=None):
    """One all-reduce of the flat gradient buffer per optimiser step.

    local_count given (the GD semantics of node_train_Gs_GD, run.py:199-204 — ONE loss over all selected nodes of all
    subgraphs): every rank has back-propagated the SUM of its rows' losses; the gradients and the row counts are summed
    over the ranks in the same buffer and divided by the global count, which is exactly the gradient of the mean loss
    over all rows, however unevenly the rows are spread (a rank without rows contributes zeros).  Returns the global count.
    local_count None: plain average of the ranks' gradients (each rank back-propagated its own mean loss)."""
    grads = [p.grad for p in model.parameters() if p.grad is not None]
    if world_size <= 1:
        if local_count is not None:
            n = float(local_count)
            for g in grads:
                g /= max(n, 1.0)
            return n
        return None
    import torch.distributed as dist
    extra = [] if local_count is None else [torch.as_tensor([float(local_count)], dtype=grads[0].dtype, device=grads[0].device)]
    flat = torch.cat([g.reshape(-1) for g in grads] + extra)
    dist.all_reduce(flat, group=group)
    n = None
    if local_count is None:
        flat /= world_size
    else:
        n = float(flat[-1])
        flat = flat[:-1] / max(n, 1.0)
    off = 0
    for g in grads:
        g.copy_(flat[off: off + g.numel()].view_as(g))
        off += g.numel()
    return n


class FusedAdam:
    """torch.optim.Adam over ONE flat buffer: the model's parameters are re-pointed at views of a single fp32 buffer and
    so are their gradients, so that (a) the optimiser step is one kernel (fitgnn_adam_step) instead of one per parameter
    and (b) the multi-GPU gradient all-reduce runs on the flat gradient buffer in place — no gather / scatter copies.
    Same update rule and defaults as the reference's optimiser (torch.optim.Adam(lr, weight_decay), run.py:341)."""

    def __init__(self, params, lr=0.01, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        self.params = [p for p in params if p.requires_grad]
        assert self.params and all(p.is_cuda and p.dtype == torch.float32 for p in self.params)
        n = sum(p.numel() for p in self.params)
        dev = self.params[0].device
        self.flat = torch.empty(n, dtype=torch.float32, device=dev)
        self.grad = torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros_like(self.flat)
        self.exp_avg_sq = torch.zeros_like(self.flat)
        off = 0
        for p in self.params:
            k = p.numel()
            self.flat[off: off + k].copy_(p.data.reshape(-1))
            p.data = self.flat[off: off + k].view_as(p)
            p.grad = self.grad[off: off + k].view_as(p)
            off += k
        self.lr, self.betas, self.eps, self.weight_decay, self.t = lr, betas, eps, weight_decay, 0

    def zero_grad(self, set_to_none=False):
        self.grad.zero_()
        off = 0
        for p in self.params:  # autograd accumulates in place as long as .grad is our view
            if p.grad is None or p.grad.data_ptr() != self.grad[off: off + 1].data_ptr():
                p.grad = self.grad[off: off + p.numel()].view_as(p)
            off += p.numel()

    def step(self):
        from . import ops
        off = 0
        for p in self.params:  # a gradient autograd replaced instead of accumulating into our view is copied in
            k = p.numel()
            if p.grad is not None and p.grad.data_ptr() != self.grad[off: off + 1].data_ptr():
                self.grad[off: off + k].copy_(p.grad.reshape(-1))
            off += k
        self.t += 1
        ops.adam_step(self.flat, self.grad, self.exp_avg, self.exp_avg_sq, self.t, self.lr, self.betas, self.eps, self.weight_decay)


def allreduce_flat_(flat_grad, world_size: int, group=None, local_count=None):
    """allreduce_gradients on a flat gradient buffer, in place (FusedAdam): one collective, no copies; the row count rides
    in a second tiny all-reduce."""
    n = float(local_count) if local_count is not None else None
    if world_size > 1:
        import torch.distributed as dist
        dist.all_reduce(flat_grad, group=group)
        if local_count is None:
            flat_grad /= world_size
            return None
        cnt = torch.tensor([float(local_count)], device=flat_grad.device)
        dist.all_reduce(cnt, group=group)
        n = float(cnt)
    if n is not None:
        flat_grad /= max(n, 1.0)
    return n


def train_step_Gs(model, pack: Pack, X, y, train_mask, optimizer, loss_fn=None, world_size=1, csr=None, group=None):
    """node_train_Gs_GD (run.py:177-215): ONE loss over every train node of every subgraph, backward, step.
    y / train_mask are global ([N]); extra / cluster rows never contribute (Pack.split_masks).  With world_size > 1 the
    pack is this rank's shard: the rank back-propagates the SUM of its rows' losses and `allreduce_gradients` divides by the
    global row count, so the step equals the single-process one for any distribution of the train rows over the ranks
    (including ranks that hold none).  loss_fn(out_rows, targets) must be mean-reduced (default: nll_loss).
    Returns the mean loss over all ranks' rows."""
    model.train()
    optimizer.zero_grad()
    out = forward_on_pack(model, pack, X, csr)
    rows = pack.split_masks(train_mask)
    tgt = y.to(out.device)[pack.gid.long().clamp(max=y.numel() - 1)]
    loss_fn = loss_fn or torch.nn.functional.nll_loss
    n_local = int(rows.sum())
    if n_local > 0:
        loss_sum = loss_fn(out[rows], tgt[rows]) * n_local
    else:
        loss_sum = out.sum() * 0.0  # keeps the graph (zero gradients) so that every rank joins the all-reduce
    loss_sum.backward()
    total = torch.stack([loss_sum.detach().float(), torch.tensor(float(n_local), device=out.device)])
    if world_size > 1:
        import torch.distributed as dist
        dist.all_reduce(total, group=group)
    if isinstance(optimizer, FusedAdam):
        allreduce_flat_(optimizer.grad, world_size, group, n_local)
    else:
        allreduce_gradients(model, world_size, group, local_count=n_local)
    optimizer.step()
    return float(total[0] / total[1].clamp(min=1.0))
