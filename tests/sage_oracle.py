"""CPU restatement (torch-CPU) of PyG SAGEConv as `SAGEConv(in_channels, out_channels)` builds it (aggr='mean',
normalize=False, root_weight=True, project=False, bias=True) and of the reference models (network.py) with
layer_name='SAGEConv'.  Test infrastructure only.

PARITY: PyG is not installed and the reference tree has no SAGE layer of its own, so nothing here is pinned against
executable reference code: the rule below restates the published PyG operator and is anchored on the hand-computed
known-answer case of tests/test_sage_host.py ("parity unpinned", like gcn_norm's duplicate / self-loop rules).

    out_i = lin_l( mean_{e=(j->i)} x_j ) + lin_r(x_i)      lin_l with bias, lin_r without
    messages flow edge_index[0] -> edge_index[1]; no self loop is added (one in edge_index is an ordinary neighbour);
    duplicate edges count once per occurrence in the sum and the count; no in-edges -> mean 0.
"""
import torch
import torch.nn.functional as F

from oracle import fitgnn_oracle as fo


def sage_conv(x, edge_index, w_l, b_l, w_r):
    """PyG SAGEConv.forward in x's dtype (pass float64 tensors for the fp64 reference)."""
    ei = torch.as_tensor(edge_index).long()
    n = x.shape[0]
    src, dst = ei[0], ei[1]
    s = torch.zeros(n, x.shape[1], dtype=x.dtype).index_add_(0, dst, x[src])
    cnt = torch.zeros(n, dtype=x.dtype).index_add_(0, dst, torch.ones(dst.numel(), dtype=x.dtype))
    mean = s / cnt.clamp(min=1).view(-1, 1)
    return F.linear(mean, w_l.to(x.dtype), b_l.to(x.dtype)) + F.linear(x, w_r.to(x.dtype))


def conv_stack(sd, x, edge_index):
    """network.py:30-33 with the SAGE layer; eval: dropout = identity."""
    for i in range(fo.num_layers_of(sd)):
        x = F.elu(sage_conv(x, edge_index, sd[f"conv.{i}.lin_l.weight"], sd[f"conv.{i}.lin_l.bias"],
                            sd[f"conv.{i}.lin_r.weight"]))
    return x


def classify_node(sd, x, edge_index):
    return F.log_softmax(F.linear(conv_stack(sd, x, edge_index), sd["lt1.weight"], sd["lt1.bias"]), dim=1)


def regress_node(sd, x, edge_index):
    return F.linear(conv_stack(sd, x, edge_index), sd["lt1.weight"], sd["lt1.bias"])


def graph_gs_forward(sd, set_gs, batch_tensor, task):
    rows = [conv_stack(sd, g["x"].float(), g["edge_index"])[g["mask"]] for gs in set_gs for g in gs]
    bt = batch_tensor.to(torch.int64)
    x = fo._pool(torch.cat(rows, 0), bt, "max" if task == "graph_cls" else "mean", int(bt.max()) + 1)
    x = F.linear(x, sd["lt1.weight"], sd["lt1.bias"])
    return F.softmax(x, dim=1) if task == "graph_cls" else x


def graph_gc_forward(sd, x, edge_index, batch, task):
    x = fo._pool(conv_stack(sd, x, edge_index), batch, "max" if task == "graph_cls" else "mean", int(batch.max()) + 1)
    x = F.linear(x, sd["lt1.weight"], sd["lt1.bias"])
    return F.softmax(x, dim=1) if task == "graph_cls" else x


def init_state_dict(num_features, hidden, num_classes, num_layers=2, seed=0, bias_scale=0.1):
    """Seeded SAGE parameters with PyG's keys (lin_l.weight, lin_l.bias, lin_r.weight) and the head lt1.*."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    dims = [num_features] + [hidden] * num_layers
    for i in range(num_layers):
        a = (1.0 / dims[i]) ** 0.5
        sd[f"conv.{i}.lin_l.weight"] = (torch.rand(dims[i + 1], dims[i], generator=g) * 2 - 1) * a
        sd[f"conv.{i}.lin_l.bias"] = (torch.rand(dims[i + 1], generator=g) * 2 - 1) * bias_scale
        sd[f"conv.{i}.lin_r.weight"] = (torch.rand(dims[i + 1], dims[i], generator=g) * 2 - 1) * a
    a = (1.0 / hidden) ** 0.5
    sd["lt1.weight"] = (torch.rand(num_classes, hidden, generator=g) * 2 - 1) * a
    sd["lt1.bias"] = (torch.rand(num_classes, generator=g) * 2 - 1) * a
    return sd
