"""CPU: the SAGEConv reference restatement, the drop-in class's parameters and options, and its refusal of CPU tensors."""
import argparse

import pytest
import torch

from tests import sage_oracle as so


def test_sage_oracle_known_answer_fp64():
    """Path 0-1-2-3 (both directions), node 4 isolated, the edge 0->1 twice, a self-loop edge 2->2; x = [1, 2, 4, 8, 16],
    W_l = [[1]], b_l = [0.5], W_r = [[10]]:
        node 0: in-edges from 1            mean 2            out = 2 + 0.5 + 10      = 12.5
        node 1: from 0, 0 (duplicate), 2   mean (1+1+4)/3=2  out = 2 + 0.5 + 20      = 22.5
        node 2: from 1, 2 (self loop), 3   mean (2+4+8)/3    out = 14/3 + 0.5 + 40
        node 3: from 2                     mean 4            out = 4 + 0.5 + 80      = 84.5
        node 4: none                       mean 0            out = 0 + 0.5 + 160     = 160.5"""
    ei = torch.tensor([[0, 1, 1, 2, 2, 3, 0, 2], [1, 0, 2, 1, 3, 2, 1, 2]])
    x = torch.tensor([[1.0], [2.0], [4.0], [8.0], [16.0]], dtype=torch.float64)
    out = so.sage_conv(x, ei, torch.tensor([[1.0]]), torch.tensor([0.5]), torch.tensor([[10.0]]))
    want = torch.tensor([[12.5], [22.5], [14.0 / 3.0 + 40.5], [84.5], [160.5]], dtype=torch.float64)
    assert out.dtype == torch.float64
    torch.testing.assert_close(out, want, rtol=0, atol=1e-12)


def _args(layer_name="SAGEConv", num_classes=4):
    return argparse.Namespace(num_layers1=2, num_features=12, hidden=32, num_classes=num_classes, layer_name=layer_name)


def test_sage_state_dict_keys_match_pyg():
    import fitgnn_b200
    conv = fitgnn_b200.nn.SAGEConv(12, 32)
    assert set(conv.state_dict()) == {"lin_l.weight", "lin_l.bias", "lin_r.weight"}
    assert conv.lin_l.weight.shape == (32, 12) and conv.lin_r.weight.shape == (32, 12) and conv.lin_r.bias is None
    sd = so.init_state_dict(12, 32, 4, seed=1)
    for cls in (fitgnn_b200.Classify_node, fitgnn_b200.Classify_graph_gc, fitgnn_b200.Classify_graph_gs):
        m = cls(_args())
        assert set(m.state_dict()) == set(sd)
        m.load_state_dict(sd)
    sd_r = dict(sd, **{"lt1.weight": sd["lt1.weight"][:1], "lt1.bias": sd["lt1.bias"][:1]})
    for cls in (fitgnn_b200.Regress_node, fitgnn_b200.Regress_graph_gc, fitgnn_b200.Regress_graph_gs):
        cls(_args()).load_state_dict(sd_r)
    fitgnn_b200.Net1(12, 32, 2, 4, layer_name="SAGEConv").load_state_dict(sd)
    fitgnn_b200.Net2(12, 32, 2, layer_name="SAGEConv").load_state_dict(sd_r)
    for name in ("GATConv", "GINConv"):
        with pytest.raises(NotImplementedError):
            fitgnn_b200.Classify_node(_args(name))


def test_sage_options():
    import fitgnn_b200
    fitgnn_b200.nn.SAGEConv(4, 8, aggr="mean", normalize=False, root_weight=True, project=False, bias=True)
    for kw in (dict(aggr="max"), dict(normalize=True), dict(root_weight=False), dict(project=True), dict(bias=False),
               dict(cached=True)):
        with pytest.raises(TypeError):
            fitgnn_b200.nn.SAGEConv(4, 8, **kw)


def test_sage_cpu_tensors_are_rejected():
    import fitgnn_b200
    conv = fitgnn_b200.nn.SAGEConv(4, 8)
    with pytest.raises(RuntimeError):
        conv(torch.zeros(3, 4), torch.zeros(2, 0, dtype=torch.long))
    ops, Err = fitgnn_b200.ops, fitgnn_b200._lib.FitgnnError
    rp, col = torch.zeros(4, dtype=torch.int32), torch.zeros(0, dtype=torch.int32)
    with pytest.raises(Err):
        ops.csr_raw_from_coo(torch.zeros(2, 0, dtype=torch.long), 3)
    with pytest.raises(Err):
        ops.spmm_mean_concat(rp, col, torch.zeros(3, 4))
    with pytest.raises(Err):
        ops.spmm_mean_root(rp, col, torch.zeros(3, 8), 4)


def test_engine_refuses_sage_where_it_is_not_built():
    """The one-call C forward and the streamed forward are GCN-only: a SAGE state_dict gets NotImplementedError before any
    device work."""
    import fitgnn_b200
    sd = so.init_state_dict(12, 32, 4)
    with pytest.raises(NotImplementedError):
        fitgnn_b200.ops.gcn_forward(None, torch.zeros(1, 12), sd)
    with pytest.raises(NotImplementedError):
        fitgnn_b200.StreamedForward(None, sd)
