"""GPU: SAGEConv on the B200 path — raw CSR builder, mean-aggregation kernels (both forms) against fp64, the drop-in
operator and the six model classes against the torch-CPU restatement (tests/sage_oracle.py), the whole-pack engine
against the drop-in model, gradients and training steps, and the refusals of the GCN-only paths."""
import argparse

import numpy as np
import pytest
import torch

from oracle import fitgnn_oracle as fo
from tests import golden_io as gio
from tests import sage_oracle as so

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
MODES = ("none", "extra", "cluster")


@pytest.fixture(scope="module")
def fg():
    import fitgnn_b200
    return fitgnn_b200


def close(got, want, rtol=1e-3):
    """max |got - want| <= rtol * max|want| (as the GCN parity tests: 1e-3 relative for fp32 logits)."""
    got = np.asarray(got.detach().cpu().double() if torch.is_tensor(got) else got, dtype=np.float64)
    want = np.asarray(want.detach().cpu().double() if torch.is_tensor(want) else want, dtype=np.float64)
    assert got.shape == want.shape, (got.shape, want.shape)
    scale = max(1e-12, float(np.abs(want).max())) if want.size else 1.0
    err = float(np.abs(got - want).max()) if want.size else 0.0
    assert err <= rtol * scale, (err, scale)


def graph_with_everything(n, e, seed, hub=None, hub_deg=0):
    """Random directed edges with self loops and duplicates; nodes >= n - 3 isolated; optionally one row with hub_deg
    in-edges."""
    rng = np.random.default_rng(seed)
    m = n - 3
    src, dst = rng.integers(0, m, e), rng.integers(0, m, e)
    src = np.concatenate([src, src[:5], np.arange(4)])   # duplicates and explicit self loops
    dst = np.concatenate([dst, dst[:5], np.arange(4)])
    if hub is not None:
        src = np.concatenate([src, rng.integers(0, m, hub_deg)])
        dst = np.concatenate([dst, np.full(hub_deg, hub)])
    return np.stack([src, dst]).astype(np.int64)


def csr_numpy(ei, n):
    src, dst = ei
    order = np.lexsort((src, dst))
    rowptr = np.concatenate([[0], np.cumsum(np.bincount(dst, minlength=n))])
    return rowptr, src[order]


def mean_fp64(rowptr, col, X, src_index=None, out_rows=None, skip_self=False, scale=None):
    X = np.asarray(X, np.float64)
    src = np.arange(X.shape[0]) if src_index is None else np.asarray(src_index)
    rows = np.arange(len(rowptr) - 1) if out_rows is None else np.asarray(out_rows)
    agg = np.zeros((len(rows), X.shape[1]))
    root = np.zeros((len(rows), X.shape[1]))
    for k, r in enumerate(rows):
        cs = np.asarray(col[rowptr[r]:rowptr[r + 1]])
        if skip_self:
            cs = cs[cs != r]
        if len(cs):
            if scale is None:
                agg[k] = X[src[cs]].mean(0)
            else:
                agg[k] = (np.asarray(scale, np.float64)[cs, None] * X[src[cs]]).sum(0)
        root[k] = X[src[r]]
    return agg, root


def planes_to_f32(t):
    hi, lo = t
    return hi.float() + lo.float()


# ------------------------------------------------------------------------------------------ raw CSR
@pytest.mark.parametrize("n,e", [(1, 0), (10, 0), (50, 200), (5000, 40000)])
def test_csr_raw_matches_numpy(fg, n, e):
    ei = graph_with_everything(n + 3, e, seed=n) if n > 1 else np.zeros((2, 0), dtype=np.int64)
    nn = n + 3 if n > 1 else n
    rowptr, col = fg.ops.csr_raw_from_coo(torch.tensor(ei, device=DEV), nn)
    want_rp, want_col = csr_numpy(ei, nn)
    assert np.array_equal(rowptr.cpu().numpy(), want_rp) and np.array_equal(col.cpu().numpy(), want_col)


# ------------------------------------------------------------------------------------------ kernels vs fp64
@pytest.mark.parametrize("width,half", [(4, 8), (12, 16), (36, 40), (100, 104), (128, 128), (512, 512), (1028, 1032)])
@pytest.mark.parametrize("skip_self", [False, True])
def test_mean_concat_matches_fp64(fg, width, half, skip_self):
    n = 700
    ei = graph_with_everything(n, 3000, seed=width, hub=5, hub_deg=1000)  # one row of ~1,000 entries
    rowptr, col = fg.ops.csr_raw_from_coo(torch.tensor(ei, device=DEV), n)
    rp, cl = rowptr.cpu().numpy(), col.cpu().numpy()
    g = torch.Generator().manual_seed(width)
    n_src = 900
    X = torch.randn(n_src, width, generator=g)
    src_index = torch.randperm(n_src, generator=g)[:n].to(torch.int32)
    out_rows = torch.tensor(np.r_[5, np.arange(n - 1, -1, -3)], dtype=torch.int32)  # hub, isolated rows, reversed order
    Xd, sd_, od = X.to(DEV), src_index.to(DEV), out_rows.to(DEV)
    agg, root = mean_fp64(rp, cl, X.numpy(), src_index.numpy(), out_rows.numpy(), skip_self)
    scale = float(np.abs(X.numpy()).max())
    for split in (False, True):
        y = fg.ops.spmm_mean_concat(rowptr, col, Xd, width, half, sd_, None, skip_self, od, split=split)
        y = (planes_to_f32(y) if split else y).cpu().numpy()
        assert y.shape == (len(out_rows), 2 * half)
        tol = (2 ** -15 if split else 2e-6) * scale  # bf16 hi/lo budget / fp32 rounding of the sum and the division
        assert np.abs(y[:, :width] - agg).max() <= tol
        assert np.abs(y[:, half:half + width] - root).max() <= tol
        assert not y[:, width:half].any() and not y[:, half + width:].any()  # pad columns written as zeros
    # determinism and variant invariance: bit-identical across calls, row selections and gid indirection
    a = fg.ops.spmm_mean_concat(rowptr, col, Xd, width, half, sd_, None, skip_self, od)
    b = fg.ops.spmm_mean_concat(rowptr, col, Xd, width, half, sd_, None, skip_self, od)
    assert torch.equal(a, b)
    full = fg.ops.spmm_mean_concat(rowptr, col, Xd[sd_.long()].contiguous(), width, half, None, None, skip_self)
    assert torch.equal(full[od.long()], a)


@pytest.mark.parametrize("width", [4, 16, 64, 512])
@pytest.mark.parametrize("skip_self", [False, True])
def test_mean_root_matches_fp64(fg, width, skip_self):
    n = 600
    ei = graph_with_everything(n, 2500, seed=width + 1, hub=7, hub_deg=1000)
    rowptr, col = fg.ops.csr_raw_from_coo(torch.tensor(ei, device=DEV), n)
    rp, cl = rowptr.cpu().numpy(), col.cpu().numpy()
    g = torch.Generator().manual_seed(width)
    n_src = 650
    Z = torch.randn(n_src, 2 * width + 4, generator=g)  # [Z_l | Z_r | spare]: root_off = width, pitch wider than needed
    bias = torch.randn(width, generator=g) * 0.1
    src_index = torch.randperm(n_src, generator=g)[:n].to(torch.int32)
    out_rows = torch.tensor(np.r_[7, np.arange(0, n, 2)], dtype=torch.int32)
    agg, _ = mean_fp64(rp, cl, Z.numpy()[:, :width], src_index.numpy(), out_rows.numpy(), skip_self)
    root = Z.numpy()[src_index.numpy()[out_rows.numpy()], width:2 * width].astype(np.float64)
    pre = agg + root + bias.numpy()
    want = np.where(pre > 0, pre, np.expm1(pre))
    scale = float(np.abs(Z.numpy()).max())
    for split in (False, True):
        y = fg.ops.spmm_mean_root(rowptr, col, Z.to(DEV), width, width, src_index.to(DEV), None, skip_self, bias.to(DEV),
                                  fg.ops.ACT_ELU, out_rows.to(DEV), split=split)
        y = (planes_to_f32(y) if split else y).cpu().numpy()
        assert np.abs(y - want).max() <= (2 ** -15 if split else 4e-6) * scale
    a = fg.ops.spmm_mean_root(rowptr, col, Z.to(DEV), width, width, src_index.to(DEV), None, skip_self, bias.to(DEV),
                              fg.ops.ACT_ELU, out_rows.to(DEV))
    b = fg.ops.spmm_mean_root(rowptr, col, Z.to(DEV), width, width, src_index.to(DEV), None, skip_self, bias.to(DEV),
                              fg.ops.ACT_ELU, out_rows.to(DEV))
    assert torch.equal(a, b)


def test_mean_src_scale_is_the_transposed_mean(fg):
    """src_scale: weighted sum, no division — on the reversed CSR with 1/count it is Mᵀ (checked against the dense
    operator in fp64)."""
    n, width = 300, 20
    ei = graph_with_everything(n, 1500, seed=9)
    csr = fg.autograd.SageCsr.from_edge_index(torch.tensor(ei, device=DEV), n)
    rp_t, col_t, inv = csr.transposed()
    M = np.zeros((n, n))
    for s, t in ei.T:
        M[t, s] += 1.0
    cnt = M.sum(1, keepdims=True)
    M = np.divide(M, cnt, out=np.zeros_like(M), where=cnt > 0)
    G = torch.randn(n, width, generator=torch.Generator().manual_seed(1))
    y = fg.ops.spmm_mean_concat(rp_t, col_t, G.to(DEV), width, width, None, inv).cpu().numpy()
    assert np.abs(y[:, :width] - M.T @ G.numpy()).max() <= 1e-5 * float(np.abs(G.numpy()).max())
    assert np.array_equal(y[:, width:], G.numpy())


def test_mean_rejects_bad_shapes(fg):
    rp, col = fg.ops.csr_raw_from_coo(torch.zeros(2, 0, dtype=torch.long, device=DEV), 4)
    X = torch.zeros(4, 8, device=DEV)
    with pytest.raises(fg._lib.FitgnnError):
        fg.ops.spmm_mean_concat(rp, col, X, 8, 4)   # half < width
    with pytest.raises(fg._lib.FitgnnError):
        fg.ops.spmm_mean_concat(rp, col, X, 6, 8)   # width not a multiple of 4
    with pytest.raises(fg._lib.FitgnnError):
        fg.ops.spmm_mean_root(rp, col, X, 8, 4)     # root half past the row
    with pytest.raises(fg._lib.FitgnnError):
        fg.ops.csr_raw_from_coo(torch.tensor([[0, 5], [1, 1]], device=DEV), 4)  # node id out of range


# ------------------------------------------------------------------------------------------ drop-in operator
@pytest.mark.parametrize("fin,fout", [(20, 64), (13, 32), (100, 16), (300, 64)])  # aggregate-first / transform-first
def test_sageconv_matches_oracle(fg, fin, fout):
    n = 400
    ei = torch.tensor(graph_with_everything(n, 2000, seed=fin))
    g = torch.Generator().manual_seed(fin)
    x = torch.randn(n, fin, generator=g)
    conv = fg.nn.SAGEConv(fin, fout)
    with torch.no_grad():
        conv.lin_l.bias.uniform_(-0.3, 0.3)
    want = torch.nn.functional.elu(so.sage_conv(x.double(), ei, conv.lin_l.weight.detach(), conv.lin_l.bias.detach(),
                                                conv.lin_r.weight.detach()))
    conv = conv.to(DEV)
    for precision in ("bf16x3", "fp32"):
        old = fg.nn.set_precision(precision)
        try:
            with torch.no_grad():
                out = conv(x.to(DEV), ei.to(DEV), act=fg.ops.ACT_ELU)
                plain = conv(x.to(DEV), ei.to(DEV))
        finally:
            fg.nn.set_precision(old)
        close(out, want)
        close(plain, so.sage_conv(x.double(), ei, *(t.detach().cpu() for t in (conv.lin_l.weight, conv.lin_l.bias,
                                                                                 conv.lin_r.weight))))


def test_sage_and_gcn_csr_caches_are_separate(fg):
    ei = torch.tensor([[0, 1, 2, 2], [1, 2, 0, 2]], device=DEV)
    x = torch.randn(3, 8, device=DEV)
    gcn, sage = fg.GCNConv(8, 8).to(DEV), fg.nn.SAGEConv(8, 8).to(DEV)
    with torch.no_grad():
        gcn(x, ei); s1 = sage(x, ei); gcn(x, ei); s2 = sage(x, ei)
    assert torch.equal(s1, s2)
    close(s1, so.sage_conv(x.cpu().double(), ei.cpu(), *(t.detach().cpu() for t in (sage.lin_l.weight, sage.lin_l.bias,
                                                                                      sage.lin_r.weight))))


# ------------------------------------------------------------------------------------------ model classes on fixtures
def _ns(F, H, C):
    return argparse.Namespace(num_layers1=2, num_features=F, hidden=H, num_classes=C, layer_name="SAGEConv")


def test_node_models_on_fixture(fg):
    d = gio.load("node_small")
    ref = gio.subgraphs(d, "extra_sub")
    x, ei = fo.collate(ref[:128])
    H, C = int(d["hidden"]), int(d["n_classes"])
    sd = so.init_state_dict(x.shape[1], H, C, seed=3)
    sd_r = dict(sd, **{"lt1.weight": sd["lt1.weight"][:1].clone(), "lt1.bias": sd["lt1.bias"][:1].clone()})
    for cls, s, ref_fn in ((fg.Classify_node, sd, so.classify_node), (fg.Regress_node, sd_r, so.regress_node)):
        m = cls(_ns(x.shape[1], H, C)); m.load_state_dict(s); m = m.to(DEV).eval()
        with torch.no_grad():
            close(m(x.to(DEV), ei.to(DEV)), ref_fn(s, x, ei))
    net1 = fg.Net1(x.shape[1], H, 2, C, layer_name="SAGEConv"); net1.load_state_dict(sd)
    net2 = fg.Net2(x.shape[1], H, 2, layer_name="SAGEConv"); net2.load_state_dict(sd_r)
    with torch.no_grad():
        close(net1.to(DEV).eval()(x.to(DEV), ei.to(DEV)), so.classify_node(sd, x, ei))
        close(net2.to(DEV).eval()(x.to(DEV), ei.to(DEV)), so.regress_node(sd_r, x, ei))


@pytest.mark.parametrize("case,task", [("graph_small", "graph_reg"), ("graph_small", "graph_cls"),
                                       ("graph_cls_small", "graph_cls")])
def test_graph_models_on_fixture(fg, case, task):
    from oracle.ref_shims import Data
    d = gio.load(case)
    n_g = int(d["n_kept"])
    subs = [gio.subgraphs(d, f"g{g}_sub") for g in range(n_g)]
    F = subs[0][0]["x"].shape[1]
    H, C = int(d["hidden"]), (1 if task == "graph_reg" else 3)
    sd = so.init_state_dict(F, H, C, seed=4)
    set_gs = [[Data(x=torch.tensor(s["x"]), edge_index=torch.tensor(s["edge_index"]), mask=torch.tensor(s["mask"]))
               for s in gs] for gs in subs]
    bt = torch.tensor(d["batch_tensor"])
    gs_cls, gc_cls = ((fg.Regress_graph_gs, fg.Regress_graph_gc) if task == "graph_reg" else
                      (fg.Classify_graph_gs, fg.Classify_graph_gc))
    m = gs_cls(_ns(F, H, C)); m.load_state_dict(sd); m = m.to(DEV).eval()
    want = so.graph_gs_forward(sd, [[dict(x=g.x, edge_index=g.edge_index, mask=g.mask) for g in gs] for gs in set_gs], bt, task)
    with torch.no_grad():
        close(m(set_gs, bt), want)
    gx = torch.tensor(np.concatenate([d[f"g{g}_gc_x"] for g in range(n_g)])).float()
    off, eis = 0, []
    for g in range(n_g):
        eis.append(d[f"g{g}_gc_edge"] + off); off += d[f"g{g}_gc_x"].shape[0]
    gei = torch.tensor(np.concatenate(eis, 1))
    gc = Data(x=gx.to(DEV), edge_index=gei.to(DEV), batch=torch.tensor(d["gc_batch"]).to(DEV))
    mgc = gc_cls(_ns(F, H, C)); mgc.load_state_dict(sd); mgc = mgc.to(DEV).eval()
    with torch.no_grad():
        close(mgc(gc), so.graph_gc_forward(sd, gx, gei, torch.tensor(d["gc_batch"]), task))


# ------------------------------------------------------------------------------------------ whole-pack engine
def _golden_pack(fg, d, mode):
    from tests.test_gpu_parity import global_features, golden_partition
    comps, cos, partition = golden_partition(fg, d, mode)
    pack = fg.build_pack(torch.tensor(d["edge_index"], device=DEV), torch.tensor(partition.part), partition.k, mode)
    return pack, global_features(d, mode, cos, comps, partition).to(DEV)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("hidden", [32, 8])  # F = 12: aggregate-first layer 0, and transform-first (F > hidden)
def test_packed_forward_matches_dropin_model(fg, mode, hidden):
    d = gio.load("node_small")
    pack, X = _golden_pack(fg, d, mode)
    F, C = d["x"].shape[1], int(d["n_classes"])
    sd = so.init_state_dict(F, hidden, C, seed=6)
    ref = gio.subgraphs(d, mode + "_sub")
    xc, eic = fo.collate(ref)
    model = fg.Classify_node(_ns(F, hidden, C)); model.load_state_dict(sd); model = model.to(DEV).eval()
    with torch.no_grad():
        full = model(xc.to(DEV), eic.to(DEV))
    tm = np.concatenate([r["test_mask"] for r in ref])
    want = full[torch.tensor(tm, device=DEV)]
    close(want, so.classify_node(sd, xc, eic)[torch.tensor(tm)])
    for precision in ("bf16x3", "fp32", "fp16"):  # fp16 is not built for SAGE: it runs bf16x3
        out, ids = fg.infer.node_infer_Gs(sd, pack, X, torch.tensor(d["test_mask"]), precision=precision)
        close(out, want)
    core = fg.PackedForward(pack, sd, rows="core")(X)
    q = ids[:: max(1, ids.numel() // 20)]
    pq = fg.infer.per_query(sd, pack, X, q)
    lookup = torch.full((pack.n_nodes,), -1, dtype=torch.long, device=DEV)
    lookup[pack.core_gid.long()] = torch.arange(pack.n_core, device=DEV)
    close(pq, core[lookup[q]], rtol=1e-5)
    with pytest.raises(ValueError):
        fg.PackedForward(pack, sd, fuse_aggregate=True)


def test_graph_level_Gs_matches_dropin_model(fg):
    d = gio.load("graph_cls_small")
    n_g = int(d["n_kept"])
    subs = [gio.subgraphs(d, f"g{g}_sub") for g in range(n_g)]
    flat = [s for gs in subs for s in gs]
    pack, Xp, _ = fg.pack_from_subgraph_list(flat, device=DEV)
    graph_of_sub = torch.tensor(np.concatenate([[g] * len(gs) for g, gs in enumerate(subs)]))
    F, H = flat[0]["x"].shape[1], int(d["hidden"])
    sd = so.init_state_dict(F, H, 3, seed=8)
    got = fg.infer.graph_level_Gs(sd, pack, Xp, graph_of_sub, task="graph_cls")
    set_gs = [[dict(x=torch.tensor(s["x"]), edge_index=torch.tensor(s["edge_index"]), mask=torch.tensor(s["mask"]))
               for s in gs] for gs in subs]
    close(got, so.graph_gs_forward(sd, set_gs, torch.tensor(d["batch_tensor"]), "graph_cls"))


def test_sage_refusals(fg):
    d = gio.load("node_small")
    pack, X = _golden_pack(fg, d, "none")
    sd = so.init_state_dict(d["x"].shape[1], 32, int(d["n_classes"]))
    with pytest.raises(NotImplementedError):
        fg.StreamedForward(pack, sd)
    with pytest.raises(NotImplementedError):
        fg.ops.gcn_forward(pack, X, sd)
    with pytest.raises(NotImplementedError):  # the peer-store head of the multi-GPU path (dist.PeerGather)
        fg.PackedForward(pack, sd)(X, peer_ptrs=[0])


# ------------------------------------------------------------------------------------------ training
@pytest.mark.parametrize("fin,fout", [(12, 32), (100, 16)])  # aggregate-first / transform-first
def test_sageconv_gradients_match_oracle(fg, fin, fout):
    n = 500
    ei = torch.tensor(graph_with_everything(n, 2500, seed=fout))
    g = torch.Generator().manual_seed(fin)
    x = torch.rand(n, fin, generator=g)
    conv = fg.nn.SAGEConv(fin, fout)
    with torch.no_grad():
        conv.lin_l.bias.uniform_(-0.1, 0.1)
    wl, bl, wr = (t.detach().clone() for t in (conv.lin_l.weight, conv.lin_l.bias, conv.lin_r.weight))
    tgt = torch.rand(n, fout, generator=g)
    torch.manual_seed(11)
    seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    mask = (fg.ops.dropout(torch.ones(n, fout, device=DEV), 0.5, seed) != 0).cpu()
    xo, wlo, blo, wro = (t.clone().requires_grad_(True) for t in (x, wl, bl, wr))
    yo = torch.nn.functional.elu(so.sage_conv(xo, ei, wlo, blo, wro)) * mask * 2.0
    lo = ((yo - tgt) ** 2).sum()
    lo.backward()
    conv = conv.to(DEV)
    for precision in ("bf16x3", "fp32"):
        old = fg.nn.set_precision(precision)
        try:
            conv.zero_grad()
            xg = x.to(DEV).requires_grad_(True)
            torch.manual_seed(11)
            out = conv(xg, ei.to(DEV), act=fg.ops.ACT_ELU, dropout_p=0.5)
            close(out, yo)
            loss = ((out - tgt.to(DEV)) ** 2).sum()
            loss.backward()
        finally:
            fg.nn.set_precision(old)
        close(loss, lo)
        close(conv.lin_l.weight.grad, wlo.grad)
        close(conv.lin_l.bias.grad, blo.grad)
        close(conv.lin_r.weight.grad, wro.grad)
        close(xg.grad, xo.grad)


def test_train_step_Gs_follows_the_oracle(fg):
    """Three train_step_Gs steps (one loss over every train row of the pack, FusedAdam) on a SAGE model against a torch-CPU
    Adam loop on the oracle over the collated subgraphs.  Dropout is switched off on both sides (the model stays in eval
    mode) so the runs are comparable."""
    d = gio.load("node_small")
    pack, X = _golden_pack(fg, d, "extra")
    ref = gio.subgraphs(d, "extra_sub")
    xc, eic = fo.collate(ref)
    yc = torch.tensor(np.concatenate([r["y"] for r in ref])).long()
    tmc = torch.tensor(np.concatenate([r["train_mask"] for r in ref]))
    F, H, C = d["x"].shape[1], 32, int(d["n_classes"])
    sd = so.init_state_dict(F, H, C, seed=12)
    model = fg.Classify_node(_ns(F, H, C)); model.load_state_dict(sd); model = model.to(DEV)
    model.eval()
    model.train = lambda mode=True: model  # keep eval mode (no dropout) through train_step_Gs's model.train()
    opt = fg.train.FusedAdam(model.parameters(), lr=0.01, weight_decay=0.0005)
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    opt_o = torch.optim.Adam(params.values(), lr=0.01, weight_decay=0.0005)
    csr = fg.train.pack_sage_csr(pack)
    for _ in range(3):
        loss = fg.train.train_step_Gs(model, pack, X, torch.tensor(d["y"]), torch.tensor(d["train_mask"]), opt, csr=csr)
        opt_o.zero_grad()
        lo = torch.nn.functional.nll_loss(so.classify_node(params, xc, eic)[tmc], yc[tmc])
        lo.backward(); opt_o.step()
        close(torch.tensor(loss), lo.detach())
    for k, v in model.state_dict().items():
        close(v, params[k], rtol=2e-3)
