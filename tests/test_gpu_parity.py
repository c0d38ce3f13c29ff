"""GPU parity tests: the CUDA path, called through the C ABI (fitgnn_b200.ops -> libfitgnn_b200.so), against the
oracle and the reference-generated golden fixtures.  Integer / index results are compared bit-exactly; fp32
results within the tolerance BASELINE.json states (1e-3 relative), written out below as RTOL."""
import numpy as np
import pytest
import torch

from oracle import fitgnn_oracle as fo
from tests import golden_io as gio

pytestmark = pytest.mark.gpu

RTOL = 1e-3  # north_star: "within 1e-3 relative for fp32 logits"
MODES = ("none", "extra", "cluster")


def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def fg():
    import fitgnn_b200
    return fitgnn_b200


def assert_close(got, want, rtol=RTOL, atol_scale=1e-2):
    """|got - want| <= rtol * |want| + rtol * atol_scale * max|want|  (elementwise 1e-3 relative, with an absolute
    floor of 1e-5 * max|want| for entries near a zero crossing)."""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, (got.shape, want.shape)
    scale = max(1.0, float(np.abs(want).max())) if want.size else 1.0
    err = np.abs(got - want)
    tol = rtol * np.abs(want) + atol_scale * rtol * scale
    assert (err <= tol).all(), f"max err {err.max():.3e} (rel-to-max {err.max() / scale:.3e})"


# ------------------------------------------------------------------------------------------ primitives
@pytest.mark.parametrize("n", [0, 1, 2, 255, 4096, 4097, 100_003, 1_500_000])
@pytest.mark.parametrize("bits", [13, 40, 64])
def test_radix_sort_matches_torch(fg, n, bits):
    g = torch.Generator(device="cuda").manual_seed(n + bits)
    hi = 2 ** min(bits, 62)
    keys = torch.randint(0, hi, (n,), generator=g, device=dev(), dtype=torch.int64)
    if bits == 64 and n:
        keys = keys | (torch.randint(0, 2, (n,), generator=g, device=dev(), dtype=torch.int64) << 63)
    vals = torch.arange(n, device=dev(), dtype=torch.int32)
    k2, v2 = fg.ops.sort_u64(keys.clone(), vals.clone(), key_bits=bits)
    # unsigned order: flip the sign bit for the comparison sort
    want_k, perm = torch.sort(keys ^ (1 << 63) if bits == 64 else keys, stable=True)
    if bits == 64:
        want_k = want_k ^ (1 << 63)
    assert torch.equal(k2, want_k)
    assert torch.equal(v2, vals[perm])  # stable


@pytest.mark.parametrize("n", [1, 7, 2048, 2049, 5_000_000])
def test_scan_matches_cumsum(fg, n):
    g = torch.Generator(device="cuda").manual_seed(n)
    x = torch.randint(0, 5, (n,), generator=g, device=dev(), dtype=torch.int32)
    out = fg.ops.scan_i32(x, with_total=True)
    want = torch.zeros(n + 1, dtype=torch.int64, device=dev())
    want[1:] = torch.cumsum(x.long(), 0)
    assert torch.equal(out.long(), want)


# ------------------------------------------------------------------------------------------ a1 GCNConv
def random_coo(n, e, seed, self_loops=True, dups=True):
    rng = np.random.default_rng(seed)
    src = rng.integers(0, n, e)
    dst = rng.integers(0, n, e)
    if not self_loops:
        keep = src != dst
        src, dst = src[keep], dst[keep]
    if dups and e > 4:
        src = np.concatenate([src, src[:3]]); dst = np.concatenate([dst, dst[:3]])
    und_s, und_d = np.concatenate([src, dst]), np.concatenate([dst, src])
    return np.stack([und_s, und_d]).astype(np.int64)


@pytest.mark.parametrize("n,e", [(1, 0), (5, 0), (40, 90), (1000, 3000), (30000, 200000)])
def test_csr_matches_gcn_norm(fg, n, e):
    ei = random_coo(n, e, seed=n + e)
    rowptr, col, dinv = fg.ops.csr_from_coo(torch.tensor(ei, device=dev()), n)
    row_o, col_o, w_o = fo.gcn_norm(torch.tensor(ei), n)
    # oracle edges (source row_o -> target col_o) as a sorted multiset per target
    order = np.lexsort((row_o.numpy(), col_o.numpy()))
    assert np.array_equal(col.detach().cpu().numpy(), row_o.numpy()[order])
    assert np.array_equal(np.diff(rowptr.detach().cpu().numpy()), np.bincount(col_o.numpy(), minlength=n))
    deg = np.bincount(col_o.numpy(), minlength=n).astype(np.float32)
    assert np.array_equal(dinv.detach().cpu().numpy(), (1.0 / np.sqrt(deg)).astype(np.float32))


def test_gcnconv_known_answer(fg):
    conv = fg.GCNConv(2, 4).to(dev())  # KAT has 3 outputs; pad the 4th with zeros (out_channels % 4)
    with torch.no_grad():
        conv.lin.weight.copy_(torch.tensor([[1., 2.], [3., 4.], [5., 6.], [0., 0.]]))
        conv.bias.copy_(torch.tensor([0.1, -0.2, 0.3, 0.0]))
    ei = torch.tensor([[0, 1, 1, 2], [1, 0, 2, 1]], device=dev())
    x = torch.tensor([[1., 0.], [0., 1.], [1., 1.]], device=dev())
    out = conv(x, ei).detach().cpu().numpy()
    want = np.array([[1.4164965809, 2.9329931619, 5.2494897428],
                     [2.3996598285, 5.2158162380, 8.8319726474],
                     [2.4164965809, 4.9329931619, 8.2494897428]])
    np.testing.assert_allclose(out[:, :3], want, rtol=1e-6)
    np.testing.assert_array_equal(out[:, 3], 0)


def test_gcnconv_matches_reference_tree_gcn_layer(fg):
    """The CUDA GCNConv against outputs of the reference tree's OWN normalisation + dense GCN layer
    (Baselines/GCOND/models/mycheby.py:393-414, gcn.py:15-52; fixture tests/golden/gcn_norm_gcond.npz, generated by
    tests/golden/make_golden_gcn_norm.py from the unmodified reference files).  Tolerance 1e-3 relative (RTOL)."""
    from tests import golden_io as gio
    d = gio.load("gcn_norm_gcond")
    n, ei = int(d["n"]), torch.tensor(d["edge_index"], device=dev())
    conv = fg.GCNConv(d["X"].shape[1], d["out"].shape[1]).to(dev())
    with torch.no_grad():
        conv.lin.weight.copy_(torch.tensor(d["weight_in_out"]).t())
        conv.bias.copy_(torch.tensor(d["bias"]))
    out = conv(torch.tensor(d["X"], device=dev()), ei).detach().cpu().numpy()
    assert_close(out, d["out"])
    # the CSR the kernels run on reproduces the reference's normalised adjacency entry by entry
    rowptr, col, dinv = fg.ops.csr_from_coo(ei, n)
    rp, c, dv = rowptr.cpu().numpy(), col.cpu().numpy(), dinv.cpu().numpy().astype(np.float64)
    dense = np.zeros((n, n))
    rows = np.repeat(np.arange(n), np.diff(rp))
    np.add.at(dense, (rows, c), dv[rows] * dv[c])
    np.testing.assert_allclose(dense, d["A_norm"], rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("n,e,fin,fout", [(7, 0, 3, 4), (300, 900, 5, 8), (2000, 9000, 100, 512), (1500, 6000, 1433, 512),
                                          (900, 4000, 600, 512), (4000, 30000, 512, 512)])
def test_gcnconv_matches_fp64(fg, n, e, fin, fout):
    ei = random_coo(n, e, seed=fin)
    g = torch.Generator().manual_seed(fin + n)
    x = torch.rand(n, fin, generator=g)
    conv = fg.GCNConv(fin, fout)
    with torch.no_grad():
        conv.bias.uniform_(-0.1, 0.1)
    want = fo.gcn_conv_fp64(x.numpy(), ei, conv.lin.weight.detach().numpy(), conv.bias.detach().numpy())
    conv = conv.to(dev())
    out = conv(x.to(dev()), torch.tensor(ei, device=dev()))
    assert_close(out.detach().cpu().numpy(), want)
    out_elu = conv(x.to(dev()), torch.tensor(ei, device=dev()), act=fg.ops.ACT_ELU)
    assert_close(out_elu.detach().cpu().numpy(), np.where(want > 0, want, np.expm1(np.minimum(want, 0))))


@pytest.mark.parametrize("width", [4, 100, 128, 132, 256, 384, 512, 1024, 1540])
def test_spmm_widths_rows_and_split(fg, width):
    n, e = 3000, 12000
    ei = random_coo(n, e, seed=width)
    rowptr, col, dinv = fg.ops.csr_from_coo(torch.tensor(ei, device=dev()), n)
    g = torch.Generator().manual_seed(width)
    n_src = 700
    Xs = torch.randn(n_src, width, generator=g)
    src_index = torch.randint(0, n_src, (n,), generator=g, dtype=torch.int32)
    bias = torch.randn(width, generator=g)
    out_rows = torch.randperm(n, generator=g)[:777].to(torch.int32)
    A = fo.normalized_adjacency_dense(ei, n)
    want = A @ Xs.numpy().astype(np.float64)[src_index.numpy()] + bias.numpy()
    want = np.where(want > 0, want, np.expm1(np.minimum(want, 0)))[out_rows.numpy()]
    got = fg.ops.spmm_symnorm(rowptr, col, dinv, Xs.to(dev()), src_index=src_index.to(dev()), bias=bias.to(dev()),
                              act=fg.ops.ACT_ELU, out_rows=out_rows.to(dev()))
    assert_close(got.detach().cpu().numpy(), want)
    hi, lo = fg.ops.spmm_symnorm(rowptr, col, dinv, Xs.to(dev()), src_index=src_index.to(dev()), bias=bias.to(dev()),
                                 act=fg.ops.ACT_ELU, out_rows=out_rows.to(dev()), split=True)
    rec = hi.float().detach().cpu().numpy().astype(np.float64) + lo.float().detach().cpu().numpy()
    assert np.abs(rec - got.detach().cpu().numpy()).max() <= 2.0 ** -15 * max(1.0, np.abs(want).max())


def test_spmm_hub_rows(fg):
    # a star with 5000 leaves + a clique: hub row goes through the CTA-split path
    n = 5200
    leaves = np.arange(1, 5001)
    src = np.concatenate([np.zeros(5000, dtype=np.int64), leaves, np.arange(5001, 5199), np.arange(5002, 5200)])
    dst = np.concatenate([leaves, np.zeros(5000, dtype=np.int64), np.arange(5002, 5200), np.arange(5001, 5199)])
    ei = np.stack([src, dst])
    rowptr, col, dinv = fg.ops.csr_from_coo(torch.tensor(ei, device=dev()), n)
    X = torch.randn(n, 512, generator=torch.Generator().manual_seed(1))
    hubs = fg.ops.find_hubs(rowptr, None, n, hub_deg=256)
    assert hubs[1] == 1 and int(hubs[0][0]) == 0
    got = fg.ops.spmm_symnorm(rowptr, col, dinv, X.to(dev()), hubs=hubs)
    want = fo.normalized_adjacency_dense(ei, n) @ X.numpy().astype(np.float64)
    assert_close(got.detach().cpu().numpy(), want)
    got2 = fg.ops.spmm_symnorm(rowptr, col, dinv, X.to(dev()))  # same rows without the hub split
    assert_close(got2.detach().cpu().numpy(), want)


@pytest.mark.parametrize("M,K,N", [(1, 1, 1), (5, 3, 7), (129, 17, 130), (1000, 1433, 512), (777, 512, 47), (4096, 100, 512)])
def test_gemm_fp32(fg, M, K, N):
    g = torch.Generator().manual_seed(M + K + N)
    A, W, b = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g), torch.randn(N, generator=g)
    want = A.double() @ W.double().T + b.double()
    got = fg.ops.gemm_bias_act(A.to(dev()), W.to(dev()), b.to(dev()))
    assert_close(got.detach().cpu().numpy(), want.numpy(), rtol=1e-5, atol_scale=1.0)
    got = fg.ops.gemm_bias_act(A.to(dev()), W.to(dev()), b.to(dev()), act=fg.ops.ACT_ELU, head=fg.ops.HEAD_LOG_SOFTMAX)
    assert_close(got.detach().cpu().numpy(), torch.log_softmax(torch.nn.functional.elu(want), 1).numpy(), rtol=1e-4, atol_scale=1.0)


def test_segment_pool(fg):
    g = torch.Generator().manual_seed(0)
    X = torch.randn(500, 64, generator=g)
    rows = torch.randperm(500, generator=g)[:300].to(torch.int32)
    seg = torch.tensor([0, 10, 10, 57, 300], dtype=torch.int32)  # includes an empty segment
    for pool, fn in ((0, lambda t: t.max(0).values), (1, lambda t: t.mean(0))):
        got = fg.ops.segment_pool(X.to(dev()), rows.to(dev()), seg.to(dev()), pool).cpu()
        for i in range(4):
            sel = X[rows[seg[i]:seg[i + 1]].long()]
            want = fn(sel) if len(sel) else torch.zeros(64)
            np.testing.assert_allclose(got[i].numpy(), want.numpy(), rtol=1e-6, atol=1e-6)


# ------------------------------------------------------------------------------------------ golden helpers
def golden_partition(fg, d, mode):
    comps = gio.components(d, mode)
    cos = gio.coarsenings_for_oracle(d, mode, comps)
    C_list = [c["C"] if c is not None else None for c in cos]
    return comps, cos, fg.coarsen.partition_from_components(comps, C_list, int(d["n"]))


def global_features(d, mode, cos, comps, partition):
    """De-duplicated feature table: X for the nodes (+ C·X rows per cluster in cluster mode)."""
    x = torch.tensor(d["x"])
    if mode != "cluster":
        return x
    xc = np.zeros((partition.k, x.shape[1]), dtype=np.float32)
    for i, (comp, co) in enumerate(zip(comps, cos)):
        s0 = int(partition.sub_offset[i])
        if co is None:
            xc[s0] = d["x"][comp[0]]
        else:
            xc[s0:s0 + co["CX"].shape[0]] = co["CX"].astype(np.float32)
    return torch.cat([x, torch.tensor(xc)], 0)


# ------------------------------------------------------------------------------------------ a8-a11 builders
@pytest.mark.parametrize("case", ["node_small", "node_mid"])
@pytest.mark.parametrize("mode", MODES)
def test_pack_builder_bit_exact(fg, case, mode):
    d = gio.load(case)
    comps, cos, partition = golden_partition(fg, d, mode)
    n = int(d["n"])
    subs = fo.build_subgraphs(d["edge_index"], d["x"], d["y"], comps, cos, mode)
    assert np.array_equal(fo.partition_vector(subs, n), partition.part)  # a9: partition order == subgraph_list order
    want = fo.expected_pack(subs, n, mode)
    ei = torch.tensor(d["edge_index"], device=dev())
    pack = fg.build_pack(ei, torch.tensor(partition.part), partition.k, mode)
    for name in ("rowptr", "col", "gid", "sub_ptr", "core_rows", "is_core", "mask"):
        got = getattr(pack, name).detach().cpu().numpy()
        assert np.array_equal(got.astype(np.int64), np.asarray(want[name]).astype(np.int64)), name
    assert np.array_equal(pack.dinv.detach().cpu().numpy(), want["dinv"])
    # a13 split masks incl. the map_dict collision quirk
    ref = gio.subgraphs(d, mode + "_sub")
    for key in ("train", "val", "test"):
        got = pack.split_masks(torch.tensor(d[key + "_mask"])).detach().cpu().numpy()
        assert np.array_equal(got, np.concatenate([r[key + "_mask"] for r in ref])), key


@pytest.mark.parametrize("case", ["node_small", "node_mid"])
@pytest.mark.parametrize("mode", MODES)
def test_projection_bit_exact_and_gc_assembly(fg, case, mode):
    d = gio.load(case)
    comps, cos, partition = golden_partition(fg, d, mode)
    ei = torch.tensor(d["edge_index"], device=dev())
    X = torch.tensor(d["x"], device=dev())
    proj = fg.coarsen.project(ei, X, partition)
    row, col, cnt = fo.project_adj_pattern(d["edge_index"], partition.part.astype(np.int64), partition.k)
    assert np.array_equal(proj["ac_row"].detach().cpu().numpy(), row)
    assert np.array_equal(proj["ac_col"].detach().cpu().numpy(), col)
    assert np.array_equal(proj["ac_cnt"].detach().cpu().numpy(), cnt)
    xc = proj["Xc"].detach().cpu().numpy()
    for i, (comp, co) in enumerate(zip(comps, cos)):
        s0 = int(partition.sub_offset[i])
        if co is not None:  # bit-exact with scipy's float64 accumulation cast to fp32 (utils.py:738)
            assert np.array_equal(xc[s0:s0 + co["CX"].shape[0]], co["CX"].astype(np.float32))
    got = fg.coarsen.assemble_gc_classification(proj, partition, comps, ei, X, torch.tensor(d["y"]),
                                                torch.tensor(d["train_mask"]), torch.tensor(d["val_mask"]),
                                                int(d["n_classes"]))
    names = ("gc_x", "gc_train_y", "gc_train_m", "gc_val_y", "gc_val_m", "gc_edge")
    for g_, name in zip(got, names):
        assert np.array_equal(g_.detach().cpu().numpy(), d[f"{mode}_{name}"]), name


# ------------------------------------------------------------------------------------------ a14 collation of a subgraph_list
@pytest.mark.parametrize("case", ["node_small", "node_mid"])
@pytest.mark.parametrize("mode", MODES)
def test_pack_from_reference_subgraph_list(fg, case, mode):
    """pack_from_subgraph_list on the REFERENCE's own subgraph_list (golden fixture: utils.py:248-266 output, the list
    main.py:131-172 saves and G_DataLoader re-collates, run.py:336): the collated CSR equals the device pack builder's
    bit for bit, and the whole-list forward equals the reference model run batch by batch (oracle, 1e-3 relative)."""
    d = gio.load(case)
    comps, cos, partition = golden_partition(fg, d, mode)
    ref = gio.subgraphs(d, mode + "_sub")
    lp, Xp, node_ids = fg.pack_from_subgraph_list(ref, device=dev())
    pack = fg.build_pack(torch.tensor(d["edge_index"], device=dev()), torch.tensor(partition.part), partition.k, mode)
    assert (lp.n_rows, lp.nnz, lp.n_sub) == (pack.n_rows, pack.nnz, pack.n_sub)
    for name in ("rowptr", "col", "dinv", "sub_ptr", "mask"):
        assert torch.equal(getattr(lp, name), getattr(pack, name)), name
    assert torch.equal(lp.gid.long(), torch.arange(lp.n_rows, device=dev()))
    real = node_ids >= 0
    assert torch.equal(node_ids[real], pack.gid.long()[real]) and bool((pack.gid.long()[~real] >= int(d["n"])).all())
    X = global_features(d, mode, cos, comps, partition).to(dev())
    assert torch.equal(Xp, X[pack.gid.long()])  # the collated batch.x == the de-duplicated table gathered through gid
    sd = gio.state_dict(d) if case == "node_small" else fo.init_state_dict(d["x"].shape[1], int(d["hidden"]),
                                                                         int(d["n_classes"]), seed=2)
    for precision in ("fp32", "bf16x3"):
        out = fg.PackedForward(lp, sd, rows="all", precision=precision)(Xp)
        want = fo.node_infer_batched(sd, ref, [np.ones(r["x"].shape[0], dtype=bool) for r in ref], "node_cls", 128)
        assert_close(out.detach().cpu().numpy(), want.numpy())
    # accepts attribute-style objects (PyG Data) as well as dicts; rejects edges that leave their subgraph
    class Obj:  # noqa: E306
        def __init__(self, g):
            self.x, self.edge_index, self.mask = torch.tensor(g["x"]), torch.tensor(g["edge_index"]), torch.tensor(g["mask"])
    lp2, Xp2, ids2 = fg.pack_from_subgraph_list([Obj(g) for g in ref[:7]], device=dev())
    assert ids2 is None and lp2.n_sub == 7 and torch.equal(Xp2, Xp[: lp2.n_rows])
    bad = dict(x=np.zeros((2, Xp.shape[1]), np.float32), edge_index=np.array([[0], [2]]))
    with pytest.raises(ValueError):
        fg.pack_from_subgraph_list([bad], device=dev())


# ------------------------------------------------------------------------------------------ a2, a5, a6 forward
@pytest.mark.parametrize("case", ["node_small", "node_mid"])
@pytest.mark.parametrize("mode", MODES)
def test_packed_forward_matches_reference_outputs(fg, case, mode):
    d = gio.load(case)
    comps, cos, partition = golden_partition(fg, d, mode)
    ei = torch.tensor(d["edge_index"], device=dev())
    pack = fg.build_pack(ei, torch.tensor(partition.part), partition.k, mode)
    X = global_features(d, mode, cos, comps, partition).to(dev())
    if case == "node_small":
        sd = gio.state_dict(d)
    else:
        sd = fo.init_state_dict(d["x"].shape[1], int(d["hidden"]), int(d["n_classes"]), seed=2)
    out, ids = fg.infer.node_infer_Gs(sd, pack, X, torch.tensor(d["test_mask"]))
    ref = gio.subgraphs(d, mode + "_sub")
    want = fo.node_infer_batched(sd, ref, [r["test_mask"] for r in ref], "node_cls", 128)
    assert_close(out.detach().cpu().numpy(), want.numpy())
    if case == "node_small":  # the outputs of the reference's own network.py run
        assert_close(out.detach().cpu().numpy(), d[f"{mode}_test_out"])
    # a6 per-query: each queried node on its own subgraph only
    q = ids[:: max(1, ids.numel() // 20)]
    pq = fg.infer.per_query(sd, pack, X, q)
    lookup = {int(v): i for i, v in enumerate(ids.detach().cpu().numpy())}
    assert_close(pq.detach().cpu().numpy(), want.numpy()[[lookup[int(v)] for v in q.detach().cpu().numpy()]])


def test_model_classes_generic_path(fg):
    """Classify_node / Regress_node called like the reference does (x, edge_index of a collated batch),
    with a reference state_dict loaded by key."""
    import argparse
    d = gio.load("node_small")
    sd = gio.state_dict(d)
    ref = gio.subgraphs(d, "extra_sub")
    x, ei = fo.collate(ref[:128])
    args = argparse.Namespace(num_layers1=2, num_features=x.shape[1], hidden=int(d["hidden"]),
                              num_classes=int(d["n_classes"]), layer_name="GCNConv")
    model = fg.Classify_node(args)
    model.load_state_dict(sd)
    model = model.to(dev()).eval()
    out = model(x.to(dev()), ei.to(dev()))
    assert_close(out.detach().cpu().numpy(), fo.classify_node(sd, x, ei).numpy())
    net1 = fg.Net1(x.shape[1], int(d["hidden"]), 2, int(d["n_classes"]))
    net1.load_state_dict(sd)
    assert_close(net1.to(dev()).eval()(x.to(dev()), ei.to(dev())).detach().cpu().numpy(), out.detach().cpu().numpy(), rtol=1e-6)
    reg = fg.Regress_node(args)
    sd_r = dict(sd); sd_r["lt1.weight"] = sd["lt1.weight"][:1].clone(); sd_r["lt1.bias"] = sd["lt1.bias"][:1].clone()
    reg.load_state_dict(sd_r)
    assert_close(reg.to(dev()).eval()(x.to(dev()), ei.to(dev())).detach().cpu().numpy(), fo.regress_node(sd_r, x, ei).numpy())
    with pytest.raises(RuntimeError):
        model.eval()(x, ei.to(dev()))  # CPU tensor: no fallback


# ------------------------------------------------------------------------------------------ a3, a4 graph level
def test_graph_level_models_match_reference(fg):
    import argparse
    from oracle.ref_shims import Data
    d = gio.load("graph_small")
    sd = gio.state_dict(d)
    n_g = int(d["n_kept"])
    set_gs = []
    for g in range(n_g):
        set_gs.append([Data(x=torch.tensor(s["x"]), edge_index=torch.tensor(s["edge_index"]), mask=torch.tensor(s["mask"]))
                       for s in gio.subgraphs(d, f"g{g}_sub")])
    args = argparse.Namespace(num_layers1=2, num_features=1, hidden=int(d["hidden"]), num_classes=1, layer_name="GCNConv")
    model = fg.Regress_graph_gs(args)
    model.load_state_dict(sd)
    model = model.to(dev()).eval()
    pred = model(set_gs, torch.tensor(d["batch_tensor"]))
    assert_close(pred.detach().cpu().numpy(), d["pred_gs"])
    # Gc variant on the collated coarsened graphs
    gx = torch.tensor(np.concatenate([d[f"g{g}_gc_x"] for g in range(n_g)])).float()
    off, eis = 0, []
    for g in range(n_g):
        eis.append(d[f"g{g}_gc_edge"] + off); off += d[f"g{g}_gc_x"].shape[0]
    gc = Data(x=gx.to(dev()), edge_index=torch.tensor(np.concatenate(eis, 1)).to(dev()), batch=torch.tensor(d["gc_batch"]).to(dev()))
    model_gc = fg.Regress_graph_gc(args)
    model_gc.load_state_dict(sd)
    assert_close(model_gc.to(dev()).eval()(gc).detach().cpu().numpy(), d["pred_gc"])
    # classification heads (max pool + softmax) against the oracle
    sd_c = fo.init_state_dict(1, int(d["hidden"]), 3, seed=5)
    args_c = argparse.Namespace(num_layers1=2, num_features=1, hidden=int(d["hidden"]), num_classes=3, layer_name="GCNConv")
    mc = fg.Classify_graph_gs(args_c); mc.load_state_dict(sd_c)
    want = fo.graph_gs_forward(sd_c, [[dict(x=g.x, edge_index=g.edge_index, mask=g.mask) for g in gs] for gs in set_gs],
                               torch.tensor(d["batch_tensor"]), "graph_cls")
    assert_close(mc.to(dev()).eval()(set_gs, torch.tensor(d["batch_tensor"])).detach().cpu().numpy(), want.numpy())
    mgc = fg.Classify_graph_gc(args_c); mgc.load_state_dict(sd_c)
    want = fo.graph_gc_forward(sd_c, gx, torch.tensor(np.concatenate(eis, 1)), torch.tensor(d["gc_batch"]), "graph_cls")
    assert_close(mgc.to(dev()).eval()(gc).detach().cpu().numpy(), want.numpy())


def test_graph_classification_matches_reference_outputs(fg):
    """Classify_graph_gs / Classify_graph_gc on the GPU against the REFERENCE's own outputs (graph_cls_small.npz:
    coarsening_classification(task='graph_cls', cluster_node), colater, network.py:118-135 and :87-95 run unmodified)."""
    import argparse
    from oracle.ref_shims import Data
    d = gio.load("graph_cls_small")
    sd = gio.state_dict(d)
    n_g = int(d["n_kept"])
    set_gs = [[Data(x=torch.tensor(s["x"]), edge_index=torch.tensor(s["edge_index"]), mask=torch.tensor(s["mask"]))
               for s in gio.subgraphs(d, f"g{g}_sub")] for g in range(n_g)]
    args = argparse.Namespace(num_layers1=2, num_features=d["g0_x"].shape[1], hidden=int(d["hidden"]),
                              num_classes=int(d["n_classes"]), layer_name="GCNConv")
    model = fg.Classify_graph_gs(args)
    model.load_state_dict(sd)
    pred = model.to(dev()).eval()(set_gs, torch.tensor(d["batch_tensor"]))
    assert_close(pred.detach().cpu().numpy(), d["pred_gs"])
    gx = torch.tensor(np.concatenate([d[f"g{g}_gc_x"] for g in range(n_g)])).float()
    off, eis = 0, []
    for g in range(n_g):
        eis.append(d[f"g{g}_gc_edge"] + off); off += d[f"g{g}_gc_x"].shape[0]
    gc = Data(x=gx.to(dev()), edge_index=torch.tensor(np.concatenate(eis, 1)).to(dev()), batch=torch.tensor(d["gc_batch"]).to(dev()))
    model_gc = fg.Classify_graph_gc(args)
    model_gc.load_state_dict(sd)
    assert_close(model_gc.to(dev()).eval()(gc).detach().cpu().numpy(), d["pred_gc"])


# ------------------------------------------------------------------------------------------ config-shaped + properties
@pytest.mark.parametrize("mode", MODES)
def test_cora_shaped_config(fg, mode):
    """configs[0]: Cora-shaped synthetic, r = 0.3, 2-layer GCN hidden 512; pack and logits vs the oracle."""
    n, e_und, F, C, ratio = fg.synth.SHAPES["cora"]
    ei = fg.synth.powerlaw_graph(n, e_und, seed=0)
    partition, comps, C_list = fg.synth.neighborhood_partition(ei, n, ratio, seed=0)
    X = fg.synth.features(n, F, seed=0, kind="bow")
    y = np.zeros(n, dtype=np.int64)
    import scipy.sparse as sp
    cos = []
    for comp, Cm in zip(comps, C_list):
        if Cm is None:
            cos.append(None)
            continue
        part_c, _ = fo.partition_of(Cm)
        relabel = np.full(n, -1); relabel[comp] = np.arange(len(comp))
        em = relabel[ei[0]] >= 0
        r, c, v = fo.project_adj_pattern(relabel[ei[:, em]], part_c, Cm.shape[0])
        adj = sp.csr_matrix((v > 0, (r, c)), shape=(Cm.shape[0], Cm.shape[0]))
        cos.append(dict(part=part_c, CX=fo.project_features(Cm, X.numpy()[comp]), adj=adj))
    subs = fo.build_subgraphs(ei, X.numpy(), y, comps, cos, mode)
    want = fo.expected_pack(subs, n, mode)
    pack = fg.build_pack(torch.tensor(ei, device=dev()), torch.tensor(partition.part), partition.k, mode)
    for name in ("rowptr", "col", "gid", "sub_ptr", "core_rows", "is_core", "mask"):
        assert np.array_equal(getattr(pack, name).detach().cpu().numpy().astype(np.int64), np.asarray(want[name]).astype(np.int64)), name
    sd = fo.init_state_dict(F, 512, C, seed=1)
    Xg = X
    if mode == "cluster":
        proj = fg.coarsen.project(torch.tensor(ei, device=dev()), X.to(dev()), partition)
        xc = proj["Xc"].cpu()
        for i, co in enumerate(cos):
            if co is None:
                xc[int(partition.sub_offset[i])] = X[comps[i][0]]
        Xg = torch.cat([X, xc], 0)
    out, ids = fg.infer.node_infer_Gs(sd, pack, Xg.to(dev()))
    ones = []
    for s in subs:
        m = np.zeros(s["x"].shape[0], dtype=bool)
        m[np.searchsorted(s["orig_idx"], s["core"])] = True
        ones.append(m)
    want_out = fo.node_infer_batched(sd, subs, ones, "node_cls", 128)
    assert_close(out.detach().cpu().numpy(), want_out.numpy())


def test_block_diagonal_independence_and_permutation(fg):
    """Size-independent properties: (i) the packed result equals the per-subgraph result; (ii) relabelling the
    nodes of the input graph permutes the outputs and nothing else."""
    n, e_und, F, C, ratio = 20000, 60000, 64, 7, 0.3
    ei = fg.synth.powerlaw_graph(n, e_und, seed=3)
    partition, comps, C_list = fg.synth.neighborhood_partition(ei, n, ratio, seed=3)
    X = fg.synth.features(n, F, seed=3)
    sd = fo.init_state_dict(F, 128, C, seed=3)
    eid = torch.tensor(ei, device=dev())
    pack = fg.build_pack(eid, torch.tensor(partition.part), partition.k, "extra")
    out, ids = fg.infer.node_infer_Gs(sd, pack, X.to(dev()))
    q = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:500]
    pq = fg.infer.per_query(sd, pack, X.to(dev()), q)
    full = torch.empty(n, C, device=dev()); full[ids.long()] = out
    assert_close(pq.detach().cpu().numpy(), full[q.to(dev())].detach().cpu().numpy(), rtol=1e-5)
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(1))
    ei_p = perm[torch.tensor(ei)]
    part_p = torch.empty(n, dtype=torch.int32); part_p[perm] = torch.tensor(partition.part)
    X_p = torch.empty_like(X); X_p[perm] = X
    pack_p = fg.build_pack(ei_p.to(dev()), part_p, partition.k, "extra")
    out_p, ids_p = fg.infer.node_infer_Gs(sd, pack_p, X_p.to(dev()))
    full_p = torch.empty(n, C, device=dev()); full_p[ids_p.long()] = out_p
    assert_close(full_p[perm.to(dev())].detach().cpu().numpy(), full.detach().cpu().numpy(), rtol=1e-4)


def test_bad_inputs_fail_loudly(fg):
    ei = torch.tensor([[0, 5], [1, 2]], device=dev())
    with pytest.raises(fg._lib.FitgnnError):
        fg.ops.csr_from_coo(ei, 3)  # node id out of range
    with pytest.raises(fg._lib.FitgnnError):
        fg.build_pack(torch.tensor([[0, 1], [1, 0]], device=dev()), torch.tensor([0, 7], dtype=torch.int32), 2, "none")
    with pytest.raises(fg._lib.FitgnnError):
        fg.ops.gemm_bias_act(torch.zeros(2, 3), torch.zeros(4, 3))  # CPU tensors


@pytest.mark.parametrize("mode", ["extra", "cluster"])
def test_physics_shaped_config_sampled(fg, mode):
    """configs[2]: Coauthor-Physics-shaped synthetic (34,493 nodes, 247,962 undirected edges, 8,415 features, ratio 0.1,
    many small subgraphs + a few huge ones).  Whole-pack invariants, then a sample of subgraphs bit-exact against the
    oracle builder and their logits against the oracle forward."""
    n, e_und, F, C, ratio = fg.synth.SHAPES["physics"]
    ei = fg.synth.powerlaw_graph(n, e_und, seed=2)
    partition, comps, C_list = fg.synth.neighborhood_partition(ei, n, ratio, seed=2)
    eid = torch.tensor(ei, device=dev())
    X = fg.synth.features(n, F, seed=2, kind="bow", device=dev())
    proj = fg.coarsen.project(eid, X, partition)
    pack = fg.build_pack(eid, torch.tensor(partition.part), partition.k, mode, proj["ac_rowptr"], proj["ac_col"])
    # invariants: every node is core exactly once; rows of a subgraph stay inside it; the CSR is symmetric
    assert sorted(pack.core_gid.cpu().tolist()) == list(range(n))
    sp = pack.sub_ptr.long()
    rows_sub = torch.repeat_interleave(torch.arange(pack.n_sub, device=dev()), sp[1:] - sp[:-1])
    deg = (pack.rowptr[1:] - pack.rowptr[:-1]).long()
    erow = torch.repeat_interleave(torch.arange(pack.n_rows, device=dev()), deg)
    assert torch.equal(rows_sub[erow], rows_sub[pack.col.long()])
    fwd_keys = erow * pack.n_rows + pack.col.long()
    bwd_keys = torch.sort(pack.col.long() * pack.n_rows + erow).values
    assert torch.equal(fwd_keys, bwd_keys)  # fwd_keys are already sorted (CSR order)
    assert torch.equal(pack.dinv, 1.0 / torch.sqrt(deg.float()))
    # sample: the 3 biggest subgraphs + 40 random ones
    sizes = (sp[1:] - sp[:-1]).cpu().numpy()
    rng = np.random.default_rng(0)
    ids = np.unique(np.concatenate([np.argsort(-sizes)[:3], rng.choice(pack.n_sub, 40, replace=False)]))
    import scipy.sparse as sp_
    xc = proj["Xc"].cpu().numpy()
    cos = []
    for i, (comp, Cm) in enumerate(zip(comps, C_list)):
        if Cm is None:
            cos.append(None); continue
        part_c, _ = fo.partition_of(Cm)
        s0, s1 = int(partition.sub_offset[i]), int(partition.sub_offset[i + 1])
        r0, r1 = int(proj["ac_rowptr"][s0]), int(proj["ac_rowptr"][s1])
        adj = sp_.csr_matrix((np.ones(r1 - r0, dtype=bool), (proj["ac_row"][r0:r1].cpu().numpy() - s0,
                                                               proj["ac_col"][r0:r1].cpu().numpy() - s0)), shape=(s1 - s0, s1 - s0))
        cos.append(dict(part=part_c, CX=xc[s0:s1], adj=adj))
    Xn = X.cpu().numpy()
    subs = fo.build_subgraphs(ei, Xn, np.zeros(n, dtype=np.int64), comps, cos, mode, only=set(ids.tolist()))
    small = fg.infer.select_subgraphs(pack, torch.tensor(ids))
    want = fo.expected_pack([subs[i] for i in ids], n, mode)
    for name in ("rowptr", "col", "sub_ptr", "core_rows", "is_core", "mask"):
        assert np.array_equal(getattr(small, name).cpu().numpy().astype(np.int64), np.asarray(want[name]).astype(np.int64)), name
    gid_want = want["gid"].copy()
    assert np.array_equal(small.gid.cpu().numpy().astype(np.int64), gid_want)
    # logits of the sampled subgraphs (bf16x3 tensor-core GEMMs, transform-first on the de-duplicated rows)
    sd = fo.init_state_dict(F, 512, C, seed=4)
    Xg = torch.cat([X, proj["Xc"]], 0) if mode == "cluster" else X
    out = fg.PackedForward(small, sd, precision="bf16x3")(Xg).detach().cpu().numpy()
    sel = []
    for i in ids:
        m = np.zeros(subs[i]["x"].shape[0], dtype=bool)
        m[np.searchsorted(subs[i]["orig_idx"], subs[i]["core"])] = True
        sel.append(m)
    want_out = fo.node_infer_batched(sd, [subs[i] for i in ids], sel, "node_cls", 128).numpy()
    assert_close(out, want_out)


def test_csr_cache_never_serves_a_stale_graph(fg):
    """The drop-in GCNConv caches gcn_norm per edge_index tensor object; a new tensor that reuses the address (and
    shape) of a freed one must not hit the old entry, and in-place edits must invalidate."""
    conv = fg.GCNConv(4, 8).to(dev()).eval()
    x = torch.rand(6, 4, device=dev())
    with torch.no_grad():
        for trial in range(20):
            g = torch.Generator().manual_seed(trial)
            src = torch.randint(0, 6, (9,), generator=g)
            dst = torch.randint(0, 6, (9,), generator=g)
            ei = torch.stack([src, dst]).to(dev())  # same shape every time; freed at the end of each iteration
            want = fo.gcn_conv_fp64(x.cpu().numpy(), ei.cpu().numpy(), conv.lin.weight.cpu().numpy(), conv.bias.cpu().numpy())
            assert_close(conv(x, ei).cpu().numpy(), want)
            del ei
        ei = torch.tensor([[0, 1], [1, 0]], device=dev())
        a = conv(x, ei).clone()
        ei[0, 0] = 2  # in-place edit bumps _version
        b = conv(x, ei)
        want = fo.gcn_conv_fp64(x.cpu().numpy(), ei.cpu().numpy(), conv.lin.weight.cpu().numpy(), conv.bias.cpu().numpy())
        assert_close(b.cpu().numpy(), want)
        assert not torch.equal(a, b)


@pytest.mark.parametrize("mode", MODES)
def test_pack_builder_duplicates_self_loops_and_isolated(fg, mode):
    """Edge cases of the input COO: duplicate edges (kept, they count twice in gcn_norm), self loops (dropped and
    re-added once), isolated nodes and 1-2 node components — all three modes against the oracle builder."""
    import scipy.sparse as sp_
    n = 400
    ei = fg.synth.powerlaw_graph(n - 30, 700, seed=9)  # the last 30 nodes stay isolated / tiny
    extra_pairs = np.array([[n - 30, n - 29], [n - 29, n - 30], [n - 28, n - 27], [n - 27, n - 28], [n - 27, n - 26], [n - 26, n - 27]]).T
    ei = np.concatenate([ei, extra_pairs], 1)
    partition, comps, C_list = fg.synth.neighborhood_partition(ei, n, 0.4, seed=9)
    rng = np.random.default_rng(9)
    dup = ei[:, rng.choice(ei.shape[1], 60, replace=False)]
    loops = np.stack([rng.integers(0, n, 25)] * 2)
    ei2 = np.concatenate([ei, dup, dup[:, :10], loops], 1)
    ei2 = np.ascontiguousarray(ei2[:, rng.permutation(ei2.shape[1])])
    X = fg.synth.features(n, 8, seed=9)
    cos = []
    for comp, Cm in zip(comps, C_list):
        if Cm is None:
            cos.append(None); continue
        part_c, _ = fo.partition_of(Cm)
        relabel = np.full(n, -1); relabel[comp] = np.arange(len(comp))
        em = relabel[ei2[0]] >= 0
        r, c, v = fo.project_adj_pattern(relabel[ei2[:, em]], part_c, Cm.shape[0])
        cos.append(dict(part=part_c, CX=fo.project_features(Cm, X.numpy()[comp]),
                        adj=sp_.csr_matrix((v > 0, (r, c)), shape=(Cm.shape[0], Cm.shape[0]))))
    subs = fo.build_subgraphs(ei2, X.numpy(), np.zeros(n, dtype=np.int64), comps, cos, mode)
    want = fo.expected_pack(subs, n, mode)
    pack = fg.build_pack(torch.tensor(ei2, device=dev()), torch.tensor(partition.part), partition.k, mode)
    for name in ("rowptr", "col", "gid", "sub_ptr", "core_rows", "is_core", "mask"):
        assert np.array_equal(getattr(pack, name).cpu().numpy().astype(np.int64), np.asarray(want[name]).astype(np.int64)), name
    assert np.array_equal(pack.dinv.cpu().numpy(), want["dinv"])
    # logits of the whole pack against the oracle forward on the reference-style subgraph list
    sd = fo.init_state_dict(8, 64, 3, seed=9)
    Xg = X
    if mode == "cluster":
        proj = fg.coarsen.project(torch.tensor(ei2, device=dev()), X.to(dev()), partition)
        xc = proj["Xc"].cpu()
        for i, co in enumerate(cos):
            if co is None:
                xc[int(partition.sub_offset[i])] = X[comps[i][0]]
        Xg = torch.cat([X, xc], 0)
    out, ids = fg.infer.node_infer_Gs(sd, pack, Xg.to(dev()))
    sel = []
    for s in subs:
        m = np.zeros(s["x"].shape[0], dtype=bool)
        m[np.searchsorted(s["orig_idx"], s["core"])] = True
        sel.append(m)
    assert_close(out.detach().cpu().numpy(), fo.node_infer_batched(sd, subs, sel, "node_cls", 128).numpy())


@pytest.mark.parametrize("mode", MODES)
def test_pack_builder_edgeless_graph(fg, mode):
    """No edges at all: every node is its own single-node subgraph with only its self loop (utils.py:352-368)."""
    n = 37
    ei = torch.zeros(2, 0, dtype=torch.long, device=dev())
    pack = fg.build_pack(ei, torch.arange(n, dtype=torch.int32), n, mode)
    assert (pack.n_rows, pack.nnz, pack.n_sub) == (n, n, n)
    assert torch.equal(pack.col.cpu(), torch.arange(n, dtype=torch.int32))
    assert torch.equal(pack.dinv.cpu(), torch.ones(n))
    sd = fo.init_state_dict(5, 16, 3, seed=1)
    X = torch.rand(n + (n if mode == "cluster" else 0), 5)
    out, ids = fg.infer.node_infer_Gs(sd, pack, X.to(dev()))
    want = fo.classify_node(sd, X[:n], torch.zeros(2, 0, dtype=torch.long))  # isolated nodes: out = lin(x) + b
    assert_close(out.detach().cpu().numpy(), want.numpy()[ids.cpu().numpy()])


def test_bench_dump_outputs_repeats_run_to_run(tmp_path):
    """`bench.py --dump-outputs DIR` on the small workload: the last timed step's logits (log_softmax rows, float32, keyed by
    float64 node ids, under 64 MB in all) come out the same from two runs with the same arguments, which is what makes two
    builds comparable output for output."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dumps = []
    for run in ("a", "b"):
        d = tmp_path / run
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--workload", "products-small", "--steps", "2",
                              "--warmup", "1", "--modes=", "--no-cpu-baseline", "--no-projection", "--no-e2e",
                              "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600, cwd=root)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])["steps"] == 2
        assert sorted(os.listdir(d)) == ["logits.npy", "node_ids.npy"]
        assert sum(os.path.getsize(d / f) for f in os.listdir(d)) <= 64 << 20
        dumps.append((np.load(d / "node_ids.npy"), np.load(d / "logits.npy")))
    (ids, logits), (ids_b, logits_b) = dumps
    n = 200000  # products-small: every node fits the sample
    assert ids.dtype == np.float64 and np.array_equal(ids, np.arange(n))
    assert logits.dtype == np.float32 and logits.shape == (n, 47) and np.isfinite(logits).all()
    lse = np.log(np.exp(logits.astype(np.float64)).sum(1))
    assert np.abs(lse).max() < 1e-4
    assert np.array_equal(ids, ids_b)
    assert np.abs(logits - logits_b).max() <= 1e-5 * max(1.0, float(np.abs(logits).max()))
