"""GPU: SAGEConv on the fp16 planes — the fp16 mean aggregation (both forms) and the root form with an fp16 output against
fp64 of the operands the kernels see, the two-segment transform (fitgnn_gemm_f16_2seg) bit for bit against fitgnn_gemm_f16 on
the materialised operand under every plan, its refusals, and PackedForward(precision="fp16" / "fp16x2") on SAGE models
against the torch-CPU restatement (tests/sage_oracle.py)."""
import numpy as np
import pytest
import torch

from oracle import fitgnn_oracle as fo
from tests import golden_io as gio
from tests import sage_oracle as so
from tests.test_gpu_sage import _golden_pack, graph_with_everything, mean_fp64

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
F16_MAX = 65504.0
U16, U32 = 2.0 ** -11, 2.0 ** -24  # fp16 rounding (to nearest) and fp32 unit roundoff


@pytest.fixture(scope="module")
def fg():
    import fitgnn_b200
    return fitgnn_b200


def _degrees(rp, cl, rows, skip_self):
    return np.array([int(np.sum(cl[rp[r]:rp[r + 1]] != r)) if skip_self else int(rp[r + 1] - rp[r]) for r in rows])


# ------------------------------------------------------------------------------------------ fp16 mean aggregation
@pytest.mark.parametrize("width", [32, 64, 512])
@pytest.mark.parametrize("skip_self", [False, True])
@pytest.mark.parametrize("concat", [False, True])
def test_mean_f16_matches_fp64(fg, width, skip_self, concat):
    n, n_src = 700, 900
    half = width + 8  # pad columns [width, half) in each half
    ei = graph_with_everything(n, 3000, seed=width, hub=5, hub_deg=1000)  # rows without neighbours, duplicates, a ~1,000-entry row
    rowptr, col = fg.ops.csr_raw_from_coo(torch.tensor(ei, device=DEV), n)
    rp, cl = rowptr.cpu().numpy(), col.cpu().numpy()
    g = torch.Generator().manual_seed(width + 7)
    X = (torch.randn(n_src, width, generator=g) * 4).half()
    X[::17, :5] = F16_MAX  # the largest finite fp16 values: the mean of such rows must stay finite
    X[3::17, 5:9] = -F16_MAX
    src_index = torch.randperm(n_src, generator=g)[:n].to(torch.int32)
    out_rows = torch.tensor(np.r_[5, np.arange(n - 1, -1, -3)], dtype=torch.int32)  # hub, isolated rows, reversed order
    Xd, sd_, od = X.to(DEV), src_index.to(DEV), out_rows.to(DEV)
    Xn = X.double().numpy()
    agg, root = mean_fp64(rp, cl, Xn, src_index.numpy(), out_rows.numpy(), skip_self)
    mabs, _ = mean_fp64(rp, cl, np.abs(Xn), src_index.numpy(), out_rows.numpy(), skip_self)
    deg = _degrees(rp, cl, out_rows.numpy(), skip_self)[:, None]
    y = fg.ops.spmm_mean_f16(rowptr, col, Xd, width, half, sd_, skip_self, od, concat=concat)
    assert y.dtype == torch.float16 and y.shape == (len(out_rows), 2 * half if concat else half)
    yn = y.double().cpu().numpy()
    assert np.isfinite(yn).all() and np.abs(yn).max() <= F16_MAX
    budget = U16 * np.abs(agg) + (deg + 1) * U32 * mabs
    assert (np.abs(yn[:, :width] - agg) <= budget).all(), float(np.abs(yn[:, :width] - agg).max())
    assert not yn[:, width:half].any()  # pad columns written as zeros
    if concat:
        assert np.array_equal(yn[:, half:half + width], root)  # the root half is a copy of the fp16 row
        assert not yn[:, half + width:].any()
    # bit-identical across calls, row selections and the gid indirection
    assert torch.equal(y, fg.ops.spmm_mean_f16(rowptr, col, Xd, width, half, sd_, skip_self, od, concat=concat))
    full = fg.ops.spmm_mean_f16(rowptr, col, Xd[sd_.long()].contiguous(), width, half, None, skip_self, concat=concat)
    assert torch.equal(full[od.long()], y)


@pytest.mark.parametrize("width", [32, 64, 512])
@pytest.mark.parametrize("skip_self", [False, True])
def test_mean_root_f16_matches_fp64(fg, width, skip_self):
    n, n_src = 600, 650
    ei = graph_with_everything(n, 2500, seed=width + 1, hub=7, hub_deg=1000)
    rowptr, col = fg.ops.csr_raw_from_coo(torch.tensor(ei, device=DEV), n)
    rp, cl = rowptr.cpu().numpy(), col.cpu().numpy()
    g = torch.Generator().manual_seed(width)
    Z = torch.randn(n_src, 2 * width + 4, generator=g)  # [Z_l | Z_r | spare]: root_off = width
    bias = torch.randn(width, generator=g) * 0.1
    src_index = torch.randperm(n_src, generator=g)[:n].to(torch.int32)
    out_rows = torch.tensor(np.r_[7, np.arange(0, n, 2)], dtype=torch.int32)
    Zn = Z.double().numpy()
    agg, _ = mean_fp64(rp, cl, Zn[:, :width], src_index.numpy(), out_rows.numpy(), skip_self)
    mabs, _ = mean_fp64(rp, cl, np.abs(Zn[:, :width]), src_index.numpy(), out_rows.numpy(), skip_self)
    root = Zn[src_index.numpy()[out_rows.numpy()], width:2 * width]
    pre = agg + root + bias.double().numpy()
    want = np.where(pre > 0, pre, np.expm1(pre))
    deg = _degrees(rp, cl, out_rows.numpy(), skip_self)[:, None]
    # the same budget, with the fp32 adds of root and bias folded into the (deg + 1) term and the ELU's ex2.approx (<= 2^-22)
    budget = U16 * np.abs(want) + (deg + 3) * U32 * (mabs + np.abs(root) + np.abs(bias.numpy())) + 2.0 ** -22
    args = (rowptr, col, Z.to(DEV), width, width, src_index.to(DEV), skip_self, bias.to(DEV), fg.ops.ACT_ELU, out_rows.to(DEV))
    y = fg.ops.spmm_mean_root_f16(*args)
    assert y.dtype == torch.float16 and y.shape == (len(out_rows), width)
    err = np.abs(y.double().cpu().numpy() - want)
    assert (err <= budget).all(), float(err.max())
    assert torch.equal(y, fg.ops.spmm_mean_root_f16(*args))
    # values beyond the fp16 range saturate to +-65504, never inf
    big = fg.ops.spmm_mean_root_f16(rowptr, col, (Z * 1e6).to(DEV), width, width, src_index.to(DEV), skip_self, None,
                                    fg.ops.ACT_NONE, out_rows.to(DEV)).double().cpu().numpy()
    ref = np.asarray(agg + root) * 1e6
    assert np.isfinite(big).all()
    sat = np.abs(ref) > 1.001 * F16_MAX
    assert sat.any() and np.array_equal(big[sat], np.sign(ref[sat]) * F16_MAX)


def test_mean_f16_rejects_bad_shapes(fg):
    rp, col = fg.ops.csr_raw_from_coo(torch.zeros(2, 0, dtype=torch.long, device=DEV), 4)
    X = torch.zeros(4, 16, dtype=torch.float16, device=DEV)
    with pytest.raises(fg._lib.FitgnnError):
        fg.ops.spmm_mean_f16(rp, col, X, 16, 8)  # half < width
    with pytest.raises(fg._lib.FitgnnError):
        fg.ops.spmm_mean_f16(rp, col, X, 12, 16)  # width not a multiple of 8
    with pytest.raises(fg._lib.FitgnnError):
        fg.ops.spmm_mean_f16(rp, col, X, 16, 16, out=torch.zeros(4, 16, dtype=torch.float16, device=DEV), concat=True)
    with pytest.raises(fg._lib.FitgnnError):
        fg.ops.spmm_mean_root_f16(rp, col, torch.zeros(4, 8, device=DEV), 8, 4)  # root half past the row


# ------------------------------------------------------------------------------------------ two-segment transform
TUNINGS = [{}, {"gemm_pair": 0}, {"gemm_pair_ws": 0}, {"gemm_ws": 0}, {"sm_reserve": 8}]


def _with_tuning(fg, sw, fn):
    old = {k: fg._lib.set_tuning(k, v) for k, v in sw.items()}
    try:
        return fn()
    finally:
        for k, v in old.items():
            fg._lib.set_tuning(k, v)


@pytest.mark.parametrize("K0,w0,w1,N", [(64, 40, 200, 256), (64, 32, 32, 32), (512, 512, 512, 512)])
@pytest.mark.parametrize("M", [1000, 5000])  # below / above the CTA-pair threshold (4096 rows)
@pytest.mark.parametrize("w_single", [False, True])
@pytest.mark.parametrize("out_f16", [False, True])
def test_gemm_2seg_bit_identical_to_materialised(fg, K0, w0, w1, N, M, w_single, out_f16):
    g = torch.Generator().manual_seed(K0 + w1 + M)
    K = K0 + w1
    nan = float("nan")
    A0 = torch.full((M, w0 + 8), nan, dtype=torch.float16)  # NaN in the pitch beyond each plane's width: never read
    A1 = torch.full((M, w1 + 8), nan, dtype=torch.float16)
    A0[:, :w0] = torch.randn(M, w0, generator=g).half()
    A1[:, :w1] = torch.randn(M, w1, generator=g).half()
    W = torch.randn(N, K, generator=g) / K ** 0.5
    bias = torch.randn(N, generator=g) * 0.1
    cat = torch.zeros(M, K, dtype=torch.float16)
    cat[:, :w0], cat[:, K0:] = A0[:, :w0], A1[:, :w1]
    A0, A1, cat, bias = A0.to(DEV), A1.to(DEV), cat.to(DEV), bias.to(DEV)
    Wp = fg.ops.split_f16(W.to(DEV), lo=not w_single)
    for sw in TUNINGS:
        def run():
            got = fg.ops.gemm_f16_2seg(A0, A1, Wp, K0, bias, fg.ops.ACT_ELU, out_f16=out_f16, a0_cols=w0, K=K, N=N)
            want = fg.ops.gemm_f16(cat, Wp, bias, fg.ops.ACT_ELU, out_f16=out_f16, K=K, N=N)
            return got, want
        got, want = _with_tuning(fg, sw, run)
        assert torch.equal(got, want), sw
    # and the product is the right one (fp64 of the rounded operands; 2^-11 per weight element under 'fp16')
    wq = (Wp[0].double() + (Wp[1].double() if Wp[1] is not None else 0))[:, :K]
    pre = cat.double() @ wq.T + bias.double()
    ref = torch.where(pre > 0, pre, torch.expm1(pre))
    assert float((got[:, :N].double() - ref).abs().max()) <= 2e-2 * max(1.0, float(ref.abs().max()))


def test_gemm_2seg_refusals(fg):
    M, N = 256, 64
    A = torch.zeros(M, 64, dtype=torch.float16, device=DEV)
    W = fg.ops.split_f16(torch.zeros(N, 192, device=DEV))
    with pytest.raises(fg._lib.FitgnnError):  # K0 not a multiple of 64
        fg.ops.gemm_f16_2seg(A, A, W, 96, K=160, N=N)
    with pytest.raises(fg._lib.FitgnnError):  # A0 wider than its segment
        fg.ops.gemm_f16_2seg(A, A, W, 64, a0_cols=72, K=128, N=N)
    buf = torch.zeros(M * 64 + 8, dtype=torch.float16, device=DEV)
    with pytest.raises(fg._lib.FitgnnError):  # A1 not 16-byte aligned
        fg.ops.gemm_f16_2seg(A, buf[1:1 + M * 64].view(M, 64), W, 64, N=N)
    with pytest.raises(fg._lib.FitgnnError):  # A1 pitch (36 halfs) not a multiple of 8
        fg.ops.gemm_f16_2seg(A, torch.zeros(M, 36, dtype=torch.float16, device=DEV), W, 64, N=N)
    with pytest.raises(fg._lib.FitgnnError):  # A0 pitch not a multiple of 8
        fg.ops.gemm_f16_2seg(torch.zeros(M, 36, dtype=torch.float16, device=DEV), A, W, 64, N=N)


# ------------------------------------------------------------------------------------------ engine
PRECISIONS = ("fp16", "fp16x2")
MARGINS = {}  # observed max |err| / max |oracle logit| per case, printed at the end of the module


def _margin(name, got, want):
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    assert got.shape == want.shape, (got.shape, want.shape)
    rel = float((got - want).abs().max()) / max(1e-12, float(want.abs().max()))
    MARGINS[name] = rel
    assert rel <= 1e-3, (name, rel)


@pytest.fixture(scope="module", autouse=True)
def _report_margins():
    yield
    if MARGINS:
        print("\nfp16 SAGE engine: largest |logit error| / largest |oracle logit| = %.2e (%s)"
              % max((v, k) for k, v in MARGINS.items()))


def _expect_launches(fwd, rows_subset):
    names = set(fwd.profile_summary())
    first = {"gemm0_unique_rows", "mean0"} if fwd.transform_first else {"mean0", "gemm0"}
    assert first <= names and "head" in names, names
    for i in range(1, fwd.L):
        assert {f"mean{i}", f"gemm{i}"} <= names, names
    # layers >= 1 run the two-segment transform (K = K0 + H) except a last layer on a row subset (concat, K = 2 K0)
    last = fwd.L - 1
    s = fwd.profile_summary()[f"gemm{last}"]
    K = 2 * fwd.K0 if rows_subset else fwd.K0 + fwd.H
    assert s["flops"] == 2 * (fwd.n_out if rows_subset else fwd.pack.n_rows) * K * fwd.H


@pytest.mark.parametrize("mode", ("none", "extra", "cluster"))
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("L", [2, 3])
def test_engine_node_small(fg, mode, precision, L):
    d = gio.load("node_small")
    pack, X = _golden_pack(fg, d, mode)
    F, C, H = d["x"].shape[1], int(d["n_classes"]), 32  # F = 12 <= H: aggregate-first layer 0
    sd = so.init_state_dict(F, H, C, num_layers=L, seed=6 + L)
    ref = gio.subgraphs(d, mode + "_sub")
    xc, eic = fo.collate(ref)
    tm = torch.tensor(np.concatenate([r["test_mask"] for r in ref]))
    want = so.classify_node(sd, xc, eic)[tm]
    out, ids = fg.infer.node_infer_Gs(sd, pack, X, torch.tensor(d["test_mask"]), precision=precision)
    _margin(f"node_small/{mode}/{precision}/L{L}", out, want)
    sdd = {k: v.to(DEV) for k, v in sd.items()}
    fwd = fg.PackedForward(pack, sdd, rows="core", precision=precision)
    assert fwd.sage_f16
    fwd.enable_profile(True)
    core = fwd(X)
    torch.cuda.synchronize()
    _expect_launches(fwd, rows_subset=fwd.out_rows is not None)
    fwd.enable_profile(False)
    run = fwd.capture(X)
    assert torch.equal(run(X), fwd(X))  # graph replay == eager, bit for bit
    q = ids[:: max(1, ids.numel() // 20)]
    pq = fg.infer.per_query(sd, pack, X, q, precision=precision)
    lookup = torch.full((pack.n_nodes,), -1, dtype=torch.long, device=DEV)
    lookup[pack.core_gid.long()] = torch.arange(pack.n_core, device=DEV)
    want_q = core[lookup[q]]  # the same rows computed in a pack of the queried subgraphs only
    assert float((pq - want_q).abs().max()) <= 1e-5 * float(want_q.abs().max())


@pytest.fixture(scope="module")
def planted(fg):
    """A mode-'none' pack of 6,000 rows (above the CTA-pair threshold) and the features, F = 200 columns."""
    n, e = 6000, 30000
    ei, part, _, k = fg.synth.planted_partition(n, e, 0.05, seed=3, device=DEV)
    part = fg.synth.relabel_partition_reference_order(part)
    X = fg.synth.features(n, 200, seed=3, device=DEV)
    pack = fg.build_pack(ei, part, k, "none")
    subs = fo.subgraphs_from_partition(ei.cpu().numpy(), X.cpu().numpy(), part.cpu().numpy(), np.arange(k))
    xc, eic = fo.collate(subs)
    nodes = torch.from_numpy(np.concatenate([s["orig_idx"] for s in subs])).long()
    return pack, X, xc, eic, nodes


@pytest.mark.parametrize("F", [100, 200])  # H = 128: aggregate-first / transform-first layer 0
@pytest.mark.parametrize("L", [2, 3])
@pytest.mark.parametrize("rows", ["core", "all", "explicit"])
@pytest.mark.parametrize("precision", PRECISIONS)
def test_engine_planted_pack(fg, planted, F, L, rows, precision):
    pack, X, xc, eic, nodes = planted
    assert pack.n_rows >= 4096
    H, C = 128, 47
    sd = so.init_state_dict(F, H, C, num_layers=L, seed=F + L)
    oracle = torch.empty(pack.n_nodes, C, dtype=torch.float64)
    oracle[nodes] = so.classify_node(sd, xc[:, :F], eic).double()
    sel = {"core": "core", "all": "all",
           "explicit": torch.arange(pack.n_rows - 1, -1, -3, device=DEV, dtype=torch.int32)}[rows]
    row_ids = {"core": pack.core_rows, "all": torch.arange(pack.n_rows, device=DEV),
               "explicit": sel if rows == "explicit" else None}[rows].long()
    fwd = fg.PackedForward(pack, {k: v.to(DEV) for k, v in sd.items()}, rows=sel, precision=precision)
    assert fwd.sage_f16 and fwd.transform_first == (F > H)
    Xf = X[:, :F].contiguous()
    fwd.enable_profile(True)
    out = fwd(Xf)
    torch.cuda.synchronize()
    _expect_launches(fwd, rows_subset=fwd.out_rows is not None)
    fwd.enable_profile(False)
    _margin(f"planted/F{F}/L{L}/{rows}/{precision}", out, oracle[pack.gid.long()[row_ids].cpu()])
    if rows == "core":
        run = fwd.capture(Xf)
        assert torch.equal(run(Xf), fwd(Xf))


@pytest.mark.parametrize("H,L", [(8, 2), (32, 1)])
@pytest.mark.parametrize("precision", PRECISIONS)
def test_ineligible_models_run_bf16x3(fg, H, L, precision):
    d = gio.load("node_small")
    pack, X = _golden_pack(fg, d, "extra")
    sd = {k: v.to(DEV) for k, v in so.init_state_dict(d["x"].shape[1], H, int(d["n_classes"]), num_layers=L, seed=2).items()}
    fwd = fg.PackedForward(pack, sd, precision=precision)
    assert not fwd.sage_f16
    assert torch.equal(fwd(X), fg.PackedForward(pack, sd, precision="bf16x3")(X))
