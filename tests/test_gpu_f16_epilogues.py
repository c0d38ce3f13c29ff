"""GPU: the fp16-plane epilogues of the tensor-core transform against fp64 references of the ROUNDED operands the kernels see
(bf16 hi + lo, one fp16 plane, fp16 hi + lo), and their invariance under the tuning switches that pick a plan.

Kernels: fitgnn_gcn_transform_aggregate_f16 (gemm0_agg of precision='fp16', incl. the plain transform with agg_desc = NULL),
fitgnn_gcn_conv_aligned_f16 (conv_fused), the deferred row scale chained into fitgnn_gemm_f16 / the bf16x3 transform, the
row-mapped fp16 head (fitgnn_gemm_f16 with row_map, fitgnn_gemm_f16_head_rows_peers), saturation of fp16-plane outputs and the
host-side refusals.  The aligned groups are synthetic (make_groups): every edge case of the aggregation sits exactly where the
kernel is fragile (12 neighbours in every row, none, both in one warp, lanes 0 and 31, padding at group tails and whole padding
groups at 128- and 256-row tile boundaries, a ragged last group).

Budget of an fp16-plane output element: |got - want| <= 2^-11 |want| + TAU16 * max|want| (the rounding of the result plus fp32
accumulation); fp32 outputs: TAU32 * max(1, max|want|)."""
import contextlib

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

TAU16 = 2e-5
TAU32 = 1e-5
F16_MAX = 65504.0
_worst = {}  # family -> worst observed |got - want| / bound


def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def fg():
    import fitgnn_b200
    return fitgnn_b200


@pytest.fixture(scope="module", autouse=True)
def report_margins():
    yield
    if _worst:
        print("\nworst |got - want| / bound: " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(_worst.items())))


def note(family, ratio):
    _worst[family] = max(_worst.get(family, 0.0), float(ratio))


@contextlib.contextmanager
def tuning(fg, **switches):
    """Set kernel-tuning switches for the block; the previous values come back in any case."""
    old = {}
    try:
        for k, v in switches.items():
            old[k] = fg._lib.set_tuning(k, v)
        yield
    finally:
        for k, v in old.items():
            fg._lib.set_tuning(k, v)


# ------------------------------------------------------------------------------------------ synthetic aligned groups
FIXED = ("mix", "all12", "all0", "edge_lanes")  # the first groups, in this order, when the pack has that many full groups


def make_groups(M, seed):
    """agg_desc (int64, fitgnn.h layout: bits 0-3 = count c <= 12, bits 4+5j..8+5j = row-in-group of the j-th neighbour) and
    dinv (fp32) of a synthetic group-aligned pack with M rows.  Neighbours are real rows of the row's own group of 32, never the
    row itself (the self term is implicit); duplicates occur.  Real rows: dinv in [0.05, 1]; padding rows: dinv = 0, desc = 0,
    at group tails and as whole groups on 128- and 256-row boundaries.  Groups 0..3: a warp mixing c = 12 and c = 0, every
    row c = 12, every row c = 0, every row listing lanes 0 and 31.  M % 32 != 0 gives a ragged last group."""
    rng = np.random.default_rng(seed)
    n_groups = (M + 31) // 32
    size = np.full(n_groups, 32)
    size[-1] = M - 32 * (n_groups - 1)
    n_real = size.copy()
    free = np.arange(n_groups) >= len(FIXED)
    tails = free & (rng.random(n_groups) < 0.25)
    n_real[tails] = np.maximum(1, size[tails] - rng.integers(1, 9, int(tails.sum())))
    bound = [g for g in range(len(FIXED), n_groups - 1) if g % 4 in (0, 3)]  # first / last group of a 128-row tile
    if bound:
        pick = set(rng.choice(bound, min(len(bound), max(2, n_groups // 64)), replace=False).tolist())
        pick |= {g for g in (7, 8) if g < n_groups - 1}  # around the first 256-row boundary
        n_real[sorted(pick)] = 0
    row = np.arange(M)
    lane, grp = row % 32, row // 32
    nr = n_real[grp]
    real = lane < nr
    cnt = rng.integers(0, 13, M)
    lanes = rng.integers(0, 1 << 20, (M, 12)) % np.maximum(nr - 1, 1)[:, None]
    lanes = lanes + (lanes >= lane[:, None])  # never the row itself
    for g, kind in enumerate(FIXED[:n_groups]):
        if size[g] != 32:
            break
        r = slice(32 * g, 32 * g + 32)
        if kind == "mix":
            cnt[r] = np.where(np.arange(32) % 2 == 0, 12, 0)
        elif kind == "all12":
            cnt[r] = 12
        elif kind == "all0":
            cnt[r] = 0
        else:
            lanes[r, 0] = np.where(np.arange(32) == 0, 31, 0)
            lanes[r, 1] = np.where(np.arange(32) == 31, 0, 31)
            cnt[r] = np.maximum(cnt[r], 2)
    cnt[(nr < 2) | ~real] = 0
    desc = cnt.astype(np.uint64)
    for j in range(12):
        desc |= np.where(j < cnt, lanes[:, j], 0).astype(np.uint64) << np.uint64(4 + 5 * j)
    dinv = np.where(real, rng.uniform(0.05, 1.0, M), 0.0).astype(np.float32)
    return torch.from_numpy(desc.view(np.int64)).to(dev()), torch.from_numpy(dinv).to(dev())


def decode(desc):
    """agg_desc -> int64 [M, 12] absolute neighbour rows, -1 past the row's count."""
    d = desc.cpu().numpy().view(np.uint64)
    cnt = (d & np.uint64(15)).astype(np.int64)
    lanes = ((d[:, None] >> (np.uint64(4) + np.uint64(5) * np.arange(12, dtype=np.uint64))) & np.uint64(31)).astype(np.int64)
    nbr = (np.arange(d.size) // 32 * 32)[:, None] + lanes
    return np.where(np.arange(12) < cnt[:, None], nbr, -1)


def aggregate64(h, nbr, dinv, scale=True):
    """s_r * (dinv[r] h[r] + sum_j dinv[c_j] h[c_j]) in fp64 on the device; s_r = dinv[r], or 1 when not scale."""
    d = dinv.double()
    idx = torch.from_numpy(nbr).to(h.device)
    out = d[:, None] * h
    for j in range(12):
        c = idx[:, j].clamp(min=0)
        out += torch.where(idx[:, j] >= 0, d[c], torch.zeros_like(d[c]))[:, None] * h[c]
    return d[:, None] * out if scale else out


def test_decode_matches_a_real_aligned_pack(fg):
    """The generator's layout is the builder's: decoding Pack.aligned's agg_desc gives the aligned CSR without its self loops,
    in CSR order."""
    from tests.test_gpu_aligned import small_subgraph_graph
    ei, part, k = small_subgraph_graph(3000, 1300, 11, max_size=12)
    ap = fg.build_pack(torch.tensor(ei, device=dev()), torch.tensor(part), k, "none").aligned(32, "degree")
    assert ap is not None and ap.agg_ok
    nbr = decode(ap.agg_desc)
    rp, col = ap.rowptr.cpu().numpy(), ap.col.cpu().numpy()
    for r in range(ap.n_rows):
        cs = list(col[rp[r]:rp[r + 1]])
        if r in cs:
            cs.remove(r)
        assert list(nbr[r][nbr[r] >= 0]) == cs, r
    # and the generator keeps to the same precondition
    desc, dinv = make_groups(1000, 0)
    nbr = decode(desc)
    d = dinv.cpu().numpy()
    rows = np.repeat(np.arange(1000), 12).reshape(1000, 12)
    on = nbr >= 0
    assert (nbr[on] // 32 == rows[on] // 32).all() and (nbr[on] != rows[on]).all() and (d[nbr[on]] > 0).all()
    assert (desc.cpu().numpy()[d == 0] == 0).all() and (d[:128] > 0).all()
    cnt = on.sum(1)
    assert (cnt[32:64] == 12).all() and (cnt[64:96] == 0).all() and {0, 12} == set(cnt[:32].tolist())
    edge = np.where(nbr[96:128] >= 0, nbr[96:128] % 32, -1)
    assert ((edge == 0).any(1) | (np.arange(32) == 0)).all() and ((edge == 31).any(1) | (np.arange(32) == 31)).all()
    assert (d[224:288] == 0).all()  # whole padding groups on both sides of the first 256-row boundary


# ------------------------------------------------------------------------------------------ operands
def operands(fg, M, K, lda, N, fmt, seed, a_scale=1.0, w_scale=1.0):
    """Kernel operands and their fp64 values (the first K columns).  fmt: 'bf16' (A, W bf16 hi/lo), 'f16w2' (A one fp16 plane,
    W fp16 hi/lo), 'f16w1' (A, W one fp16 plane each).  Columns K..lda hold finite garbage: the TMA maps end at K."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    A = torch.randn(M, lda, generator=g, device=dev()) * a_scale
    W = torch.randn(N, lda, generator=g, device=dev()) * (w_scale / K ** 0.5)
    if fmt == "bf16":
        Ak, Wk = fg.ops.split_bf16(A), fg.ops.split_bf16(W)
        A64, W64 = Ak[0].double() + Ak[1].double(), Wk[0].double() + Wk[1].double()
    else:
        Ak = fg.ops.split_f16(A, lo=False)[0]
        Wk = fg.ops.split_f16(W, lo=(fmt == "f16w2"))
        A64 = Ak.double()
        W64 = Wk[0].double() + (Wk[1].double() if Wk[1] is not None else 0.0)
    return Ak, Wk, A64[:, :K], W64[:, :K]


def make_bias(kind, N, seed):
    if kind is None:
        return None
    g = torch.Generator(device="cuda").manual_seed(seed + 7)
    if kind == "aligned":
        return torch.randn(N, generator=g, device=dev()) * 0.3
    b = (torch.randn(N + 1, generator=g, device=dev()) * 0.3)[1:]  # 4 bytes past a 16-byte boundary: the scalar bias path
    assert b.data_ptr() % 16 == 4
    return b


def act64(x, act):
    return torch.nn.functional.elu(x) if act == 1 else x


def check_f16(family, got, want, tau=TAU16, extra=None):
    """fp16-plane output against fp64: 2^-11 |want| + tau * max|want| (+ extra, a per-element term for rounded inputs)."""
    assert got.dtype == torch.float16 and bool(torch.isfinite(got).all())
    err = (got.double() - want).abs()
    bound = 2.0 ** -11 * want.abs() + tau * float(want.abs().max())
    if extra is not None:
        bound = bound + extra
    ratio = float((err / bound).max())
    note(family, ratio)
    if extra is None:  # share of the tau term used by what the rounding of the result does not explain
        note(family + " (tau share)", float((err - 2.0 ** -11 * want.abs()).clamp(min=0).max()) / (tau * float(want.abs().max())))
    assert ratio <= 1.0, f"{family}: worst |got - want| / bound = {ratio:.3g}"


def satfinite_half(x):
    return x.clamp(-F16_MAX, F16_MAX).half()


# ------------------------------------------------------------------------------------------ 1. transform + aggregate vs fp64
ELU, NONE = 1, 0
TA_CASES = [
    # the headline call of precision='fp16' (gemm0_agg): fp16 A with the bias folded into a constant-1 column, one W plane,
    # K = 101 at pitch 104, N = 512, deferred row scale, ELU, no bias; >= 148 * 256 rows: W-stationary, several m-blocks per CTA
    pytest.param(37900, 101, 104, 512, "f16w1", 1, ELU, None, True, id="headline"),
    pytest.param(32, 8, 8, 136, "bf16", 0, ELU, "aligned", True, id="one_group-K8-N136"),
    pytest.param(32, 512, 512, 512, "f16w2", 0, NONE, None, True, id="one_group-K512"),
    pytest.param(4095, 64, 64, 200, "f16w2", 1, NONE, "misaligned", True, id="M4095-N200"),
    pytest.param(4097, 128, 128, 384, "bf16", 1, ELU, "misaligned", True, id="M4097-N384-bf16"),
    pytest.param(4097, 512, 512, 512, "f16w1", 0, ELU, "aligned", True, id="M4097-K512"),
    pytest.param(40000, 104, 104, 136, "f16w2", 1, ELU, "aligned", True, id="wstat-N136"),
    pytest.param(38001, 101, 104, 200, "bf16", 0, ELU, "misaligned", True, id="wstat-bf16-N200-ragged"),
    pytest.param(5000, 101, 104, 512, "bf16", 0, ELU, None, False, id="plain-bf16"),
    pytest.param(4096, 101, 104, 200, "f16w1", 0, ELU, "misaligned", False, id="plain-f16-N200"),
    pytest.param(4095, 8, 8, 384, "f16w1", 0, NONE, "aligned", False, id="plain-K8-N384"),
]


@pytest.mark.parametrize("M,K,lda,N,fmt,defer,act,bias_kind,agg", TA_CASES)
def test_transform_aggregate_f16_matches_fp64(fg, M, K, lda, N, fmt, defer, act, bias_kind, agg):
    """G = s_r (dinv[r] h[r] + sum_j dinv[c_j] h[c_j]), h = act(A W^T + b), s_r = dinv[r] or 1 (defer_row_scale), one fp16
    plane; padding rows exactly 0.  agg = False: the plain transform act(A W^T + b)."""
    seed = M + K + N
    Ak, Wk, A64, W64 = operands(fg, M, K, lda, N, fmt, seed)
    if K == 101:  # the bias fold: constant 1 in the pad column of A, the bias in W's
        if fmt == "bf16":
            Ak[0][:, 100], Ak[1][:, 100] = 1.0, 0.0
        else:
            Ak[:, 100] = 1.0
        A64[:, 100] = 1.0
    bias = make_bias(bias_kind, N, seed)
    desc, dinv = make_groups(M, seed) if agg else (None, None)
    got = fg.ops.gcn_transform_aggregate_f16(Ak, Wk, bias, act, desc, dinv, K=K, N=N, defer_row_scale=bool(defer))
    h = act64(A64 @ W64.T + (bias.double() if bias is not None else 0.0), act)
    want = aggregate64(h, decode(desc), dinv, scale=not defer) if agg else h
    check_f16("transform_aggregate_f16" if agg else "transform_f16", got, want)
    if agg:
        pad = dinv == 0
        assert int(pad.sum()) > 0 or M == 32
        assert bool((got[pad] == 0).all())


# ------------------------------------------------------------------------------------------ 2. same operands, same bits
AGG_SWITCHES = [{"agg_wide": -1}, {"agg_wide": 1}, {"agg_wide": 2}, {"agg_wide": 3}, {"gemm_ws": 0}, {"gemm_prefetch": 1},
                {"sm_reserve": 6}, {"agg_wide": 1, "gemm_ws": 0, "sm_reserve": 6}, {"agg_wide": 3, "gemm_prefetch": 1, "sm_reserve": 6},
                {"agg_wide": 2, "gemm_ws": 0, "gemm_prefetch": 1}]


@pytest.mark.parametrize("M,K,lda,N,defer,bias_kind", [(37988, 101, 104, 512, 1, "aligned"), (5000, 128, 128, 384, 0, "misaligned"),
                                                       (4095, 512, 512, 200, 1, None)])
def test_fused_aggregation_bits_do_not_depend_on_the_plan(fg, M, K, lda, N, defer, bias_kind):
    """The fp16-plane output of the bf16 transform-aggregate is the fp32 output rounded once (satfinite); every fused-aggregation
    output (bf16 hi/lo, fp32, fp16 from bf16 planes, fp16 from an fp16 plane) is bit-identical under every tuning switch."""
    seed = M + N
    A_b, W_b, _, _ = operands(fg, M, K, lda, N, "bf16", seed)
    A_h, W_h, _, _ = operands(fg, M, K, lda, N, "f16w1", seed + 1)
    bias = make_bias(bias_kind, N, seed)
    desc, dinv = make_groups(M, seed)

    def run():
        return (fg.ops.gcn_transform_aggregate(A_b, W_b, bias, ELU, desc, dinv, K=K, N=N, split_out=True, defer_row_scale=defer),
                fg.ops.gcn_transform_aggregate(A_b, W_b, bias, ELU, desc, dinv, K=K, N=N, split_out=False, defer_row_scale=defer),
                fg.ops.gcn_transform_aggregate_f16(A_b, W_b, bias, ELU, desc, dinv, K=K, N=N, defer_row_scale=bool(defer)),
                fg.ops.gcn_transform_aggregate_f16(A_h, W_h, bias, ELU, desc, dinv, K=K, N=N, defer_row_scale=bool(defer)))

    (hi, lo), f32, f16_b, f16_h = run()
    assert torch.equal(f16_b, satfinite_half(f32))
    for sw in AGG_SWITCHES:
        with tuning(fg, **sw):
            (hi2, lo2), f32_2, f16_b2, f16_h2 = run()
        for name, a, b in (("hi", hi, hi2), ("lo", lo, lo2), ("fp32", f32, f32_2), ("fp16<-bf16", f16_b, f16_b2),
                           ("fp16<-fp16", f16_h, f16_h2)):
            assert torch.equal(a, b), f"{name} differs under {sw}"


# ------------------------------------------------------------------------------------------ 3. conv (aggregation on the accumulators)
CONV_CASES = [
    pytest.param(3000, 512, 512, "f16w2", ELU, "aligned", id="single_cta-M3000-two_planes"),
    pytest.param(20000, 128, 256, "f16w1", NONE, "misaligned", id="single_cta-K128"),
    pytest.param(5000, 256, 512, "f16w2", ELU, None, id="stream_pairs-two_planes"),
    pytest.param(6000, 512, 384, "f16w1", ELU, "misaligned", id="stream_pairs-N384"),
    pytest.param(38000, 512, 512, "f16w1", ELU, "aligned", id="wstat_pairs"),
]
CONV_SWITCHES = [{"gemm_pair": 0}, {"gemm_pair_ws": 0}, {"sm_reserve": 6}, {"gemm_pair_ws": 0, "sm_reserve": 6},
                 {"gemm_pair": 0, "sm_reserve": 6}, {"gemm_ws": 0}]


@pytest.mark.parametrize("M,K,N,fmt,act,bias_kind", CONV_CASES)
def test_conv_aligned_f16_matches_fp64(fg, M, K, N, fmt, act, bias_kind):
    """Y[r] = act(dinv[r] (dinv[r] p[r] + sum_j dinv[c_j] p[c_j]) + b), p = A W^T; a padding row (dinv = 0) holds act(b) rounded
    to fp16; bit-identical under gemm_pair, gemm_pair_ws, sm_reserve and gemm_ws."""
    seed = M + K + N + 1
    Ak, Wk, A64, W64 = operands(fg, M, K, K, N, fmt, seed)
    bias = make_bias(bias_kind, N, seed)
    desc, dinv = make_groups(M, seed)
    got = fg.ops.gcn_conv_aligned_f16(Ak, Wk, bias, act, desc, dinv, K=K, N=N)
    b64 = bias.double() if bias is not None else torch.zeros(N, dtype=torch.float64, device=dev())
    want = act64(aggregate64(A64 @ W64.T, decode(desc), dinv) + b64, act)
    check_f16("conv_aligned_f16", got, want)
    pad = dinv == 0
    assert int(pad.sum()) > 0
    assert bool((got[pad] == got[pad][0]).all())  # every padding row holds the same act(b), rounded once
    pad_row = act64(b64, act)
    if act == NONE:
        assert torch.equal(got[pad][0], pad_row.half())
    else:
        assert bool(((got[pad][0].double() - pad_row).abs() <= 2.0 ** -11 * pad_row.abs() + 1e-6).all())
    for sw in CONV_SWITCHES:
        with tuning(fg, **sw):
            again = fg.ops.gcn_conv_aligned_f16(Ak, Wk, bias, act, desc, dinv, K=K, N=N)
        assert torch.equal(again, got), f"differs under {sw}"


# ------------------------------------------------------------------------------------------ 4. deferred row scale, end to end
@pytest.mark.parametrize("precision", ["fp16", "bf16x3"])
def test_deferred_row_scale_two_layers_match_fp64(fg, precision):
    """transform_aggregate(defer_row_scale=1) -> next transform with row_scale = dinv (the fused schedule's last two GEMMs) equals
    the undeferred composition act(Â act(A W0^T) W1^T + b1) in fp64; the intermediate's own rounding is budgeted per element
    (2^-11 for the fp16 plane, 2^-16 for bf16 hi/lo) through |G| |W1|^T."""
    M, K, lda, H = 4100, 101, 104, 512
    fmt = "f16w1" if precision == "fp16" else "bf16"
    A0, W0, A64, W064 = operands(fg, M, K, lda, H, fmt, 3)
    _, W1, _, W164 = operands(fg, 1, H, H, H, fmt, 4)
    b1 = make_bias("aligned", H, 5)
    desc, dinv = make_groups(M, 6)
    G = aggregate64(torch.nn.functional.elu(A64 @ W064.T), decode(desc), dinv)
    want = torch.nn.functional.elu(G @ W164.T + b1.double())
    spread = G.abs() @ W164.abs().T
    if precision == "fp16":
        Gd = fg.ops.gcn_transform_aggregate_f16(A0, W0, None, ELU, desc, dinv, K=K, N=H, defer_row_scale=True)
        got = fg.ops.gemm_f16(Gd, W1, b1, ELU, row_scale=dinv, out_f16=True, K=H, N=H)
        check_f16("deferred_chain_f16", got, want, extra=2.0 ** -11 * spread)
    else:
        Gd = fg.ops.gcn_transform_aggregate(A0, W0, None, ELU, desc, dinv, K=K, N=H, split_out=True, defer_row_scale=True)
        got = fg.ops.gemm_bias_act(Gd, W1, b1, ELU, K=H, N=H, precision=fg.ops.GEMM_BF16X3, row_scale=dinv)
        bound = 2.0 ** -16 * spread + TAU32 * max(1.0, float(want.abs().max()))
        ratio = float(((got.double() - want).abs() / bound).max())
        note("deferred_chain_bf16x3", ratio)
        assert ratio <= 1.0, ratio


# ------------------------------------------------------------------------------------------ 5. fp16 head with a row map
def row_maps(M, seed):
    """name -> (row_map int32 [M] on the device, number of destination rows)."""
    rng = np.random.default_rng(seed)
    ident = np.arange(M)
    # aligned-pack shape: long runs of consecutive destinations broken by -1 padding rows; runs cross 32- and 128-row
    # boundaries (rows 20..45 and 110..150 stay unbroken) and rows 192..223 are a whole warp of padding
    pad = rng.random(M) < 0.06
    pad[20:46] = False
    pad[110:151] = False
    pad[192:224] = True
    aligned = np.where(pad, -1, np.cumsum(~pad) - 1)
    # identity with a whole warp of -1
    warp = np.where((ident >= 64) & (ident < 96), -1, ident - 32 * (ident >= 96))
    perm = rng.permutation(M)
    # destinations: a sorted random subset of 2M rows (gaps stay unmapped), and some rows dropped
    sub = np.sort(rng.choice(2 * M, M, replace=False))
    sub[rng.random(M) < 0.1] = -1
    maps = {"identity": (ident, M), "aligned": (aligned, int((~pad).sum())), "warp_of_pad": (warp, M - 32),
            "permutation": (perm, M), "subset_with_gaps": (sub, 2 * M)}
    return {k: (torch.from_numpy(v.astype(np.int32)).to(dev()), n) for k, (v, n) in maps.items()}


HEADS = {0: lambda z: z, 1: lambda z: torch.log_softmax(z, 1), 2: lambda z: torch.softmax(z, 1)}


@pytest.mark.parametrize("N", [1, 7, 16, 47, 48, 64, 65, 200, 256])
def test_f16_head_rows_matches_fp64(fg, N):
    """gemm_f16(head, row_map): every head, one and two W planes, the bulk row copies (ldy = pad4(N), N <= 64) and per-row
    stores (wider pitch), five row maps.  Mapped rows against fp64; unmapped rows keep the sentinel; pitch padding zero when
    ldy = pad4(N), untouched otherwise; head_bulk 0 / 1 write identical buffers."""
    M, K = 1000, 512
    maps = row_maps(M, N)
    sentinel = 7.0
    for planes in (2, 1):
        A, Wp, A64, W64 = operands(fg, M, K, K, N, "f16w2" if planes == 2 else "f16w1", N + planes)
        bias = make_bias("aligned", N, N)
        for head, fn in HEADS.items():
            act = ELU if head == 0 else NONE
            z = fn(act64(A64 @ W64.T + bias.double(), act))
            for mi, (name, (rmap, n_dst)) in enumerate(maps.items()):
                ldy = fg.ops.pad4(N) + (4 if (mi + head + planes) % 2 else 0)
                outs = []
                for bulk in (1, 0):
                    out = torch.full((n_dst, ldy), sentinel, device=dev())
                    with tuning(fg, head_bulk=bulk):
                        fg.ops.gemm_f16(A, Wp, bias, act, head, row_map=rmap, out=out, K=K, N=N)
                    outs.append(out)
                assert torch.equal(outs[0], outs[1]), f"head_bulk changes the bits ({name}, head {head}, ldy {ldy})"
                out = outs[0]
                rl = rmap.long()
                on = rl >= 0
                got = out[rl[on], :N].double()
                want = z[on]
                bound = TAU32 * max(1.0, float(want.abs().max()))
                ratio = float((got - want).abs().max()) / bound
                note(f"head_f16_{'fast' if N <= 64 else 'two_pass'}", ratio)
                assert ratio <= 1.0, f"{name} head {head} planes {planes}: {ratio:.3g}"
                mapped = torch.zeros(n_dst, dtype=torch.bool, device=dev())
                mapped[rl[on]] = True
                assert bool((out[~mapped] == sentinel).all()), name
                if ldy > N:
                    fill = 0.0 if ldy == fg.ops.pad4(N) else sentinel
                    assert bool((out[mapped][:, N:] == fill).all()), f"pitch padding of {name}, ldy {ldy}"


@pytest.mark.parametrize("N", [47, 200])
def test_f16_head_rows_peers_equal_the_single_output(fg, N):
    """gemm_f16_head_rows_peers into 1 and 3 local buffers (standing in for the ranks' gather buffers) writes every buffer
    exactly as gemm_f16 with the same row map writes its one output."""
    M, K = 1000, 512
    rmap, n_dst = row_maps(M, 3)["aligned"]
    A, Wp, _, _ = operands(fg, M, K, K, N, "f16w2", 9)
    bias = make_bias("aligned", N, 9)
    ldy = fg.ops.pad4(N)
    want = torch.full((n_dst, ldy), 3.0, device=dev())
    fg.ops.gemm_f16(A, Wp, bias, NONE, fg.ops.HEAD_LOG_SOFTMAX, row_map=rmap, out=want, K=K, N=N)
    for n_peers in (1, 3):
        bufs = [fg.ops.PeerBuffer(4 * n_dst * ldy, dev()) for _ in range(n_peers)]
        try:
            tens = [pb.tensor((n_dst, ldy)) for pb in bufs]
            for t in tens:
                t.fill_(3.0)
            fg.ops.gemm_f16_head_rows_peers(A, Wp, bias, NONE, fg.ops.HEAD_LOG_SOFTMAX, rmap, [pb.ptr for pb in bufs], ldy,
                                            K=K, N=N)
            for t in tens:
                assert torch.equal(t, want)
            del tens, t
        finally:
            torch.cuda.synchronize()
            for pb in bufs:
                pb.close()


# ------------------------------------------------------------------------------------------ 6. saturation
def check_saturated(family, got, want):
    """Elements beyond the fp16 range are +-65504 (never inf / NaN); the others keep the fp16 budget."""
    assert got.dtype == torch.float16 and bool(torch.isfinite(got).all()), f"{family}: inf / NaN in an fp16-plane output"
    over = want.abs() > F16_MAX * (1 + 2.0 ** -10)
    assert int((want > F16_MAX * 1.01).sum()) > 0 and int((want < -F16_MAX * 1.01).sum()) > 0
    assert torch.equal(got[over].double(), torch.sign(want[over]) * F16_MAX), family
    inside = want.abs() < F16_MAX * (1 - 2.0 ** -10)
    check_f16(family + "_saturating", got[inside], want[inside], tau=TAU16 * float(want.abs().max()) / float(want[inside].abs().max()))


def test_fp16_plane_outputs_saturate(fg):
    """cvt.rn.satfinite: outputs beyond +-65504 are stored as +-65504 by the transform-aggregate, the conv and gemm_f16."""
    M, K, N = 5000, 256, 512
    A, Wp, A64, W64 = operands(fg, M, K, K, N, "f16w1", 21, a_scale=8.0, w_scale=4e3)
    desc, dinv = make_groups(M, 21)
    nbr = decode(desc)
    p = A64 @ W64.T
    assert float(p.abs().max()) > 2 * F16_MAX
    got = fg.ops.gcn_transform_aggregate_f16(A, Wp, None, NONE, desc, dinv, K=K, N=N)
    check_saturated("transform_aggregate_f16", got, aggregate64(p, nbr, dinv))
    got = fg.ops.gcn_conv_aligned_f16(A, Wp, None, NONE, desc, dinv, K=K, N=N)
    check_saturated("conv_aligned_f16", got, aggregate64(p, nbr, dinv))
    got = fg.ops.gemm_f16(A, Wp, None, NONE, out_f16=True, K=K, N=N)
    check_saturated("gemm_f16", got, p)


# ------------------------------------------------------------------------------------------ 7. refusals
def test_host_side_refusals(fg):
    """Shapes the fp16-plane epilogues do not take raise FitgnnError before anything is launched (the output stays as it was)."""
    L, ptr, sp, Err = fg._lib.lib(), fg._lib.ptr, fg._lib.stream_ptr, fg._lib.FitgnnError
    M, K = 512, 128
    A_b, W_b, _, _ = operands(fg, M, K, K, 256, "bf16", 31)
    A_h, W_h, _, _ = operands(fg, M, K, K, 256, "f16w2", 32)
    desc, dinv = make_groups(M, 33)
    rmap = torch.arange(M, dtype=torch.int32, device=dev())

    def refused(rc, code, Y):
        before = Y.clone()
        with pytest.raises(Err, match=code):
            fg._lib.check(rc)
        torch.cuda.synchronize()
        assert torch.equal(Y, before)

    def ta(in_f16, a_hi, a_lo, w, N, Y, ldy, agg=True):
        return L.fitgnn_gcn_transform_aggregate_f16(in_f16, ptr(a_hi), ptr(a_lo), K, ptr(w[0]), ptr(w[1]), K, None, M, K, N, ELU,
                                                    ptr(desc) if agg else None, ptr(dinv), 0, ptr(Y), ldy, sp())

    Y = torch.full((M, 520), 5.0, dtype=torch.float16, device=dev())
    # the fused aggregation needs N > 128
    refused(ta(1, A_h, None, (W_h[0][:128], W_h[1][:128]), 128, Y, 128), "EUNSUP", Y)
    refused(ta(0, A_b[0], A_b[1], (W_b[0][:128], W_b[1][:128]), 128, Y, 128), "EUNSUP", Y)
    refused(L.fitgnn_gcn_conv_aligned_f16(ptr(A_h), K, ptr(W_h[0][:128]), None, K, None, M, K, 128, ELU, ptr(desc), ptr(dinv),
                                          ptr(Y), 128, sp()), "EUNSUP", Y)
    # an fp16 output pitch that is not a multiple of 16 bytes
    refused(ta(1, A_h, None, W_h, 256, Y, 260), "EUNSUP", Y)
    refused(ta(0, A_b[0], A_b[1], W_b, 256, Y, 260, agg=False), "EUNSUP", Y)
    refused(L.fitgnn_gcn_conv_aligned_f16(ptr(A_h), K, ptr(W_h[0]), ptr(W_h[1]), K, None, M, K, 256, ELU, ptr(desc), ptr(dinv),
                                          ptr(Y), 260, sp()), "EUNSUP", Y)
    refused(L.fitgnn_gemm_f16(ptr(A_h), K, ptr(W_h[0]), ptr(W_h[1]), K, None, None, M, K, 256, ELU, 0, ptr(Y), 260, 1, None, sp()),
            "EUNSUP", Y)
    # A_lo must match in_f16
    refused(ta(1, A_h, A_h, W_h, 256, Y, 256), "EINVAL", Y)
    refused(ta(0, A_b[0], None, W_b, 256, Y, 256), "EINVAL", Y)
    # an fp16-plane output carries no head and no row map
    refused(L.fitgnn_gemm_f16(ptr(A_h), K, ptr(W_h[0]), ptr(W_h[1]), K, None, None, M, K, 48, NONE, 1, ptr(Y), 48, 1, None, sp()),
            "EUNSUP", Y)
    refused(L.fitgnn_gemm_f16(ptr(A_h), K, ptr(W_h[0]), ptr(W_h[1]), K, None, None, M, K, 256, NONE, 0, ptr(Y), 256, 1, ptr(rmap),
                              sp()), "EUNSUP", Y)
