"""GPU: the plain dense transform (FITGNN_GEMM_BF16X3 without aggregation, its batched form fitgnn_gemm_tn, and the exact-fp32
path) against fp64 references of the operands the kernels actually read, element by element; its invariance under the tuning
switches that pick a plan; and the bounds of what it reads and writes.

Reference: bf16x3 reads hi + lo of each plane (exact in fp64); fitgnn_gemm_tn and the fp32 path read the fp32 values.
Budget of an fp32 output element (S = |row_scale| * sum_k |a_k| |w_k| + |b|):
  bf16x3, gemm_tn:   |got - want| <= 2^-24 |want| + TAU * S (+ 2^-21 after the approximate ELU)
  fp32 (FMA chain):  |got - want| <= 2^-23 |want| + (K + 1) 2^-24 S
  heads:             TAU32 * max(1, max|want|), plus the logits' own budget carried through the (log-)softmax.

Dispatch of gemm_bf16x3() (no aggregation) and the plans of tc::launch() on 148 SMs, and the cases here that select each:
  branch / plan                         condition                                                   cases
  16-column tile                        N <= 16                                                     t16-*
  32 / 48 / 64-column tiles             N <= 32 / 48 / 64                                           t32-*, t48-*, t64-*
  128-column tile                       N <= 128                                                    t128-*
  256-column tile, single CTA           N > 128 and (K <= 128 or M < 4096 or a head)                t256-*
  128-column, 16 epilogue warps         N > 128, K <= 128, no head, gemm_wide = 1                   wide-*
  CTA pair (cta_group::2), streaming    N > 128, K > 128, M >= 4096, no head, gemm_pair = 1         pair-*
  single CTA, W-stationary              resident W + 2 A stages fit, m_tiles >= 4 (sms / n_tiles)   ws-* (M = 40000, K = 64)
  CTA pair, W-stationary (bf16 hi/lo)   K in (128, 192], N > 256 (n_tiles = 2), M >= 37633          pair_ws-* (M = 40000, K = 192)
  streaming forced                      gemm_ws = 0 / gemm_pair_ws = 0                              test_plans_give_identical_bits
The fast single-pass head serves tiles of <= 64 columns, the two-pass head the 128- and 256-column tiles."""
import contextlib
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
# per unit of S: the dropped lo*lo term (<= 2^-16 |a||w| per product) and the tensor cores' fp32 accumulation; measured 5.6e-6
TAU_BF16X3 = 1e-5
# gemm_tn is compared with its fp32 operands: their split adds up to 2 * 2^-16 per product (measured 2.5e-5, at R = 1)
TAU_TN = 4e-5
TAU32 = 1e-5
ELU_ABS = 2.0 ** -21  # ex2.approx-based ELU of the tensor-core epilogue
SENT = -1024.0        # sentinel of every canary (exact in fp32 and bf16)
NONE, ELU = 0, 1
IDENT, LOGSM, SOFTMAX = 0, 1, 2
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


def vp(t):
    """Raw device address of a tensor or view (pitched and offset views included; None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def raw_gemm(fg, prec, a, a_lo, lda, w, w_lo, ldw, bias, M, K, N, act, head, y, y_lo, ldy, row_scale=None):
    """fitgnn_gemm_rowscale_bias_act_split on raw addresses: operands and outputs may be views into larger buffers."""
    return fg._lib.lib().fitgnn_gemm_rowscale_bias_act_split(prec, vp(a), vp(a_lo), lda, vp(w), vp(w_lo), ldw, vp(row_scale),
                                                             vp(bias), M, K, N, act, head, vp(y), vp(y_lo), ldy,
                                                             fg._lib.stream_ptr())


# ------------------------------------------------------------------------------------------ operands and references
def planes(fg, rows, K, seed, scale=1.0):
    """bf16 hi/lo planes [rows, K] of a seeded fp32 matrix and their exact fp64 value hi + lo."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    X = torch.randn(rows, K, generator=g, device=dev()) * scale
    hi, lo = fg.ops.split_bf16(X)
    return (hi, lo), hi.double() + lo.double()


def make_bias(kind, N, seed, shift=0.0):
    if kind is None:
        return None
    g = torch.Generator(device="cuda").manual_seed(seed + 7)
    if kind == "aligned":
        return torch.randn(N, generator=g, device=dev()) * 0.3 + shift
    b = (torch.randn(N + 1, generator=g, device=dev()) * 0.3 + shift)[1:]  # 4 bytes past a 16-byte boundary: the scalar bias path
    assert b.data_ptr() % 16 == 4
    return b


def sample_rows(M):
    """All rows of a small M; of a large one the first and last 700 and the rows around every 128-row boundary."""
    if M <= 5000:
        return torch.arange(M, device=dev())
    edges = (np.arange(128, M, 128)[:, None] + np.array([-2, -1, 0, 1])).ravel()
    idx = np.unique(np.concatenate([np.arange(700), np.arange(M - 700, M), edges]))
    return torch.from_numpy(idx[idx < M]).to(dev())


def ref64(A64, W64, bias, act, rs=None):
    """(want, S, pre): act(rs * A W^T + b) in fp64, its budget scale S = |rs| |A| |W|^T + |b|, and the pre-activation."""
    pre = A64 @ W64.T
    S = A64.abs() @ W64.abs().T
    if rs is not None:
        r = rs.double()[:, None]
        pre, S = pre * r, S * r.abs()
    if bias is not None:
        pre = pre + bias.double()
        S = S + bias.double().abs()
    return (torch.nn.functional.elu(pre) if act == ELU else pre), S, pre


def check_tc(family, got, want, S, act, tau=TAU_BF16X3):
    """Element-wise budget of a tensor-core product: 2^-24 |want| + tau S (+ the approximate ELU's absolute error)."""
    got = got.double()
    assert bool(torch.isfinite(got).all()), f"{family}: non-finite output"
    err = (got - want).abs()
    slack = U * want.abs() + (ELU_ABS if act == ELU else 0.0)
    ratio = float((err / (slack + tau * S)).max())
    note(family, ratio)
    note(family + " (tau share)", float(((err - slack).clamp(min=0) / S.clamp(min=1e-30)).max()) / tau)
    assert ratio <= 1.0, f"{family}: worst |got - want| / bound = {ratio:.3g}"


def head64(z, head):
    return {IDENT: z, LOGSM: torch.log_softmax(z, 1), SOFTMAX: torch.softmax(z, 1)}[head]


def check_head(family, got, z, ez, head):
    """(Log-)softmax of fp64 logits z whose kernel values may be off by ez (per element): TAU32 * max(1, max|want|) plus ez carried
    through the head (log-softmax: ez_i + max_row ez; softmax: p_i (ez_i + max_row ez))."""
    want = head64(z, head)
    got = got.double()
    assert bool(torch.isfinite(got).all()), f"{family}: non-finite head output"
    carry = ez + ez.max(1, keepdim=True).values
    if head == SOFTMAX:
        carry = 1.01 * want * carry
    bound = TAU32 * max(1.0, float(want.abs().max())) + carry
    ratio = float(((got - want).abs() / bound).max())
    note(family, ratio)
    assert ratio <= 1.0, f"{family}: worst |got - want| / bound = {ratio:.3g}"
    if head == SOFTMAX:
        assert float((got.sum(1) - 1).abs().max()) <= TAU32, f"{family}: softmax rows do not sum to 1"
    elif head == LOGSM:
        assert float(got.max(1).values.max()) <= 0.0, f"{family}: log-softmax above 0"


def split_ok(y, hi, lo):
    """hi == rn_bf16(y), lo == rn_bf16(y - hi) against the fp32 result of the same operands."""
    want_hi = y.to(torch.bfloat16)
    return torch.equal(hi, want_hi) and torch.equal(lo, (y - want_hi.float()).to(torch.bfloat16))


# ------------------------------------------------------------------------------------------ 1. dispatch matrix vs fp64
DISPATCH_CASES = [
    # id: plan-M-K-N                                 M      K    N     bias          act  switches
    pytest.param(1, 8, 1, "aligned", NONE, {}, id="t16-M1-K8-N1"),
    pytest.param(127, 64, 16, None, ELU, {}, id="t16-M127-K64-N16"),
    pytest.param(128, 72, 17, "misaligned", NONE, {}, id="t32-M128-K72-N17"),
    pytest.param(129, 136, 32, "aligned", ELU, {}, id="t32-M129-K136-N32"),
    pytest.param(255, 520, 33, None, NONE, {}, id="t48-M255-K520-N33"),
    pytest.param(256, 8, 47, "misaligned", ELU, {}, id="t48-M256-K8-N47"),
    pytest.param(257, 128, 48, "aligned", NONE, {}, id="t48-M257-K128-N48"),
    pytest.param(4095, 192, 49, "aligned", ELU, {}, id="t64-M4095-K192-N49"),
    pytest.param(4096, 72, 64, None, NONE, {}, id="t64-M4096-K72-N64"),
    pytest.param(4097, 64, 65, "misaligned", ELU, {}, id="t128-M4097-K64-N65"),
    pytest.param(1, 520, 127, "aligned", NONE, {}, id="t128-M1-K520-N127"),
    pytest.param(129, 136, 128, None, ELU, {}, id="t128-M129-K136-N128"),
    pytest.param(255, 64, 129, "aligned", ELU, {}, id="t256-M255-K64-N129"),
    pytest.param(4097, 128, 255, "misaligned", NONE, {}, id="t256-M4097-K128-N255"),
    pytest.param(4095, 192, 256, "aligned", ELU, {}, id="t256-M4095-K192-N256"),
    pytest.param(257, 520, 1436, "aligned", ELU, {}, id="t256-M257-K520-N1436"),
    pytest.param(4096, 136, 257, "aligned", NONE, {}, id="pair-M4096-K136-N257"),
    pytest.param(4097, 520, 511, None, ELU, {}, id="pair-M4097-K520-N511"),
    pytest.param(4097, 192, 1436, "misaligned", NONE, {}, id="pair-M4097-K192-N1436"),
    pytest.param(4097, 72, 257, "aligned", ELU, {"gemm_wide": 1}, id="wide-M4097-K72-N257"),
    pytest.param(40000, 128, 512, None, NONE, {"gemm_wide": 1}, id="wide_ws-M40000-K128-N512"),
    pytest.param(40000, 64, 511, "aligned", ELU, {}, id="ws-M40000-K64-N511"),
    pytest.param(40000, 192, 512, "aligned", ELU, {}, id="pair_ws-M40000-K192-N512"),
]


@pytest.mark.parametrize("M,K,N,bias_kind,act,switches", DISPATCH_CASES)
def test_dispatch_matches_fp64(fg, request, M, K, N, bias_kind, act, switches):
    """act(A W^T + b) element-wise against fp64 at every tile width and plan; with N % 8 == 0 the split planes of the same
    call are the fp32 result rounded (hi) and its remainder rounded (lo)."""
    family = request.node.callspec.id.split("-")[0]
    seed = M + 3 * K + 7 * N
    A, A64 = planes(fg, M, K, seed)
    W, W64 = planes(fg, N, K, seed + 1, scale=K ** -0.5)
    bias = make_bias(bias_kind, N, seed)
    with tuning(fg, **switches):
        got = fg.ops.gemm_bias_act(A, W, bias, act, K=K, N=N, precision=fg.ops.GEMM_BF16X3)
        split = fg.ops.gemm_bias_act(A, W, bias, act, K=K, N=N, precision=fg.ops.GEMM_BF16X3, split_out=True) if N % 8 == 0 else None
    rows = sample_rows(M)
    want, S, _ = ref64(A64[rows], W64, bias, act)
    check_tc(f"bf16x3 {family}", got[rows], want, S, act)
    if split is not None:
        assert split_ok(got, *split), "split planes differ from the rounded fp32 result"


@pytest.mark.parametrize("M,K,N,head", [(300, 136, 47, IDENT), (4097, 192, 512, IDENT), (700, 64, 33, LOGSM), (700, 136, 200, LOGSM),
                                        (700, 72, 129, SOFTMAX), (700, 520, 64, SOFTMAX)])
def test_row_scale_matches_fp64(fg, M, K, N, head):
    """head(act(rs[m] (A W^T)[m] + b)) with a row scale that includes zero and negative factors, on the 48-, 64-, 128- and
    256-column tiles and the CTA pair; the two-pass head (N > 64) must use the scaled row for its statistics too."""
    seed = M + K + N + head
    A, A64 = planes(fg, M, K, seed)
    W, W64 = planes(fg, N, K, seed + 1, scale=K ** -0.5)
    bias = make_bias("aligned", N, seed)
    g = torch.Generator(device="cuda").manual_seed(seed)
    rs = torch.rand(M, generator=g, device=dev()) * 2.0
    rs[::17] = 0.0
    rs[5::13] *= -1.0
    act = ELU if head == IDENT else NONE
    got = fg.ops.gemm_bias_act(A, W, bias, act, head, K=K, N=N, precision=fg.ops.GEMM_BF16X3, row_scale=rs)
    z, S, _ = ref64(A64, W64, bias, act, rs)
    if head == IDENT:
        check_tc("bf16x3 row_scale", got, z, S, act)
        if N % 8 == 0:
            hi, lo = fg.ops.gemm_bias_act(A, W, bias, act, K=K, N=N, precision=fg.ops.GEMM_BF16X3, row_scale=rs, split_out=True)
            assert split_ok(got, hi, lo)
    else:
        check_head("head row_scale", got, z, U * z.abs() + TAU_BF16X3 * S, head)


# ------------------------------------------------------------------------------------------ 2. plan invariance
PLAN_SHAPES = [(40000, 64, 512), (40000, 192, 512), (4097, 520, 1436), (4097, 72, 257), (3000, 136, 64), (300, 8, 17)]
SWITCHES = [{"gemm_ws": 0}, {"gemm_pair": 0}, {"gemm_pair_ws": 0}, {"gemm_wide": 1}, {"gemm_prefetch": 1}, {"sm_reserve": 6},
            {"gemm_ws": 0, "gemm_pair": 0, "sm_reserve": 6}, {"gemm_wide": 1, "gemm_prefetch": 1, "sm_reserve": 6},
            {"gemm_pair_ws": 0, "gemm_prefetch": 1}, {"gemm_wide": 1, "gemm_ws": 0}]


@pytest.mark.parametrize("M,K,N", PLAN_SHAPES)
def test_plans_give_identical_bits(fg, M, K, N):
    """Every plan accumulates each output element in the same k order: the fp32 output and the split planes are bit-identical
    under gemm_ws, gemm_pair, gemm_pair_ws, gemm_wide, gemm_prefetch, sm_reserve and combinations."""
    A, _ = planes(fg, M, K, M + N)
    W, _ = planes(fg, N, K, M + N + 1, scale=K ** -0.5)
    bias = make_bias("aligned", N, N)

    def run():
        y = fg.ops.gemm_bias_act(A, W, bias, ELU, K=K, N=N, precision=fg.ops.GEMM_BF16X3)
        s = fg.ops.gemm_bias_act(A, W, bias, ELU, K=K, N=N, precision=fg.ops.GEMM_BF16X3, split_out=True) if N % 8 == 0 else None
        return y, s

    y0, s0 = run()
    for sw in SWITCHES:
        with tuning(fg, **sw):
            y1, s1 = run()
        assert torch.equal(y0, y1), f"fp32 output differs under {sw}"
        if s0 is not None:
            assert torch.equal(s0[0], s1[0]) and torch.equal(s0[1], s1[1]), f"split planes differ under {sw}"


def test_column_and_row_slices_give_identical_bits(fg):
    """W[:n] gives the first n columns of the full product (tiles of 16 .. 256 columns and the CTA pair against each other), and
    A[:m] its first m rows."""
    M, K, N = 4100, 136, 512
    A, _ = planes(fg, M, K, 11)
    W, _ = planes(fg, N, K, 12, scale=K ** -0.5)
    bias = make_bias("misaligned", N, 13)
    full = fg.ops.gemm_bias_act(A, W, bias, ELU, K=K, N=N, precision=fg.ops.GEMM_BF16X3)
    for n in (16, 32, 48, 64, 128, 256, 300):
        part = fg.ops.gemm_bias_act(A, (W[0][:n], W[1][:n]), bias[:n], ELU, K=K, N=n, precision=fg.ops.GEMM_BF16X3)
        assert torch.equal(part, full[:, :n]), f"W[:{n}]"
    for m in (1, 127, 128, 129, 1000, 4095):
        part = fg.ops.gemm_bias_act((A[0][:m], A[1][:m]), W, bias, ELU, K=K, N=N, precision=fg.ops.GEMM_BF16X3)
        assert torch.equal(part, full[:m]), f"A[:{m}]"


# ------------------------------------------------------------------------------------------ 3. bounds of what is written
CANARY_SHAPES = [(129, 64, 16), (300, 72, 47), (257, 136, 33), (1000, 136, 200), (4097, 192, 300)]


def pitched(rows, ldy, dtype, offset_elems=0):
    """A sentinel-filled [rows, ldy] buffer starting offset_elems past a 256-byte boundary, and the flat storage behind it."""
    flat = torch.full((offset_elems + rows * ldy,), SENT, dtype=dtype, device=dev())
    return flat[offset_elems:].view(rows, ldy), flat


def outside_untouched(buf, flat, M, N, offset_elems, zero_to=None):
    """Nothing outside [M, N] changed, except columns [N, zero_to) of rows < M, which must hold zeros."""
    mask = torch.ones_like(buf, dtype=torch.bool)
    mask[:M, :N] = False
    if zero_to is not None and zero_to > N:
        mask[:M, N:zero_to] = False
        if not bool((buf[:M, N:zero_to] == 0).all()):
            return False
    return bool((buf[mask] == SENT).all()) and bool((flat[:offset_elems] == SENT).all())


@pytest.mark.parametrize("M,K,N", CANARY_SHAPES)
def test_outputs_stay_inside_M_by_N(fg, M, K, N):
    """Y is a view into a sentinel-filled buffer with 5 extra rows and ldy > N.  The per-thread path (odd ldy; a base 4 bytes past
    alignment) writes exactly [M, N]; the TMA-store path (ldy % 4 == 0, aligned; split planes with ldy % 8 == 0) also writes zeros
    up to the 16-byte boundary after column N (pad4(N) fp32, pad8(N) bf16), heads included; every path gives the bits of a call
    into a tight buffer."""
    A, _ = planes(fg, M, K, M + N)
    W, _ = planes(fg, N, K, M + N + 1, scale=K ** -0.5)
    bias = make_bias("aligned", N, N)
    BF = fg.ops.GEMM_BF16X3
    heads = (IDENT, LOGSM, SOFTMAX) if N <= 256 else (IDENT,)
    for head in heads:
        act = ELU if head == IDENT else NONE
        tight = fg.ops.gemm_bias_act(A, W, bias, act, head, K=K, N=N, precision=BF)
        for name, ldy, off, zero_to in (("tma", fg.ops.pad4(N) + 8, 0, fg.ops.pad4(N)), ("odd_ldy", N + (1 if N % 2 == 0 else 2), 0, None),
                                        ("offset_4B", fg.ops.pad4(N) + 4, 1, None)):
            buf, flat = pitched(M + 5, ldy, torch.float32, off)
            fg._lib.check(raw_gemm(fg, BF, A[0], A[1], K, W[0], W[1], K, bias, M, K, N, act, head, buf, None, ldy))
            assert torch.equal(buf[:M, :N], tight), f"{name} head {head}: bits differ from the tight call"
            assert outside_untouched(buf, flat, M, N, off, zero_to), f"{name} head {head}: wrote outside [M, N]"
    hi_t, lo_t = fg.ops.gemm_bias_act(A, W, bias, ELU, K=K, N=N, precision=BF, split_out=True) if N % 8 == 0 else (None, None)
    ldy = fg.ops.pad8(N) + 8
    hi, fhi = pitched(M + 5, ldy, torch.bfloat16)
    lo, flo = pitched(M + 5, ldy, torch.bfloat16)
    fg._lib.check(raw_gemm(fg, BF, A[0], A[1], K, W[0], W[1], K, bias, M, K, N, ELU, IDENT, hi, lo, ldy))
    assert outside_untouched(hi, fhi, M, N, 0, fg.ops.pad8(N)) and outside_untouched(lo, flo, M, N, 0, fg.ops.pad8(N)), \
        "split planes wrote outside [M, pad8(N)) or not zeros past N"
    y = fg.ops.gemm_bias_act(A, W, bias, ELU, K=K, N=N, precision=BF)
    assert split_ok(y, hi[:M, :N], lo[:M, :N])
    if hi_t is not None:
        assert torch.equal(hi[:M, :N], hi_t) and torch.equal(lo[:M, :N], lo_t)


def row_maps(M, seed):
    """name -> (row_map int32 [M], number of destination rows)."""
    rng = np.random.default_rng(seed)
    ident = np.arange(M)
    warp = np.where((ident >= 64) & (ident < 96), -1, ident - 32 * (ident >= 96))  # a whole warp of -1
    perm = rng.permutation(M)
    sub = np.sort(rng.choice(2 * M, M, replace=False))  # a sorted subset of 2M rows: the gaps are never mapped
    sub[rng.random(M) < 0.1] = -1
    maps = {"warp_of_pad": (warp, M - 32), "permutation": (perm, M), "subset_with_gaps": (sub, 2 * M)}
    return {k: (torch.from_numpy(v.astype(np.int32)).to(dev()), n) for k, (v, n) in maps.items()}


@pytest.mark.parametrize("N", [7, 47, 64, 65, 200])
def test_head_rows_bounds_and_values(fg, N):
    """gemm_head_rows (bf16x3): mapped rows against fp64; rows with row_map < 0 and rows never mapped keep the sentinel; pitch
    columns are zero when ldy == pad4(N) (bulk row copies and per-row stores alike) and untouched when ldy > pad4(N); head_bulk 0
    and 1 write identical buffers."""
    M, K = 1000, 136
    A, A64 = planes(fg, M, K, N)
    W, W64 = planes(fg, N, K, N + 1, scale=K ** -0.5)
    bias = make_bias("aligned", N, N)
    for head in (IDENT, LOGSM, SOFTMAX):
        act = ELU if head == IDENT else NONE
        z, S, _ = ref64(A64, W64, bias, act)
        for mi, (name, (rmap, n_dst)) in enumerate(row_maps(M, N + head).items()):
            for ldy in (fg.ops.pad4(N), fg.ops.pad4(N) + 4):
                outs = []
                for bulk in (1, 0):
                    out = torch.full((n_dst, ldy), SENT, device=dev())
                    with tuning(fg, head_bulk=bulk):
                        fg.ops.gemm_head_rows(A, W, bias, act, head, rmap, out, K=K, N=N)
                    outs.append(out)
                assert torch.equal(outs[0], outs[1]), f"head_bulk changes the bits ({name}, head {head}, ldy {ldy})"
                out = outs[0]
                rl = rmap.long()
                on = rl >= 0
                got = out[rl[on], :N]
                if head == IDENT:
                    check_tc("head_rows identity", got, z[on], S[on], act)
                else:
                    check_head(f"head_rows {'fast' if N <= 64 else 'two_pass'}", got, z[on], U * z[on].abs() + TAU_BF16X3 * S[on],
                               head)
                mapped = torch.zeros(n_dst, dtype=torch.bool, device=dev())
                mapped[rl[on]] = True
                assert bool((out[~mapped] == SENT).all()), f"{name}: an unmapped row was written"
                if ldy > N:
                    fill = 0.0 if ldy == fg.ops.pad4(N) else SENT
                    assert bool((out[mapped][:, N:] == fill).all()), f"pitch columns of {name}, ldy {ldy}"


# ------------------------------------------------------------------------------------------ 4. bounds of what is read
@pytest.mark.parametrize("M,K,N", [(300, 72, 47), (1000, 136, 200), (4097, 192, 257), (40000, 64, 511)])
def test_reads_stay_inside_K_and_N(fg, M, K, N):
    """A and W planes with a pitch wider than K whose extra columns hold NaN, NaN rows past M in A and past N in W: the output is
    finite and bit-identical to a call on tight buffers."""
    A, _ = planes(fg, M, K, M + N)
    W, _ = planes(fg, N, K, M + N + 1, scale=K ** -0.5)
    bias = make_bias("aligned", N, N)
    BF = fg.ops.GEMM_BF16X3
    tight = fg.ops.gemm_bias_act(A, W, bias, ELU, K=K, N=N, precision=BF)
    lda, ldw = K + 16, K + 8

    def nan_pad(p, rows, ld):
        buf = torch.full((rows, ld), float("nan"), dtype=torch.bfloat16, device=dev())
        buf[: p.shape[0], : p.shape[1]] = p
        return buf

    Aw = [nan_pad(p, M + 3, lda) for p in A]
    Ww = [nan_pad(p, N + 5, ldw) for p in W]
    y = torch.empty(M, N, device=dev())
    fg._lib.check(raw_gemm(fg, BF, Aw[0], Aw[1], lda, Ww[0], Ww[1], ldw, bias, M, K, N, ELU, IDENT, y, None, N))
    assert bool(torch.isfinite(y).all()) and torch.equal(y, tight)
    if N <= 256:
        y = torch.empty(M, N, device=dev())
        fg._lib.check(raw_gemm(fg, BF, Aw[0], Aw[1], lda, Ww[0], Ww[1], ldw, bias, M, K, N, NONE, LOGSM, y, None, N))
        assert torch.equal(y, fg.ops.gemm_bias_act(A, W, bias, NONE, LOGSM, K=K, N=N, precision=BF))


def test_bias_alignment_and_null_bias_give_identical_bits(fg):
    """At every tile width and on the CTA pair: a bias 4 bytes past alignment (the scalar bias path) gives the bits of an aligned
    copy, and bias = NULL the bits of a zero bias."""
    K = 136
    for M, N in ((300, 16), (300, 32), (300, 48), (300, 64), (300, 128), (300, 256), (4097, 300)):
        A, _ = planes(fg, M, K, N)
        W, _ = planes(fg, N, K, N + 1, scale=K ** -0.5)
        mis = make_bias("misaligned", N, N)
        for head in (IDENT, LOGSM) if N <= 256 else (IDENT,):
            act = ELU if head == IDENT else NONE

            def run(b):
                return fg.ops.gemm_bias_act(A, W, b, act, head, K=K, N=N, precision=fg.ops.GEMM_BF16X3)

            assert torch.equal(run(mis), run(mis.clone())), f"N {N} head {head}: misaligned bias"
            assert torch.equal(run(None), run(torch.zeros(N, device=dev()))), f"N {N} head {head}: NULL bias"


def test_empty_M_and_host_side_refusals(fg):
    """M = 0 returns OK without writing; shapes the transform does not take raise FitgnnError before anything is launched and the
    output keeps its sentinel."""
    L, Err = fg._lib.lib(), fg._lib.FitgnnError
    BF, F32 = fg.ops.GEMM_BF16X3, fg.ops.GEMM_FP32
    M, K = 256, 64
    A, _ = planes(fg, M, K, 1)
    W, _ = planes(fg, 300, K, 2)
    Af = torch.randn(M, K, device=dev())
    Y = torch.full((M, 304), SENT, device=dev())
    Yb = torch.full((M, 304), SENT, dtype=torch.bfloat16, device=dev())
    rs = torch.ones(M, device=dev())

    def refused(rc, code):
        with pytest.raises(Err, match=code):
            fg._lib.check(rc)
        torch.cuda.synchronize()
        assert bool((Y == SENT).all()) and bool((Yb == SENT).all())

    assert raw_gemm(fg, BF, A[0], A[1], K, W[0], W[1], K, None, 0, K, 300, ELU, IDENT, Y, None, 304) == 0
    assert raw_gemm(fg, F32, Af, None, K, Af, None, K, None, 0, K, 200, NONE, LOGSM, Y, None, 304) == 0
    torch.cuda.synchronize()
    assert bool((Y == SENT).all())
    refused(raw_gemm(fg, BF, A[0], A[1], K, W[0], W[1], K, None, M, K, 257, NONE, LOGSM, Y, None, 304), "EUNSUP")  # head, N > 256
    refused(raw_gemm(fg, BF, A[0], A[1], K, W[0], W[1], K, None, M, K, 64, NONE, LOGSM, Yb, Yb, 304), "EUNSUP")  # split + head
    refused(raw_gemm(fg, F32, Af, None, K, Af, None, K, None, M, K, 64, NONE, IDENT, Y, None, 304, row_scale=rs), "EUNSUP")
    refused(raw_gemm(fg, BF, A[0], A[1], K - 8, W[0], W[1], K, None, M, K, 64, NONE, IDENT, Y, None, 304), "EINVAL")  # lda < K
    # a plane pitch that is not a multiple of 8 elements cannot be described to the TMA unit
    Ap = torch.zeros(M, K + 4, dtype=torch.bfloat16, device=dev())
    refused(raw_gemm(fg, BF, Ap, Ap, K + 4, W[0], W[1], K, None, M, K, 64, NONE, IDENT, Y, None, 304), "EUNSUP")
    refused(raw_gemm(fg, BF, A[0], A[1], K, W[0], W[1], K, None, M, K, 64, NONE, IDENT, Yb, Yb, 68), "EUNSUP")  # split pitch 68


# ------------------------------------------------------------------------------------------ 5. heads
@pytest.mark.parametrize("N", [1, 2, 16, 17, 32, 33, 47, 48, 49, 64, 65, 128, 129, 200, 256])
def test_heads_match_fp64(fg, N):
    """log_softmax and softmax fused into the transform: plain logits, ELU before the head, and logits with a spread of ~200
    shifted by +100 (an unshifted exp overflows) including rows of equal logits (A row = 0, constant bias)."""
    M, K = 700, 136
    A, A64 = planes(fg, M, K, N)
    Aw, Aw64 = planes(fg, M, K, N + 2)
    for p in Aw:
        p[5] = 0
        p[M - 1] = 0
    Aw64[5] = 0
    Aw64[M - 1] = 0
    W, W64 = planes(fg, N, K, N + 1, scale=K ** -0.5)
    Ww, Ww64 = planes(fg, N, K, N + 3, scale=50.0 * K ** -0.5)
    fam = "fast" if N <= 64 else "two_pass"
    for head in (LOGSM, SOFTMAX):
        for variant, (a, a64, w, w64, bias, act) in {
                "plain": (A, A64, W, W64, make_bias("aligned", N, N), NONE),
                "elu": (A, A64, W, W64, make_bias("misaligned", N, N), ELU),
                "wide": (Aw, Aw64, Ww, Ww64, torch.full((N,), 100.0, device=dev()), NONE)}.items():
            got = fg.ops.gemm_bias_act(a, w, bias, act, head, K=K, N=N, precision=fg.ops.GEMM_BF16X3)
            z, S, _ = ref64(a64, w64, bias, act)
            if variant == "wide":
                assert float(z.max()) > 88.0
                assert N < 16 or float((z.max(1).values - z.min(1).values).max()) > 150.0
            ez = U * z.abs() + TAU_BF16X3 * S + (ELU_ABS if act == ELU else 0.0)
            check_head(f"head {fam}", got, z, ez, head)
            if variant == "wide":
                flat = head64(torch.zeros(1, N, dtype=torch.float64, device=dev()), head)
                for r in (5, M - 1):
                    assert float((got[r].double() - flat[0]).abs().max()) <= TAU32 * max(1.0, float(flat.abs().max()))


# ------------------------------------------------------------------------------------------ 6. fitgnn_gemm_tn
TN_CASES = [(1, 1, 1), (1, 255, 129), (63, 7, 16), (63, 1, 257), (64, 255, 17), (64, 7, 1), (65, 257, 33), (65, 255, 16),
            (4095, 7, 129), (4095, 257, 17), (4096, 257, 257), (4096, 1, 33), (4097, 1, 16), (4097, 7, 257), (8193, 255, 1),
            (8193, 257, 129), (5000, 64, 32), (5000, 128, 128), (9000, 33, 256)]


@pytest.mark.parametrize("R,out,inn", TN_CASES)
def test_gemm_tn_matches_fp64(fg, R, out, inn):
    """dW = G^T A over R rows against fp64 of the fp32 operands, element-wise; bit-identical across runs, under sm_reserve and
    gemm_pair (the reduction order is fixed), and for row-strided G and A."""
    g = torch.Generator(device="cuda").manual_seed(R + out + inn)
    Gw = torch.randn(R, out + 5, generator=g, device=dev())
    Aw = torch.randn(R, inn + 3, generator=g, device=dev())
    G, A = Gw[:, :out], Aw[:, :inn]
    Gc, Ac = G.contiguous(), A.contiguous()
    got = fg.ops.gemm_tn(Gc, Ac)
    G64, A64 = Gc.double(), Ac.double()
    want = G64.T @ A64
    S = G64.abs().T @ A64.abs()
    check_tc("gemm_tn", got, want, S, NONE, tau=TAU_TN)
    assert torch.equal(got, fg.ops.gemm_tn(Gc, Ac))
    assert torch.equal(got, fg.ops.gemm_tn(G, A)), "row-strided operands"
    for sw in ({"sm_reserve": 6}, {"gemm_pair": 0}):
        with tuning(fg, **sw):
            assert torch.equal(got, fg.ops.gemm_tn(Gc, Ac)), f"differs under {sw}"


# ------------------------------------------------------------------------------------------ 7. exact-fp32 path
@pytest.mark.parametrize("M,K,N", [(300, 136, 47), (1000, 100, 200), (129, 37, 257), (2000, 520, 130)])
def test_fp32_loaders_and_bounds(fg, M, K, N):
    """GEMM_FP32 against the FMA-chain bound (K + 1) 2^-24 S; the vector loader (lda % 4 == 0, 16-byte aligned) and the scalar
    one (odd pitch; a base 4 bytes past alignment) give the same bits; outputs outside [M, N] keep the sentinel."""
    F32 = fg.ops.GEMM_FP32
    g = torch.Generator(device="cuda").manual_seed(M + K + N)
    A = torch.randn(M, K, generator=g, device=dev())
    W = torch.randn(N, K, generator=g, device=dev()) * K ** -0.5
    bias = make_bias("aligned", N, N)
    for act in (NONE, ELU):
        got = fg.ops.gemm_bias_act(A, W, bias, act, K=K, N=N)
        want, S, _ = ref64(A.double(), W.double(), bias, act)
        err = (got.double() - want).abs()
        ratio = float((err / (2 * U * want.abs() + (K + 1) * U * S)).max())
        note("fp32", ratio)
        assert ratio <= 1.0, ratio
        for name, a_pitch, a_off, w_pitch, w_off in (("odd_pitch", K + 1, 0, K + 3, 0), ("offset_4B", K, 1, K, 1),
                                                     ("A_only", K + 1, 0, K, 0), ("W_only", K, 0, K, 1)):
            a_buf, _ = pitched(M, a_pitch, torch.float32, a_off)
            w_buf, _ = pitched(N, w_pitch, torch.float32, w_off)
            a_buf[:, :K] = A
            w_buf[:, :K] = W
            ldy = N + 3
            y, flat = pitched(M + 4, ldy, torch.float32, 1)
            fg._lib.check(raw_gemm(fg, F32, a_buf, None, a_pitch, w_buf, None, w_pitch, bias, M, K, N, act, IDENT, y, None, ldy))
            assert torch.equal(y[:M, :N], got), f"{name}: the scalar loader changes the bits"
            assert outside_untouched(y, flat, M, N, 1), f"{name}: wrote outside [M, N]"


@pytest.mark.parametrize("N", [33, 257, 1000])
def test_fp32_row_softmax(fg, N):
    """GEMM_FP32 with a head (row_softmax, any N) against fp64; the pitch columns and the rows after M are untouched."""
    M, K = 500, 72
    g = torch.Generator(device="cuda").manual_seed(N)
    A = torch.randn(M, K, generator=g, device=dev())
    W = torch.randn(N, K, generator=g, device=dev()) * (4.0 * K ** -0.5)
    bias = make_bias("aligned", N, N)
    z, S, _ = ref64(A.double(), W.double(), bias, NONE)
    ez = 2 * U * z.abs() + (K + 1) * U * S
    for head in (LOGSM, SOFTMAX):
        ldy = N + 3
        y, flat = pitched(M + 2, ldy, torch.float32)
        fg._lib.check(raw_gemm(fg, fg.ops.GEMM_FP32, A, None, K, W, None, K, bias, M, K, N, NONE, head, y, None, ldy))
        check_head("fp32 row_softmax", y[:M, :N], z, ez, head)
        assert outside_untouched(y, flat, M, N, 0)
