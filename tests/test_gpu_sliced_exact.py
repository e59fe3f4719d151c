"""The sliced tensor-core products (csrc/umma_gemm.cu) and the dense MLP built on them (csrc/dense_mlp.cu) against the
host model of tests/_sliced_model.py, bit for bit.

The int8 kinds are deterministic integer arithmetic: the slicing kernels must write the model's digits and exponents
byte for byte and the products must equal the model's fp64 results exactly (torch.equal), entry by entry.  That catches
what a whole-matrix error scale cannot: an exponent read from the wrong row or column of a tile, a wrong digit in a
small row, an error in a row 1e-6 of the largest one.  The operands spread their row and column maxima over many
binades and have all-zero rows and columns (the exponent sentinel path); the shapes straddle the 128 x 64 tiles and the
64-byte K blocks.  fp32 (TF32) products accumulate in fp32 in tensor memory, which the host cannot reproduce: they are
held per entry to a bound derived below."""
import numpy as np
import pytest
import torch

import _sliced_model as sm

pytestmark = pytest.mark.gpu

KIND_IDS = {sm.I8: "I8", sm.I8X: "I8X", sm.TF32: "TF32"}


def _sl():
    from pnode_b200 import sliced
    return sliced


def _kernel_slices(s):
    """(slices [S, rows, k] as int8 digits or int32 float bit patterns, exponents or None) of a Sliced operand: the
    first k entries of every pitch row."""
    S = 2 if s.kind == sm.TF32 else sm.KINDS[s.kind].S
    pitch = s.buf.numel() // (S * s.rows)
    if s.kind == sm.TF32:
        return s.buf.view(torch.int32).view(S, s.rows, pitch // 4)[:, :, :s.k].cpu().numpy(), None
    return s.buf.view(torch.int8).view(S, s.rows, pitch)[:, :, :s.k].cpu().numpy(), s.exp.cpu().numpy().astype(np.int64)


def _model_slices(x, kind):
    """The model's slices of the operand x (rows = operand rows)."""
    if kind == sm.TF32:
        hi, lo = sm.tf32_split(x)
        return np.stack([hi.view(np.int32), lo.view(np.int32)]), None
    return sm.slice_rows(x, kind)


def _source(rows, cols, kind, seed):
    """Rows and columns scaled over 2^-300 ... 2^300 (fp32: 2^-60 ... 2^60), entries within a row spread over 2^-40,
    one all-zero row and one all-zero column."""
    g = np.random.default_rng(seed)
    span = 60 if kind == sm.TF32 else 300
    x = g.standard_normal((rows, cols)) * 2.0 ** g.integers(-span, span + 1, (rows, 1)).astype(np.float64)
    x *= 2.0 ** g.integers(-20, 1, (1, cols)).astype(np.float64)
    x[:, ::3] *= 2.0 ** -g.integers(0, 21, (rows, len(range(0, cols, 3)))).astype(np.float64)
    if rows > 2:
        x[rows // 2] = 0.0
    if cols > 2:
        x[:, cols // 3] = 0.0
    return x.astype(np.float32) if kind == sm.TF32 else x


def _device(x, pad):
    """x on the device with a leading dimension of cols + pad (pad > 0: a strided source)."""
    dt = torch.float32 if x.dtype == np.float32 else torch.float64
    wide = torch.full((x.shape[0], x.shape[1] + pad), float("nan"), dtype=dt, device="cuda")
    wide[:, :x.shape[1]] = torch.from_numpy(x).cuda()
    return wide[:, :x.shape[1]]


def _check_slices(s, x, kind, what):
    q, e = _kernel_slices(s)
    mq, me = _model_slices(x, kind)
    assert q.shape == mq.shape, (what, q.shape, mq.shape)
    bad = np.argwhere(q != mq)
    assert bad.size == 0, "%s: %d digits differ, first (slice, row, col) %s: kernel %d, model %d" % (
        what, len(bad), tuple(bad[0]), q[tuple(bad[0])], mq[tuple(bad[0])])
    if e is not None:
        assert np.array_equal(e, me), (what, np.argwhere(e != me)[:5].ravel(), e[e != me][:5], me[e != me][:5])


@pytest.mark.parametrize("kind", [sm.I8, sm.I8X, sm.TF32], ids=KIND_IDS.get)
@pytest.mark.parametrize("rows,k,pad", [(37, 1, 0), (50, 5, 3), (20, 63, 0), (33, 333, 0), (130, 65, 7), (3, 1000, 24)])
def test_slice_rows_match_the_model(kind, rows, k, pad):
    sl = _sl()
    x = _source(rows, k, kind, seed=rows * 7 + k)
    s = sl.slice_rows(_device(x, pad), extended=kind == sm.I8X)
    _check_slices(s, x, kind, "slice_rows %dx%d" % (rows, k))


@pytest.mark.parametrize("kind", [sm.I8, sm.I8X, sm.TF32], ids=KIND_IDS.get)
@pytest.mark.parametrize("rows", [100, 256, 257, 1000])
def test_slice_cols_and_column_sums_match(kind, rows):
    """Column slicing over one and several 256-row exponent blocks (atomicMax) and 128-row slicing blocks, strided
    source, and the column sums: colsum += coef * sum_r x[r][c] within 1e-15 (fp32: 1e-6) of coef * sum_r |x[r][c]|."""
    sl = _sl()
    cols = 70
    x = _source(rows, cols, kind, seed=rows)
    x[rows - 1, 5] = x[0, 5] * 3.0  # column maxima in the last row block
    colsum = torch.zeros((cols,), dtype=torch.float32 if kind == sm.TF32 else torch.float64, device="cuda")
    coef = -0.75
    s = sl.slice_cols(_device(x, 9), colsum=colsum, coef=coef, extended=kind == sm.I8X)
    _check_slices(s, np.ascontiguousarray(x.T), kind, "slice_cols %dx%d" % (rows, cols))
    from fractions import Fraction
    got = colsum.cpu().double().numpy()
    for c in range(cols):
        exact = Fraction(coef) * sum(Fraction(float(v)) for v in x[:, c])
        scale = abs(coef) * float(np.abs(x[:, c].astype(np.float64)).sum())
        tol = 1e-6 if kind == sm.TF32 else 1e-15
        assert abs(float(Fraction(float(got[c])) - exact)) <= tol * scale, c


# ---- int8 products: bit-identical to the model ---------------------------------------------------------------------
EPILOGUES = [dict(), dict(bias=True), dict(bias=True, relu=True), dict(mask=True, alpha=-0.3),
             dict(accumulate=True, alpha=0.2), dict(bias=True, relu=True, mask=True, accumulate=True, alpha=1.7, wide=True),
             dict(mask=True, alpha=3.0, wide=True)]


def _operands(M, N, K, seed):
    """A [M][K], B [N][K]: row and column maxima over 2^-60 ... 2^60, entries within a row spread over 2^-30, a zero
    row of A and a zero row of B (a zero column of C).  Products stay far above the fp64 underflow range, so the
    power-of-two scalings of the epilogue are exact."""
    g = np.random.default_rng(seed)
    a = g.standard_normal((M, K)) * 2.0 ** g.integers(-60, 61, (M, 1)).astype(np.float64)
    b = g.standard_normal((N, K)) * 2.0 ** g.integers(-60, 61, (N, 1)).astype(np.float64)
    a = np.where(g.random((M, K)) < 0.3, a * 2.0 ** -g.integers(0, 31, (M, K)).astype(np.float64), a)
    if M > 2:
        a[M // 2] = 0.0
    if N > 2:
        b[N // 3] = 0.0
    return a, b


def _run_product(kind, a, b, epi, seed):
    """(kernel result, model result, untouched margins equal) for one product with the epilogue options epi."""
    sl = _sl()
    M, N = a.shape[0], b.shape[0]
    g = np.random.default_rng(seed)
    scale = np.abs(a).max(1)[:, None] * np.abs(b).max(1)[None, :]
    bias = g.standard_normal(N) * scale.max(0) if epi.get("bias") else None
    mask = None
    if epi.get("mask"):
        mask = g.standard_normal((M, N))
        mask[g.random((M, N)) < 0.1] = 0.0  # mask > 0 is strict
    acc = g.standard_normal((M, N)) * scale if epi.get("accumulate") else None
    wide = epi.get("wide", False)
    pad = 5 if wide else 0
    out_full = torch.full((M, N + 2 * pad), -7.25, dtype=torch.float64, device="cuda")
    out = out_full[:, pad:pad + N]  # wide: ldc > N, and the columns on both sides must stay untouched
    if acc is not None:
        out.copy_(torch.from_numpy(acc))
    dmask = None if mask is None else _device(mask, 11 if wide else 0)
    kw = dict(alpha=epi.get("alpha", 1.0), relu=bool(epi.get("relu")), accumulate=acc is not None)
    sa = sl.slice_rows(_device(a, 13 if wide else 0), extended=kind == sm.I8X)
    sb = sl.slice_rows(_device(b, 3 if wide else 0), extended=kind == sm.I8X)
    sl.gemm(sa, sb, out=out, bias=None if bias is None else torch.from_numpy(bias).cuda(), mask=dmask, **kw)
    ref = sm.gemm(a, b, kind, alpha=kw["alpha"], bias=bias, relu=kw["relu"], mask=mask, acc=acc)
    full = out_full.cpu()
    margins = bool((full[:, :pad] == -7.25).all() and (full[:, pad + N:] == -7.25).all())
    return full[:, pad:pad + N], torch.from_numpy(ref), margins


def _assert_exact(got, ref, what):
    if torch.equal(got, ref):
        return
    bad = (got != ref).nonzero()
    r, c = bad[0].tolist()
    raise AssertionError("%s: %d of %d entries differ, first [%d, %d]: kernel %r, model %r" % (
        what, len(bad), got.numel(), r, c, got[r, c].item(), ref[r, c].item()))


@pytest.mark.parametrize("kind", [sm.I8, sm.I8X], ids=KIND_IDS.get)
@pytest.mark.parametrize("M", [1, 127, 128, 129, 300])
@pytest.mark.parametrize("N", [1, 63, 64, 65, 200])
def test_products_are_bit_identical_to_the_model(kind, M, N):
    """Every K of {1, 63, 64, 65, 1000}; the epilogue options rotate over the grid so that each runs at many shapes."""
    for iK, K in enumerate([1, 63, 64, 65, 1000]):
        epi = EPILOGUES[(M + 3 * N + iK) % len(EPILOGUES)]
        a, b = _operands(M, N, K, seed=M * 1000 + N * 10 + iK)
        got, ref, margins = _run_product(kind, a, b, epi, seed=K)
        what = "%s %dx%dx%d %s" % (KIND_IDS[kind], M, N, K, epi)
        _assert_exact(got, ref, what)
        assert margins, what + ": wrote outside the output columns"


@pytest.mark.parametrize("kind,M,N,K", [(sm.I8, 130, 65, 16384), (sm.I8X, 129, 65, 16385), (sm.I8X, 5, 3, 65535)],
                         ids=["I8-16384", "I8X-16385", "I8X-65535"])
def test_long_reductions_are_bit_identical(kind, M, N, K):
    a, b = _operands(M, N, K, seed=K)
    got, ref, _ = _run_product(kind, a, b, dict(bias=True, accumulate=True, alpha=0.6), seed=1)
    _assert_exact(got, ref, "%s K=%d" % (KIND_IDS[kind], K))


def test_i8x_int32_edge():
    """The alternating operand x (digits 64, -64, 64, ...) against its negation: diagonal 7 reaches 2^31 - 32768 at
    K = 65535, which the int32 accumulators hold (bit-identical to the model), and 2^31 at K = 65536, which they
    cannot: that reduction length is refused."""
    from pnode_b200.errors import Error
    sl = _sl()
    x = sm.alternating_operand(65535)
    got, ref, _ = _run_product(sm.I8X, -x, x, {}, seed=0)
    _assert_exact(got, ref, "I8X K=65535 alternating")
    x = sm.alternating_operand(65536)
    sa = sl.slice_rows(_device(-x, 0), extended=True)
    sb = sl.slice_rows(_device(x, 0), extended=True)
    with pytest.raises(Error, match="exceeds 65535 for PNODE_SLICED_I8X"):
        sl.gemm(sa, sb)
    torch.cuda.synchronize()


# ---- TF32 products: per-entry bound --------------------------------------------------------------------------------
def _tf32_bound(K):
    """|c - a b^T| <= tol * sum_k |a_k b_k| per entry, with
      slices      3xTF32 drops lo.lo (<= 2^-22 |ab|: |lo| <= 2^-11 |x|) and the tensor core reads lo as TF32, i.e. with
                  up to 2^-10 of it lost in hi.lo and lo.hi (<= 2^-21 |ab| each, times 1 + 2^-11 for |hi| <= |x| (1 + 2^-11))
      accumulate  3K fp32 additions into the tensor-memory accumulator, each losing at most 2^-23 (rounding or
                  truncation) of a partial sum bounded by sum |ab| (first order)
      store       the final fp32 value: 2^-24"""
    return (2.0 ** -22 + 2 * 2.0 ** -21) * (1 + 2.0 ** -10) + 3 * K * 2.0 ** -23 + 2.0 ** -24


@pytest.mark.parametrize("M,N,K", [(1, 1, 1), (127, 65, 63), (129, 64, 64), (300, 200, 65), (128, 63, 200),
                                   (37, 5, 1000)])
@pytest.mark.parametrize("sign", ["mixed", "positive"])
def test_tf32_products_per_entry(M, N, K, sign):
    """positive: entries hi + lo with lo 0.3 ... 0.49 units of hi's last TF32 bit, all of one sign: losing the lo slices
    moves every entry by about 5e-4 of sum |ab|, above the bound at every K here (7x above it for K <= 200)."""
    sl = _sl()
    g = np.random.default_rng(M + N + K)
    if sign == "positive":
        def pos(r):
            j = g.integers(-8, 9, (r, 1)).astype(np.float64)
            hi = (1024 + g.integers(0, 1024, (r, K))) / 1024.0 * 2.0 ** j  # TF32 values in [2^j, 2^(j+1))
            return (hi + g.uniform(0.3, 0.49, (r, K)) * 2.0 ** (j - 10)).astype(np.float32)
        a, b = pos(M), pos(N)
    else:
        a = (g.standard_normal((M, K)) * 2.0 ** g.integers(-20, 21, (M, 1))).astype(np.float32)
        b = (g.standard_normal((N, K)) * 2.0 ** g.integers(-20, 21, (N, 1))).astype(np.float32)
        if M > 2:
            a[M // 2] = 0.0
    c = sl.gemm(sl.slice_rows(_device(a, 0)), sl.slice_rows(_device(b, 7))).cpu().double().numpy()
    a64, b64 = a.astype(np.float64), b.astype(np.float64)
    ref = a64 @ b64.T
    absum = np.abs(a64) @ np.abs(b64).T
    tol = _tf32_bound(K)
    err = np.abs(c - ref)
    ok = err <= tol * absum
    assert ok.all(), "%d entries above %.3g: worst %.3g of sum |ab|" % ((~ok).sum(), tol, (err / np.maximum(absum, 1e-300)).max())


# ---- dense MLP (pnode_dmlp_*): the chained products against the model ----------------------------------------------
@pytest.mark.parametrize("batch", [300, 16385])
def test_dense_mlp_matches_the_model_chain(batch):
    """fp64 KS right-hand side (n = 64, hidden = 200, 5 layers, out_scale -1): the forward output and J^T w are the model's
    products chained layer by layer, bit for bit (rows sliced by rows, W by rows for the forward and by columns for the
    VJP, the post-ReLU activation as the mask, out_scale as alpha).  batch 300 leaves ragged 32-row tiles and needs
    more than 256 rows per column; 16385 switches the layout to the 8-digit kind.  mu: every output unit's weight row
    is bit-identical to the model, and each unit's weight row and bias entry is held on its own to fp64 autograd:
    within 1e-12 of its own |terms| (the norm of that row of |G|^T |X|, and sum_b |G_bj|).  Not of its own norm: the
    46-bit products are exact to their operands' row maxima, so a row whose terms cancel over the batch moves further
    (at batch 300 up to 5e-12 of its norm, 8e-13 of its |terms|)."""
    from _workloads import KSExplicit
    from pnode_b200.densemlp import DenseMlpCallbacks, recognise_relu_mlp

    n, hidden = 64, 200
    func = KSExplicit(n, hidden=hidden, dtype=torch.float64, seed=3)
    with torch.no_grad():  # some dead and some strongly active hidden units, biases of both signs
        for i, m in enumerate(func.F[::2]):
            m.bias.copy_(torch.randn(m.bias.shape, generator=torch.Generator().manual_seed(i)) * 0.02)
    func = func.cuda()
    meta = torch.empty(batch, n, dtype=torch.float64, device="cuda")
    lins, out_scale = recognise_relu_mlp(func, meta)
    cb = DenseMlpCallbacks(func, meta.shape, lins, out_scale)
    kind = sm.I8X if batch > 16384 else sm.I8
    g = torch.Generator().manual_seed(batch)
    u = 0.5 * torch.randn(batch, n, generator=g, dtype=torch.float64)
    u[1] = 0.0
    w = torch.randn(batch, n, generator=g, dtype=torch.float64)
    w[:, 7] = 0.0
    coef = 0.37

    ud = u.cuda().reshape(-1)
    cb.begin(True, keep=True)
    out = cb.f(0.0, ud, keep=True)
    mu = torch.zeros(cb.nparams, dtype=torch.float64, device="cuda")
    vu, _ = cb.vjp_accumulate(0.0, ud, w.cuda().reshape(-1), mu, coef)
    out, vu, mu = out.view(batch, n).cpu(), vu.view(batch, n).cpu(), mu.cpu()
    assert cb.reused_activations == 1

    Ws = [lin.weight.detach().cpu().numpy() for lin in lins]
    bs = [lin.bias.detach().cpu().numpy() for lin in lins]
    L = len(lins)
    X = [u.numpy()]
    for l in range(L):
        last = l == L - 1
        X.append(sm.gemm(X[l], Ws[l], kind, alpha=out_scale if last else 1.0, bias=bs[l], relu=not last))
    _assert_exact(out, torch.from_numpy(X[L]), "forward batch %d" % batch)
    G, gscale, dW = w.numpy(), out_scale, [None] * L
    for l in range(L - 1, -1, -1):
        dW[l] = sm.gemm(np.ascontiguousarray(G.T), np.ascontiguousarray(X[l].T), kind, alpha=coef * gscale, acc=0.0)
        G = sm.gemm(G, np.ascontiguousarray(Ws[l].T), kind, alpha=gscale, mask=X[l] if l > 0 else None)
        gscale = 1.0
    _assert_exact(vu, torch.from_numpy(G), "J^T w batch %d" % batch)

    # fp64 autograd, with the pre-activation gradients kept for the bars of the bias entries
    x = u.clone().requires_grad_(True)
    Wt = [torch.from_numpy(W).clone().requires_grad_(True) for W in Ws]
    bt = [torch.from_numpy(b).clone().requires_grad_(True) for b in bs]
    h, zs, hs = x, [], []
    for l in range(L):
        hs.append(h)
        z = torch.nn.functional.linear(h, Wt[l], bt[l])
        z.retain_grad()
        zs.append(z)
        h = torch.relu(z) if l < L - 1 else z
    (out_scale * h).backward(w)
    assert (x.grad - torch.from_numpy(G)).abs().max() <= 1e-12 * x.grad.abs().max()
    bad = []
    for l in range(L):
        wo, bo = cb._desc.mu_w_off[l], cb._desc.mu_b_off[l]
        rows_out, cols_in = Ws[l].shape
        mw = mu[wo:wo + rows_out * cols_in].view(rows_out, cols_in)
        mb = mu[bo:bo + rows_out]
        _assert_exact(mw, torch.from_numpy(dW[l]), "mu W%d batch %d" % (l, batch))
        rw, rb = coef * Wt[l].grad, coef * bt[l].grad
        gabs = coef * zs[l].grad.abs().sum(0)
        wabs = coef * (zs[l].grad.abs().T @ hs[l].detach().abs())
        for j in range(rows_out):
            den = float(wabs[j].norm())
            e = float((mw[j] - rw[j]).norm())
            if not e <= 1e-12 * den:
                bad.append("layer %d unit %d weight row: %.3g, |terms| %.3g" % (l, j, e, den))
            if not abs(float(mb[j] - rb[j])) <= 1e-12 * float(gabs[j]):
                bad.append("layer %d unit %d bias: %.3g, sum |terms| %.3g" % (l, j, float(mb[j] - rb[j]), float(gabs[j])))
    assert not bad, "; ".join(bad[:20])
