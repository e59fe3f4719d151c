"""The host model of the sliced products (tests/_sliced_model.py) against exact arithmetic, on the CPU.

tests/test_gpu_sliced_exact.py holds the kernels of csrc/umma_gemm.cu to this model bit for bit, so the model itself has
to be right: its digits reconstruct every entry to half a unit of the last digit, its products stay within the truncation
bound of the slicing (include/pnode_b200.h, DESIGN.md 4a) against exact rational products, and its diagonal sums show
which reduction lengths fit the int32 accumulators of the tensor cores."""
from fractions import Fraction

import numpy as np
import pytest

import _sliced_model as sm

KIND_IDS = {sm.I8: "I8", sm.I8X: "I8X"}


def _case_slices_rows():
    """Rows of the slice test of tests/test_gpu_umma.py (randn scaled 1e-6 ... 1e3, one zero row) plus rows at and
    below the exponent clamp, subnormal entries, powers of two and rows with entries 2^-60 below their maximum.  Row
    maxima of 2^960 and above are outside the range of the slicing (the leading digit would leave its byte)."""
    rng = np.random.default_rng(1)
    x = rng.standard_normal((50, 333)) * np.logspace(-6, 3, 50)[:, None]
    x[7] = 0.0
    extra = rng.standard_normal((10, 333))
    extra[0] = rng.uniform(-0.999, 0.999, 333) * 2.0 ** 960  # the largest row maxima the slicing takes: e = 960
    extra[1] = rng.uniform(-0.999, 0.999, 333) * 2.0 ** -961  # below the clamp: e = -960, fewer bits of the row kept
    extra[2] *= 2.0 ** -955
    extra[3] *= 2.0 ** -1000
    extra[4] = 2.0 ** -1074 * rng.integers(-1000, 1000, 333)  # subnormal entries only
    extra[5] = 2.0 ** rng.integers(-30, 30, 333).astype(np.float64)
    extra[6] = rng.standard_normal(333) * 2.0 ** -rng.integers(0, 60, 333).astype(np.float64)
    extra[7] = 63.999999999999 * np.sign(rng.standard_normal(333))  # just below a power of two
    extra[8] = 64.0                                                  # exactly a power of two
    extra[9, :] = 0.0
    extra[9, 5] = -1.5
    return np.concatenate([x, extra])


@pytest.mark.parametrize("kind", [sm.I8, sm.I8X], ids=KIND_IDS.get)
def test_digits_reconstruct_to_half_a_unit_of_the_last_digit(kind):
    k = sm.KINDS[kind]
    x = _case_slices_rows()
    q, e = sm.slice_rows(x, kind)
    amax = np.abs(x).max(1)
    nz = amax > 0
    assert (e[~nz] == 0).all()
    assert (amax[nz] < np.ldexp(1.0, e[nz])).all()
    clamped = (e == sm.EXP_CLAMP) | (e == -sm.EXP_CLAMP)
    assert (amax[nz & ~clamped] >= np.ldexp(0.5, e[nz & ~clamped])).all()  # the smallest such e
    assert int(np.abs(q[0]).max()) <= k.lead_max and int(np.abs(q[1:].astype(np.int64)).max()) <= k.digit_max
    last = 2.0 ** -(sm.LEAD_BITS + k.B * (k.S - 1) + 1)  # half a unit of the last digit: 2^-47 (I8), 2^-56 (I8X)
    for r in range(x.shape[0]):  # exact: fractions, entry by entry
        scale = Fraction(2) ** int(e[r])
        for c in range(0, x.shape[1], 7):
            v = sum(Fraction(int(q[s, r, c])) / Fraction(2) ** (sm.LEAD_BITS + k.B * s) for s in range(k.S)) * scale
            assert abs(v - Fraction(x[r, c])) <= Fraction(last) * scale, (r, c)
    # the column slicing is the row slicing of the transpose
    qc, ec = sm.slice_cols(x[:, :40], kind)
    qt, et = sm.slice_rows(np.ascontiguousarray(x[:, :40].T), kind)
    assert np.array_equal(qc, qt) and np.array_equal(ec, et)


def test_tf32_pair():
    rng = np.random.default_rng(2)
    x = (rng.standard_normal(4096) * 2.0 ** rng.integers(-120, 120, 4096)).astype(np.float32)
    x[:4] = [0.0, -0.0, 1.0 + 2.0 ** -11, 1.0 + 3 * 2.0 ** -11]  # ties: to even (down, then up)
    hi, lo = sm.tf32_split(x)
    assert (hi.view(np.uint32) & 0x1FFF == 0).all()
    assert np.array_equal(hi.astype(np.float64) + lo.astype(np.float64), x.astype(np.float64))
    normal = np.abs(x) >= 2.0 ** -126
    assert (np.abs(lo[normal].astype(np.float64)) <= np.abs(hi[normal].astype(np.float64)) * 2.0 ** -11).all()
    assert hi[2] == 1.0 and hi[3] == np.float32(1.0 + 2.0 ** -9)


def _exact_product(a, b, r, c):
    return sum((Fraction(x) * Fraction(y) for x, y in zip(a[r], b[c])), Fraction(0))


@pytest.mark.parametrize("kind", [sm.I8, sm.I8X], ids=KIND_IDS.get)
def test_model_product_within_the_truncation_bound(kind):
    """Per entry: |C - A B^T| <= tau 2^(ea_i + eb_j) K + 2^-53 sum_k |a_ik b_jk| (the truncation of the slicing and the
    one fp64 rounding of the epilogue) against exact rational products."""
    rng = np.random.default_rng(3 + kind)
    M, N, K = 9, 7, 45
    a = rng.standard_normal((M, K)) * 2.0 ** rng.integers(-40, 40, (M, 1)).astype(np.float64)
    b = rng.standard_normal((N, K)) * 2.0 ** rng.integers(-40, 40, (N, 1)).astype(np.float64)
    a[2] *= 2.0 ** -rng.integers(0, 50, K).astype(np.float64)  # entries spread over many binades within one row
    a[4] = 0.0
    b[1] = 0.0
    a[5] = b[6] * 2.0 ** 7  # cancellation: a_5 . (-b_6) terms
    b[6, K // 2:] *= -1.0
    C = sm.gemm(a, b, kind)
    qa, ea = sm.slice_rows(a, kind)
    qb, eb = sm.slice_rows(b, kind)
    D, dmax = sm.diagonals(qa, qb)
    hi, lo = sm.horner(D, kind)
    assert np.array_equal(C, sm.epilogue(hi, lo, ea, eb, kind))  # the two ways of forming the Horner sums agree
    tau = sm.truncation_bound(kind)
    assert tau < (3e-13 if kind == sm.I8 else 1e-15)
    assert (dmax <= sm.INT32_MAX).all()
    for r in range(M):
        for c in range(N):
            err = abs(Fraction(C[r, c]) - _exact_product(a, b, r, c))
            absum = sum(abs(Fraction(x) * Fraction(y)) for x, y in zip(a[r], b[c]))
            bound = Fraction(tau) * Fraction(2) ** int(ea[r] + eb[c]) * K + Fraction(2.0 ** -53) * absum
            assert err <= bound, (r, c, float(err), float(bound))


def test_epilogue_order():
    """bias before alpha, then ReLU, mask > 0 and the accumulated value, each in fp64."""
    D = np.zeros((6, 2, 3), dtype=np.int64)
    D[0] = [[4096, -4096, 2048], [0, 1, -1]]  # 1, -1, 0.5 at exponents 0
    C = sm.epilogue(*sm.horner(D, sm.I8), np.array([0, 3]), np.array([0, 0, -2]), sm.I8, alpha=-2.0, bias=np.array([0.25, 0.0, 1.0]),
                    relu=True, mask=np.array([[1.0, 1.0, 0.0], [1.0, -1.0, 1.0]]), acc=np.full((2, 3), 10.0))
    # row 0: (1 + .25) * -2 -> relu 0;  (-1 + 0) * -2 = 2;  masked;  row 1: 0;  masked;  (-2^-12 * 2^3 / 4 + 1) * -2 -> 0
    assert np.array_equal(C, [[10.0, 12.0, 10.0], [10.0, 10.0, 10.0]])


INT32_TABLE = [  # (kind, K, what): the largest diagonal sum the digit ranges allow, and the concrete alternating product
    (sm.I8, 16384, "bound"), (sm.I8X, 65535, "bound"), (sm.I8X, 65535, "alternating"), (sm.I8X, 65536, "alternating")]


@pytest.mark.parametrize("kind,K,what", INT32_TABLE,
                         ids=["%s-K%d-%s" % (KIND_IDS[k], K, w) for k, K, w in INT32_TABLE])
def test_int32_table(kind, K, what):
    """int32 accumulators (no saturation) hold every diagonal of I8 up to K = 16384 and of I8X up to K = 65535; the
    alternating I8X operand reaches 2^31 on diagonal 7 at K = 65536, which wraps."""
    if what == "bound":
        worst = sm.diagonal_bound(kind, K)
        print("%s K=%d worst |D_d| per diagonal: %s" % (KIND_IDS[kind], K, worst))
        assert max(worst) <= sm.INT32_MAX
        assert max(sm.diagonal_bound(kind, K + 1 if kind == sm.I8X else 2 * K)) > sm.INT32_MAX  # the caps are tight
        return
    x = sm.alternating_operand(K)
    qa, ea = sm.slice_rows(-x, kind)
    qb, eb = sm.slice_rows(x, kind)
    assert ea[0] == 0 and eb[0] == 0
    assert qb[:, 0, 0].tolist() == [64 * (-1) ** s for s in range(8)]
    D, dmax = sm.diagonals(qa, qb)
    print("I8X K=%d alternating operand: |D_d| = %s" % (K, dmax.tolist()))
    assert int(D[7, 0, 0]) == 8 * 4096 * K
    if K == 65535:
        assert int(dmax.max()) == 2 ** 31 - 32768 <= sm.INT32_MAX
    else:
        assert int(D[7, 0, 0]) == 2 ** 31 > sm.INT32_MAX
        # a wrapping accumulator turns +2^31 into -2^31: the product moves by 2^32 units of diagonal 7
        good = sm.epilogue(*sm.horner(D, kind), ea, eb, kind)[0, 0]
        bad = sm.epilogue(*sm.horner(sm.wrap_int32(D), kind), ea, eb, kind)[0, 0]
        assert bad - good == pytest.approx(-2.0 ** 32 * 2.0 ** -(12 + 7 * 7), rel=1e-3)
        exact = -Fraction(x[0, 0]) ** 2 * K
        print("exact %.17g, correct accumulators %.17g, wrapped %.17g (rel. error %.2e)"
              % (exact, good, bad, abs(bad - exact) / abs(exact)))
        assert abs(Fraction(good) - exact) <= Fraction(1e-15) * abs(exact) < abs(Fraction(bad) - exact)
