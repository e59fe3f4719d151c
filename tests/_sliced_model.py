"""Host model of the sliced operands and tensor-core products of csrc/umma_gemm.cu (numpy, no GPU).

The int8 kinds make every product deterministic integer arithmetic, so this model reproduces the kernels bit for bit.
It follows the kernels' steps, not a reformulation of them:

  row exponent   e = exponent_above(row max): the smallest e with amax < 2^e, clamped to [-960, 960]; an all-zero row
                 publishes 0
  digits         v = x * 2^(6 - e);  S times: q = rint(v), v = (v - q) * 2^B.  I8 (dense base 256): a digit above 127 is
                 lowered by 256 with a carry into the next more significant digit, from the least significant one up
  column slicing the same digits of x^T (column exponents)
  TF32 pair      hi = tf32_round(x) (round to nearest even on the float32 bit pattern, 13 bits dropped), lo = x - hi
  diagonals      D_d = sum_{i+j=d} Q^A_i (Q^B_j)^T, exact: float64 products of integer matrices whose partial sums stay
                 below 2^53 (horner_sums forms the epilogue's sums of them with fewer products)
  epilogue       hi = Horner_{d<NH}(D_d) and lo = Horner_{d>=NH}(D_d) in int64, x = hi 2^-(12+B(NH-1)) + lo 2^-(12+B(S-1)),
                 then * 2^ea, * 2^eb, + bias, * alpha, ReLU, mask > 0, + accumulate (in this order, one fp64 rounding each)
"""
import numpy as np

I8, TF32, I8X = 0, 1, 2
LEAD_BITS = 6
EXP_CLAMP = 960
INT32_MAX = 2 ** 31 - 1


class Kind:
    def __init__(self, slices, base_bits, dense, nh, lead_max, digit_max):
        self.S, self.B, self.dense, self.NH = slices, base_bits, dense, nh
        self.lead_max, self.digit_max = lead_max, digit_max  # largest |digit| of slice 0 / of the other slices


# I8: 6 balanced base-256 digits (the carry can raise the leading digit to 65); I8X: 8 base-128 digits in [-64, 64]
KINDS = {I8: Kind(6, 8, True, 3, 65, 128), I8X: Kind(8, 7, False, 4, 64, 64)}


def exponent_above(amax):
    """Smallest e with amax < 2^e, clamped to [-EXP_CLAMP, EXP_CLAMP]; 0 where amax == 0."""
    amax = np.asarray(amax, dtype=np.float64)
    _, e = np.frexp(amax)  # amax = m 2^e, 0.5 <= m < 1
    e = np.clip(e.astype(np.int64), -EXP_CLAMP, EXP_CLAMP)
    return np.where(amax > 0, e, 0)


def digits(v, kind):
    """int64 digits [S, ...] of values already scaled to |v| < 2^LEAD_BITS (the remainder after S digits is dropped)."""
    k = KINDS[kind]
    r = np.array(v, dtype=np.float64)
    q = np.empty((k.S,) + r.shape, dtype=np.int64)
    for s in range(k.S):
        d = np.rint(r)
        r = (r - d) * float(1 << k.B)
        q[s] = d.astype(np.int64)
    if k.dense:
        for s in range(k.S - 1, 0, -1):
            up = q[s] > 127
            q[s] -= 256 * up
            q[s - 1] += up
    return q


def slice_rows(x, kind):
    """(digits int8 [S, rows, k], exponents int64 [rows]) of the operand x (reduction over the columns of x)."""
    x = np.asarray(x, dtype=np.float64)
    e = exponent_above(np.abs(x).max(axis=1))
    q = digits(x * np.ldexp(1.0, LEAD_BITS - e)[:, None], kind)
    return q.astype(np.int8), e


def slice_cols(x, kind):
    """Digits and exponents of the operand x^T (operand row c = column c of x)."""
    return slice_rows(np.asarray(x, dtype=np.float64).T, kind)


def reconstruct(q, e, kind):
    """x = 2^e sum_s q_s 2^-(LEAD + B s), exact in fp64 for the digits of a finite fp64 source."""
    k = KINDS[kind]
    x = np.zeros(q.shape[1:], dtype=np.float64)
    for s in range(k.S):
        x += q[s].astype(np.float64) * 2.0 ** -(LEAD_BITS + k.B * s)
    return x * np.ldexp(1.0, e)[:, None]


def tf32_split(x):
    """(hi, lo) float32 with hi = tf32_round(x), lo = x - hi: the TF32 slices."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    u = x.view(np.uint32)
    special = (u & np.uint32(0x7F800000)) == np.uint32(0x7F800000)
    r = (u + np.uint32(0xFFF) + ((u >> np.uint32(13)) & np.uint32(1))) & np.uint32(0xFFFFE000)
    hi = np.where(special, x, r.view(np.float32))
    return hi, (x - hi).astype(np.float32)


def diagonals(qa, qb):
    """D [S, M, N] int64 with D_d = sum_{i+j=d} qa_i qb_j^T (exact), and max |D_d| per diagonal."""
    S = qa.shape[0]
    assert qb.shape[0] == S and qa.shape[2] == qb.shape[2]
    D = np.empty((S, qa.shape[1], qb.shape[1]), dtype=np.int64)
    for d in range(S):
        # one product over the concatenated pairs (i, d - i): integers below 2^53 at every step, so exact in any order
        A = np.concatenate([qa[i] for i in range(d + 1)], axis=1).astype(np.float64)
        B = np.concatenate([qb[d - i] for i in range(d + 1)], axis=1).astype(np.float64)
        P = A @ B.T
        assert np.abs(P).max(initial=0.0) < 2.0 ** 53
        D[d] = P.astype(np.int64)
    return D, np.abs(D).reshape(S, -1).max(axis=1, initial=0)


def horner(D, kind):
    """The epilogue's int64 Horner sums (hi over the first NH diagonals, lo over the rest) of the diagonal sums D."""
    k = KINDS[kind]
    radix = np.int64(1 << k.B)
    hi = np.zeros(D.shape[1:], dtype=np.int64)
    lo = np.zeros(D.shape[1:], dtype=np.int64)
    for d in range(k.NH):
        hi = hi * radix + D[d]
    for d in range(k.NH, k.S):
        lo = lo * radix + D[d]
    return hi, lo


def horner_sums(qa, qb, kind):
    """horner(diagonals(qa, qb)) with S + NH float64 products instead of S (S + 1) / 2: for each i, qa_i times the digits
    qb_j of the same Horner sum combined with their weights 2^(B (top - i - j)).  Exact: the combined digits are
    integers below 2^28 and every partial sum stays below 2^53 for K <= 65536."""
    k = KINDS[kind]
    a = qa.astype(np.float64)
    b = qb.astype(np.float64)

    def part(dlo, dhi, top):  # sum over dlo <= i + j < dhi of qa_i qb_j^T 2^(B (top - i - j))
        acc = np.zeros((qa.shape[1], qb.shape[1]), dtype=np.int64)
        for i in range(min(dhi, k.S)):
            js = [j for j in range(k.S) if dlo <= i + j < dhi]
            if js:
                comb = sum(b[j] * float(1 << (k.B * (top - i - j))) for j in js)
                P = a[i] @ comb.T
                assert np.abs(P).max(initial=0.0) < 2.0 ** 53
                acc += P.astype(np.int64)
        return acc

    return part(0, k.NH, k.NH - 1), part(k.NH, k.S, k.S - 1)


def epilogue(hi, lo, ea, eb, kind, alpha=1.0, bias=None, relu=False, mask=None, acc=None):
    """The fp64 result of umma_gemm_kernel from the Horner sums (hi, lo) of the diagonals."""
    k = KINDS[kind]
    x = hi.astype(np.float64) * 2.0 ** -(2 * LEAD_BITS + k.B * (k.NH - 1))
    if k.S > k.NH:
        x = x + lo.astype(np.float64) * 2.0 ** -(2 * LEAD_BITS + k.B * (k.S - 1))  # exact product: fma == mul + add
    x = x * np.ldexp(1.0, np.asarray(ea))[:, None]
    x = x * np.ldexp(1.0, np.asarray(eb))[None, :]
    if bias is not None:
        x = x + np.asarray(bias, dtype=np.float64)[None, :]
    x = x * float(alpha)
    if relu:
        x = np.where(x > 0.0, x, 0.0)
    if mask is not None:
        x = np.where(np.asarray(mask, dtype=np.float64) > 0.0, x, 0.0)
    return x + (0.0 if acc is None else np.asarray(acc, dtype=np.float64))


def wrap_int32(D):
    """What a wrapping int32 accumulator holds for the exact diagonal sums D."""
    return ((D + 2 ** 31) % 2 ** 32) - 2 ** 31


def gemm(a, b, kind, **epi):
    """Model of pnode_sliced_gemm(slice_rows(a), slice_rows(b)) with its epilogue options (C = a b^T)."""
    qa, ea = slice_rows(a, kind)
    qb, eb = slice_rows(b, kind)
    assert max(diagonal_bound(kind, a.shape[1])) <= INT32_MAX  # every diagonal fits the int32 accumulators
    hi, lo = horner_sums(qa, qb, kind)
    return epilogue(hi, lo, ea, eb, kind, **epi)


def truncation_bound(kind):
    """tau with |model product - exact product| <= tau 2^(ea_i + eb_j) K per entry, before the epilogue's fp64 rounding.

    Each entry is a = 2^e (sum_{s<S} q_s 2^-(6+Bs) + r) with |r| <= 2^-(7+B(S-1)) (half a unit of the last digit) and
    |a| < 2^e.  The product keeps the slice pairs i + j < S:
      dropped pairs   sum_{d=S}^{2S-2} (2S-1-d) max|q_i q_j| 2^-(12+Bd)
      remainders      2 |r| (1 + |r|) + |r|^2  (a_hat r_b + r_a b_hat + r_a r_b, |a_hat| < 1 + |r|)"""
    k = KINDS[kind]
    r = 2.0 ** -(7 + k.B * (k.S - 1))
    dropped = sum((2 * k.S - 1 - d) * float(k.digit_max) ** 2 * 2.0 ** -(12 + k.B * d) for d in range(k.S, 2 * k.S - 1))
    return dropped + 2 * r * (1 + r) + r * r


def diagonal_bound(kind, K):
    """Largest |D_d| the digit ranges allow at reduction length K, per diagonal."""
    k = KINDS[kind]
    out = []
    for d in range(k.S):
        per = 0
        for i in range(d + 1):
            qi = k.lead_max if i == 0 else k.digit_max
            qj = k.lead_max if d - i == 0 else k.digit_max
            per += qi * qj
        out.append(per * K)
    return out


def alternating_operand(K):
    """x = sum_{s<8} (-1)^s 2^(-7s) in every entry: row exponent 0 and I8X digits 64, -64, 64, ...  The product of
    -x and x reaches 8 * 4096 * K on diagonal 7, which is 2^31 (one past INT32_MAX) at K = 65536."""
    x = sum((-1) ** s * 2.0 ** (-7 * s) for s in range(8))
    return np.full((1, K), x, dtype=np.float64)
