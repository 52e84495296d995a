"""The arithmetic of the panel query's int8 update (limbo_b200/csrc/query_i8.cu), restated in numpy: L is scaled per row and V by
the fixed 2^e_V >= sigma_f, both are split into 7 signed base-2^7 digit planes with round-to-nearest, the 28 digit pairs with
i + j < 7 are summed per digit-sum group in exact integer arithmetic and recombined in fp64.  Checked here: the digits stay in
[-64, 64], the group sums stay inside the int32 bound the kernel relies on (7 * 64^2 * K), the digits reconstruct their operand,
and the blocked solve with the truncated products gives sigma^2 within 1e-12 of the plain fp64 solve."""
import numpy as np
import pytest

S = 7


def _digits(A, e):
    """S planes of round-to-nearest base-2^7 digits of A * 2^(6 - e) (e broadcast against A)."""
    x = A * np.exp2(6.0 - e)
    out = []
    for _ in range(S):
        d = np.rint(x)
        out.append(d)
        x = (x - d) * 128.0
    return out


def _row_exp(L):
    m = np.abs(L).max(axis=1, keepdims=True)
    e = np.where(m > 0, np.frexp(np.where(m > 0, m, 1.0))[1], -1000)
    return e.astype(float)


def _oz_update(L, V, ev):
    """L V from the digit products, with the group sums returned for the bound checks."""
    er = _row_exp(L)
    a, b = _digits(L, er), _digits(V, ev)
    acc = []
    out = np.zeros((L.shape[0], V.shape[1]))
    for g in range(S - 1, -1, -1):
        sg = sum(a[i].astype(np.int64) @ b[g - i].astype(np.int64) for i in range(g + 1))
        acc.append(sg)
        out += sg.astype(float) * 2.0 ** (-12 - 7 * g)
    return out * np.exp2(er + ev), a, b, acc


def _problem(N, M, D=6, noise=0.01):
    from limbo_b200 import synth

    def k(A, B):
        sa, sb = (A ** 2).sum(1), (B ** 2).sum(1)
        return np.exp(-0.5 * np.maximum(sa[:, None] + sb[None, :] - 2 * A @ B.T, 0))
    X = synth.points(1234, N, D)
    Xq = synth.points(1235, M, D)
    K = k(X, X)
    K[np.diag_indices(N)] += noise + 1e-8
    L = np.linalg.cholesky(K)
    Ks = np.concatenate([k(X, Xq), k(X, X[:64])], 1)  # candidates and training points (sigma^2 ~ noise)
    return L, Ks


def _solve(L, Ks, sb, oz):
    import scipy.linalg as sl
    N = L.shape[0]
    V = np.zeros_like(Ks)
    ev = float(np.frexp(1.0)[1])  # sigma_f = 1: |V| <= 1 < 2^1
    stats = []
    for s0 in range(0, N, sb):
        T = Ks[s0:s0 + sb].copy()
        if s0:
            if oz:
                P, a, b, acc = _oz_update(L[s0:s0 + sb, :s0], V[:s0], ev)
                stats.append((a, b, acc, s0))
                T -= P
            else:
                T -= L[s0:s0 + sb, :s0] @ V[:s0]
        V[s0:s0 + sb] = sl.solve_triangular(L[s0:s0 + sb, s0:s0 + sb], T, lower=True)
    return 1.0 + 0.01 - (V ** 2).sum(0), V, stats


@pytest.mark.parametrize("N,sb", [(768, 256), (1024, 256)])
def test_digit_products_bounds_and_error(N, sb):
    L, Ks = _problem(N, 192)
    ref, Vref, _ = _solve(L, Ks, sb, False)
    s2, _, stats = _solve(L, Ks, sb, True)
    assert np.abs(Vref).max() <= 1.0 + 1e-12        # |V| <= sigma_f: the fixed scale of V holds
    for a, b, acc, K in stats:
        assert max(np.abs(d).max() for d in a + b) <= 64
        assert max(np.abs(x).max() for x in acc) <= S * 64 * 64 * K < 2 ** 31
    assert np.abs(s2 - ref).max() <= 1e-12


def test_digits_reconstruct():
    rng = np.random.default_rng(5)
    A = rng.standard_normal((64, 300)) * np.exp2(rng.integers(-20, 5, size=(64, 1)))
    e = _row_exp(A)
    d = _digits(A, e)
    rec = sum(di * 2.0 ** (-7 * i) for i, di in enumerate(d)) * np.exp2(e - 6)
    # 7 digits carry 6 + 6 * 7 + 1 = 49 bits below the row maximum
    assert np.all(np.abs(rec - A) <= np.exp2(e - 6 - 7 * (S - 1) - 1))
    assert max(np.abs(x).max() for x in d) <= 64


def test_int32_bound_covers_the_largest_supported_k():
    # the kernel's exactness bound (query_i8.cu MAX_K): K = 74898 still fits, the next K does not
    assert S * 64 * 64 * 74898 < 2 ** 31 <= S * 64 * 64 * 74899
    # N = 65536 (K <= 63488 for the last 2048-row super-block) is inside it
    assert 65536 - 2048 <= 74898
