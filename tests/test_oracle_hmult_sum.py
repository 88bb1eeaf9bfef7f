"""CPU tests of the lazily relinearised sum of products' oracle definition (tests/orc_hmult_sum.py, the reference for
hml_hmult_sum).  With real keys (test_oracle_semantics.Scheme) the sum decrypts to sum_i m_ai * m_bi / q_{L-1}; with one term it
is orc_hmult bit for bit; for n >= 2 it is not the sum of the products' hmults, which is why it has a definition of its own."""
import numpy as np
import pytest

from orc_hmult_sum import hmult_sum
from test_oracle_semantics import CASES, Scheme, negacyclic_mul


def setup(N, ML, L, A, KQ, seed, n, squares=False, key_secret=None):
    sc = Scheme(N, ML, A, seed=seed)
    s_from = negacyclic_mul(sc.s, sc.s, N) if key_secret is None else key_secret(sc)
    evk = sc.switch_key(s_from, KQ)
    scale = 1 << 30
    ma = [[scale * sc.rnd.randint(-8, 8) for _ in range(N)] for _ in range(n)]
    mb = ma if squares else [[scale * sc.rnd.randint(-8, 8) for _ in range(N)] for _ in range(n)]
    cts_a = [sc.encrypt(m, L) for m in ma]
    cts_b = cts_a if squares else [sc.encrypt(m, L) for m in mb]
    want = [0] * N
    for a, b in zip(ma, mb):
        want = [x + y for x, y in zip(want, negacyclic_mul(a, b, N))]
    return sc, evk, cts_a, cts_b, [v / sc.o.moduli[L - 1] for v in want]


def max_err(got, want):
    return max(abs(g - w) for g, w in zip(got, want))


@pytest.mark.parametrize("N,ML,L,A,KQ", CASES)
@pytest.mark.parametrize("n,squares", [(2, False), (4, False), (3, True)])
def test_sum_decrypts_to_the_rescaled_sum_of_products(N, ML, L, A, KQ, n, squares):
    """decrypt(op) ~ sum_i m_ai * m_bi / q_{L-1}.  Noise: n times the bound of test_hmult_decrypts_to_the_rescaled_product (each
    term brings its fresh-noise cross products; one key switch and one rescale rounding for the whole sum)."""
    sc, evk, cts_a, cts_b, want = setup(N, ML, L, A, KQ, 5000 + N + 7 * L + A + n, n, squares)
    got = sc.decrypt(hmult_sum(sc.o, L, cts_a, cts_b, evk, KQ), L - 1)
    assert max(abs(v) for v in want) > 2 ** 22
    assert max_err(got, want) < n * 64 * N


@pytest.mark.parametrize("N,ML,L,A,KQ", [(64, 4, 4, 2, 4), (64, 5, 3, 2, 5), (128, 6, 6, 3, 6), (64, 3, 2, 3, 2)])
def test_one_term_is_hmult(N, ML, L, A, KQ):
    sc, evk, cts_a, cts_b, _ = setup(N, ML, L, A, KQ, 51 + N + L, 1)
    assert np.array_equal(hmult_sum(sc.o, L, cts_a, cts_b, evk, KQ), sc.o.hmult(L, cts_a[0], cts_b[0], evk, KQ))
    assert np.array_equal(hmult_sum(sc.o, L, cts_a, cts_a, evk, KQ), sc.o.hmult(L, cts_a[0], cts_a[0], evk, KQ))


@pytest.mark.parametrize("N,ML,L,A,KQ", [(64, 4, 4, 2, 4), (128, 6, 6, 3, 6)])
def test_sum_is_not_the_sum_of_hmults(N, ML, L, A, KQ):
    sc, evk, cts_a, cts_b, want = setup(N, ML, L, A, KQ, 53 + N, 4)
    for n in (2, 4):
        got = hmult_sum(sc.o, L, cts_a[:n], cts_b[:n], evk, KQ)
        ref = sc.o.hmult(L, cts_a[0], cts_b[0], evk, KQ)
        for a, b in zip(cts_a[1:n], cts_b[1:n]):
            ref = sc.o.hadd(L - 1, ref, sc.o.hmult(L, a, b, evk, KQ))
        assert not np.array_equal(got, ref)
        # ... yet both decrypt to the same message (within the noise): equally valid results
        x, y = sc.decrypt(got, L - 1), sc.decrypt(ref, L - 1)
        assert max(abs(u - v) for u, v in zip(x, y)) < 2 * n * 64 * N


def test_negative_control_key_for_another_secret_does_not_decrypt():
    """the bound above is meaningful: relinearising with a key that moves s'^2 instead of s^2 leaves an error of the size of Q"""
    N, ML, L, A, KQ = 64, 4, 4, 2, 4

    def other_square(sc):
        s2 = [sc.rnd.choice((-1, 0, 1)) for _ in range(N)]
        return negacyclic_mul(s2, s2, N)

    sc, evk, cts_a, cts_b, want = setup(N, ML, L, A, KQ, 57, 2, key_secret=other_square)
    got = sc.decrypt(hmult_sum(sc.o, L, cts_a, cts_b, evk, KQ), L - 1)
    assert max_err(got, want) > 2 ** 60
