"""CPU tests that pin the oracle against first-principles definitions (tier T1) — no GPU needed."""
import numpy as np
import pytest

from orc import Oracle, uniform_limbs


def is_prime(n):
    if n < 2:
        return False
    for p in (2, 3, 5, 7, 11, 13, 17, 19, 23, 29, 31, 37):
        if n % p == 0:
            return n == p
    d, s = n - 1, 0
    while d % 2 == 0:
        d //= 2
        s += 1
    for a in (2, 3, 5, 7, 11, 13, 17, 19, 23, 29, 31, 37):
        x = pow(a, d, n)
        if x in (1, n - 1):
            continue
        for _ in range(s - 1):
            x = x * x % n
            if x == n - 1:
                break
        else:
            return False
    return True


@pytest.mark.parametrize("N,w,ml,al", [(16, 36, 6, 2), (256, 36, 5, 3), (65536, 36, 45, 15), (32768, 36, 28, 28),
                                       (2048, 20, 12, 4), (256, 20, 70, 10), (8192, 24, 40, 10), (65536, 28, 45, 15), (65536, 32, 45, 15),
                                       (4096, 33, 16, 2), (65536, 35, 45, 15)])
def test_moduli_rule(N, w, ml, al):
    o = Oracle(N, w, ml, al)
    # independent python restatement of the rule: primes = 1 mod 2N, scanned downward from 2^w
    want, c = [], ((2**w - 2) // (2 * N)) * 2 * N + 1
    while len(want) < ml + al:
        if is_prime(c):
            want.append(c)
        c -= 2 * N
    assert o.moduli == want
    for m, psi in zip(o.moduli, o.psi):
        assert 2 ** (w - 1) < m < 2**w and m % (2 * N) == 1
        assert pow(psi, N, m) == m - 1  # primitive 2N-th root


@pytest.mark.parametrize("N,w", [(16, 36), (64, 36), (256, 36), (64, 20), (256, 28), (64, 33), (256, 35)],
                         ids=["16", "64", "256", "64-w20", "256-w28", "64-w33", "256-w35"])
def test_fast_ntt_equals_definition(N, w):
    o = Oracle(N, w, 3, 2)
    for mi in range(o.n_mod):
        a = uniform_limbs([o.moduli[mi]], N, 7 + mi)[0]
        fast = o.ntt(mi, a)
        assert np.array_equal(fast, o.ntt_direct(mi, a))
        # definition spelled out in python: ahat[k] = a(psi^(2 brv(k)+1))
        m, psi, logn = o.moduli[mi], o.psi[mi], N.bit_length() - 1
        for k in (0, 1, N // 2, N - 1):
            brv = int(format(k, "0%db" % logn)[::-1], 2)
            x = pow(psi, 2 * brv + 1, m)
            assert int(fast[k]) == sum(int(a[n]) * pow(x, n, m) for n in range(N)) % m
        assert np.array_equal(o.intt(mi, fast), a)
        assert np.array_equal(o.intt_direct(mi, fast), a)


@pytest.mark.parametrize("N", [16, 128])
def test_pointwise_product_is_negacyclic_schoolbook(N):
    o = Oracle(N, 36, 2, 1)
    for mi in range(o.n_mod):
        a = uniform_limbs([o.moduli[mi]], N, 1)[0]
        b = uniform_limbs([o.moduli[mi]], N, 2)[0]
        prod_eval = o.ewe(mi, o.ntt(mi, a), o.ntt(mi, b), None, None)
        assert np.array_equal(o.intt(mi, prod_eval), o.schoolbook(mi, a, b))


@pytest.mark.parametrize("N,g", [(16, 5), (64, 25), (256, 5), (256, 2 * 256 - 1), (64, 3)])
def test_automorphism_eval_gather_matches_coefficient_definition(N, g):
    o = Oracle(N, 36, 2, 1)
    for mi in range(o.n_mod):
        a = uniform_limbs([o.moduli[mi]], N, 3)[0]
        want = o.ntt(mi, o.automorph_coeff(mi, g, a))
        got = o.automorph_eval(g, o.ntt(mi, a))
        assert np.array_equal(got, want)
    perm = o.automorph_index(g)
    assert sorted(perm.tolist()) == list(range(N))


def test_ewe_variants():
    o = Oracle(64, 36, 2, 1)
    m = o.moduli[1]
    x = [uniform_limbs([m], 64, 10 + i)[0] for i in range(4)]
    xi = [[int(v) for v in a] for a in x]
    assert o.ewe(1, x[0], x[1], x[2], x[3]).tolist() == [(a * b + c * d) % m for a, b, c, d in zip(*xi)]
    assert o.ewe(1, x[0], x[1], x[2], x[3], sub=True).tolist() == [(a * b - c * d) % m for a, b, c, d in zip(*xi)]
    assert o.ewe(1, x[0], None, x[2], None).tolist() == [(a + c) % m for a, c in zip(xi[0], xi[2])]
    assert o.ewe(1, x[0], x[1], None, None).tolist() == [(a * b) % m for a, b in zip(xi[0], xi[1])]


def test_bconv_matches_bigint_crt_up_to_multiple_of_D():
    """fast base conversion = (x + e*D) mod m with 0 <= e < n_src (no correction term)."""
    N = 32
    o = Oracle(N, 36, 6, 3)
    src = [1, 2, 4]
    D = 1
    for i in src:
        D *= o.moduli[i]
    x = np.stack([uniform_limbs([o.moduli[i]], N, 20 + i)[0] for i in src])
    for dst in (0, 3, 6, 8):
        m = o.moduli[dst]
        got = o.bconv(src, dst, x)
        for n in range(N):
            # exact CRT lift with python big ints
            tot = 0
            for k, i in enumerate(src):
                qi = o.moduli[i]
                hat = D // qi
                tot += (int(x[k, n]) * pow(hat, -1, qi) % qi) * hat
            assert int(got[n]) == tot % m
            lift = tot % D
            assert (tot - lift) % D == 0 and 0 <= (tot - lift) // D < len(src)


def _ks_reference_python(o, L, d, evk, evk_q):
    """Independent big-int restatement of hybrid key switching on coefficient vectors (tiny N only)."""
    N, A, ML = o.N, o.alpha, o.max_level
    ext = o.ext_mod_idx(L)
    beta = -(-L // A)
    P = 1
    for j in range(A):
        P *= o.moduli[ML + j]
    acc = [[None] * len(ext) for _ in range(2)]
    dc = [o.intt(i, d[i]) for i in range(L)]
    for e, mi in enumerate(ext):
        m = o.moduli[mi]
        for c in range(2):
            tot = np.zeros(N, dtype=object)
            for j in range(beta):
                idx = list(range(j * A, min(L, (j + 1) * A)))
                if mi in idx:
                    t = dc[mi]
                else:
                    Dj = 1
                    for i in idx:
                        Dj *= o.moduli[i]
                    t = np.zeros(N, dtype=object)
                    for i in idx:
                        qi = o.moduli[i]
                        hat = Dj // qi
                        y = [int(v) * pow(hat, -1, qi) % qi for v in dc[i]]
                        t = t + np.array([yy * (hat % m) for yy in y], dtype=object)
                    t = np.array([int(v) % m for v in t], dtype=np.uint64)
                that = o.ntt(mi, np.asarray(t, dtype=np.uint64))
                el = e if e < L else evk_q + (e - L)
                k = evk[j, c, el]
                tot = tot + np.array([int(a) * int(b) for a, b in zip(that, k)], dtype=object)
            acc[c][e] = np.array([int(v) % m for v in tot], dtype=np.uint64)
    outs = []
    for c in range(2):
        u = [o.intt(ML + j, acc[c][L + j]) for j in range(A)]
        out = np.zeros((L, N), dtype=np.uint64)
        for i in range(L):
            m = o.moduli[i]
            v = np.zeros(N, dtype=object)
            for j in range(A):
                pj = o.moduli[ML + j]
                hat = P // pj
                v = v + np.array([(int(x) * pow(hat, -1, pj) % pj) * (hat % m) for x in u[j]], dtype=object)
            vhat = o.ntt(i, np.array([int(x) % m for x in v], dtype=np.uint64))
            pinv = pow(P % m, -1, m)
            out[i] = np.array([(int(a) - int(b)) * pinv % m for a, b in zip(acc[c][i], vhat)], dtype=np.uint64)
        outs.append(out)
    return outs


@pytest.mark.parametrize("ML,L,A", [(6, 6, 2), (6, 5, 2), (5, 2, 3), (4, 4, 4), (7, 7, 3), (3, 1, 2)])
def test_keyswitch_matches_bigint_restatement(ML, L, A):
    N = 16
    o = Oracle(N, 36, ML, A)
    beta = -(-L // A)
    d = uniform_limbs(o.moduli[:L], N, 30)
    for evk_q in (L, ML):
        kmods = o.moduli[:evk_q] + o.moduli[ML:]
        evk = uniform_limbs(kmods, N, 31, lead=(beta, 2))
        want = _ks_reference_python(o, L, d, evk, evk_q)
        for direct in (0, 1):
            o.set_direct(direct)
            got = o.keyswitch(L, d, evk, evk_q)
            assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


def test_rescale_and_hmult_tiers_agree():
    N, ML, A, L = 16, 5, 2, 5
    o = Oracle(N, 36, ML, A)
    beta = -(-L // A)
    a = uniform_limbs(o.moduli[:L], N, 50, lead=(2,))
    b = uniform_limbs(o.moduli[:L], N, 51, lead=(2,))
    evk = uniform_limbs(o.moduli[:L] + o.moduli[ML:], N, 52, lead=(beta, 2))
    o.set_direct(0)
    fast = o.hmult(L, a, b, evk, L)
    rot_fast = o.hrotate(L, a, evk, L, 5)
    o.set_direct(1)
    assert np.array_equal(o.hmult(L, a, b, evk, L), fast)
    assert np.array_equal(o.hrotate(L, a, evk, L, 5), rot_fast)
    o.set_direct(0)
    # rescale definition spelled out: (c_l - [c_{L-1}]_{q_l}) * q_{L-1}^-1
    x = a[0]
    r = o.intt(L - 1, x[L - 1])
    got = o.rescale(L, x)
    for l in range(L - 1):
        m = o.moduli[l]
        rl = o.ntt(l, r % np.uint64(m))
        qinv = pow(o.moduli[L - 1] % m, -1, m)
        want = [(int(c) - int(t)) * qinv % m for c, t in zip(x[l], rl)]
        assert got[l].tolist() == want


def test_threads_do_not_change_results():
    N, ML, A, L = 64, 6, 2, 6
    o = Oracle(N, 36, ML, A)
    a = uniform_limbs(o.moduli[:L], N, 60, lead=(2,))
    b = uniform_limbs(o.moduli[:L], N, 61, lead=(2,))
    evk = uniform_limbs(o.moduli[:L] + o.moduli[ML:], N, 62, lead=(3, 2))
    Oracle.set_threads(1)
    one = o.hmult(L, a, b, evk, L)
    Oracle.set_threads(4)
    many = o.hmult(L, a, b, evk, L)
    Oracle.set_threads(1)
    assert np.array_equal(one, many)
