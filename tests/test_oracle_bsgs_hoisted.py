"""CPU tests of the double-hoisted BSGS linear transform's oracle definition (tests/orc_bsgs.py, the reference for
hml_hrotate_bsgs_hoisted).  With real keys (test_oracle_semantics.Scheme) the transform decrypts to
sum_j sigma_{G_j}( sum_i p_{j,i} * sigma_{b_i}(m) ); its corner cases are the rotation sum and the hoisted rotation bit for bit;
with several baby and giant steps it is not the textbook-hoisted composition, which is why it has a definition of its own."""
import numpy as np
import pytest

from orc_bsgs import hrotate_bsgs_hoisted
from orc_rotsum import hrotate_sum_hoisted
from test_oracle_semantics import CASES, Scheme, automorph_coeff, negacyclic_mul


def small_pt(sc):
    return [sc.rnd.randint(-2, 2) for _ in range(sc.N)]


def setup(N, ML, L, A, KQ, seed, babies, giants):
    """keys for every non-identity element, a message, its encryption and n2 x n1 small plaintexts laid out for level KQ"""
    sc = Scheme(N, ML, A, seed=seed)
    keys = {g: sc.switch_key(automorph_coeff(sc.s, g, N), KQ) for g in set(babies) | set(giants) if g % (2 * N) != 1}
    msg = [(1 << 20) * sc.rnd.randint(-8, 8) for _ in range(N)]   # the transform stays below q_0 / 2 at L = 1
    ct = sc.encrypt(msg, L)
    polys = [[small_pt(sc) for _ in babies] for _ in giants]
    ext = list(range(KQ)) + [ML + j for j in range(A)]
    pts = [[sc.to_eval(p, ext) for p in row] for row in polys]
    return sc, keys, msg, ct, polys, pts


def run(sc, L, KQ, ct, babies, giants, keys, pts):
    return hrotate_bsgs_hoisted(sc.o, L, ct, babies, [keys.get(g) for g in babies], giants, [keys.get(g) for g in giants], KQ, pts, KQ)


def expected(N, msg, babies, giants, polys):
    want = [0] * N
    for G, row in zip(giants, polys):
        inner = [0] * N
        for b, p in zip(babies, row):
            inner = [x + y for x, y in zip(inner, negacyclic_mul(p, automorph_coeff(msg, b, N), N))]
        want = [x + y for x, y in zip(want, automorph_coeff(inner, G, N))]
    return want


def noise_bound(N, n1, n2):
    """every baby key switch's noise (< 64 N, test_oracle_semantics) times a plaintext with coefficients in [-2, 2]
    (|pt|_1 <= 2N), the fresh noise times the plaintexts, and one key switch per giant step; far below the 2^20-scaled signal"""
    return (n1 + 1) * n2 * 2 * N * 64 * N


@pytest.mark.parametrize("N,ML,L,A,KQ", CASES + [(64, 4, 1, 2, 1)])
@pytest.mark.parametrize("giant_identity", [True, False])
def test_bsgs_decrypts_to_the_linear_transform(N, ML, L, A, KQ, giant_identity):
    """baby steps {1, 5, 25}, giant steps {1, 125} or {125, 2N - 1}"""
    babies, giants = [1, 5, 25], ([1, 125] if giant_identity else [125, 2 * N - 1])
    sc, keys, msg, ct, polys, pts = setup(N, ML, L, A, KQ, 6000 + N + 7 * L + A + giant_identity, babies, giants)
    got = sc.decrypt(run(sc, L, KQ, ct, babies, giants, keys, pts), L)
    want = expected(N, msg, babies, giants, polys)
    err = max(abs(got[k] - want[k]) for k in range(N))
    assert max(abs(v) for v in want) > 2 ** 24
    assert err < noise_bound(N, len(babies), len(giants)), err


def test_negative_control_plaintexts_without_p_limbs_do_not_decrypt():
    """the bound above is meaningful: with the plaintexts' P-limbs zeroed the accumulators are no longer consistent over Q*P
    and the ModDown result is garbage of the size of Q"""
    N, ML, L, A, KQ = 64, 4, 4, 2, 4
    babies, giants = [1, 5, 25], [1, 125]
    sc, keys, msg, ct, polys, pts = setup(N, ML, L, A, KQ, 61, babies, giants)
    for row in pts:
        for p in row:
            p[KQ:] = 0
    got = sc.decrypt(run(sc, L, KQ, ct, babies, giants, keys, pts), L)
    want = expected(N, msg, babies, giants, polys)
    assert max(abs(got[k] - want[k]) for k in range(N)) > 2 ** 60


@pytest.mark.parametrize("N,ML,L,A,KQ", [(64, 4, 4, 2, 4), (64, 5, 3, 2, 5), (128, 6, 6, 3, 6), (64, 4, 1, 2, 1)])
def test_one_identity_giant_step_is_the_rotation_sum(N, ML, L, A, KQ):
    """n2 = 1, G_0 = 1 and no identity baby step: hrotate_sum_hoisted bit for bit"""
    babies = [5, 25, 2 * N - 1]
    sc, keys, msg, ct, polys, pts = setup(N, ML, L, A, KQ, 62 + N + L, babies, [1])
    got = run(sc, L, KQ, ct, babies, [1], keys, pts)
    assert np.array_equal(got, hrotate_sum_hoisted(sc.o, L, ct, [keys[g] for g in babies], KQ, babies, pts[0], KQ))


@pytest.mark.parametrize("N,ML,L,A,KQ", [(64, 4, 4, 2, 4), (64, 5, 3, 2, 5), (128, 6, 6, 3, 6), (64, 4, 1, 2, 1)])
@pytest.mark.parametrize("g_of", [lambda N: 5, lambda N: 2 * N - 1])
def test_identity_baby_and_one_giant_step_is_the_hoisted_rotation(N, ML, L, A, KQ, g_of):
    """n1 = 1, b_0 = 1, pt = 1, n2 = 1, G_0 = g: the inner sum is ct itself, so the op is hrotate_hoisted bit for bit"""
    sc = Scheme(N, ML, A, seed=63 + N + L)
    g = g_of(N)
    rk = sc.switch_key(automorph_coeff(sc.s, g, N), KQ)
    ct = sc.encrypt([(1 << 30) * sc.rnd.randint(-8, 8) for _ in range(N)], L)
    ones = np.ones((KQ + A, N), dtype=np.uint64)
    got = hrotate_bsgs_hoisted(sc.o, L, ct, [1], [None], [g], [rk], KQ, [[ones]], KQ)
    assert np.array_equal(got, sc.o.hrotate_hoisted(L, ct, [rk], KQ, [g])[0])


@pytest.mark.parametrize("N,ML,L,A,KQ", [(64, 4, 4, 2, 4), (128, 6, 6, 3, 6)])
def test_bsgs_is_not_the_textbook_hoisted_composition(N, ML, L, A, KQ):
    """n1, n2 >= 2: hoisted baby rotations, pmult / hadd per giant step, then a full rotation per giant step differ bit for
    bit from the double-hoisted result, yet both decrypt to the same message within the noise"""
    babies, giants = [1, 5, 25], [1, 125]
    sc, keys, msg, ct, polys, pts = setup(N, ML, L, A, KQ, 64 + N, babies, giants)
    got = run(sc, L, KQ, ct, babies, giants, keys, pts)
    o = sc.o
    rotated = dict(zip(babies[1:], o.hrotate_hoisted(L, ct, [keys[b] for b in babies[1:]], KQ, babies[1:])))
    rotated[1] = ct
    ref = None
    for G, row in zip(giants, pts):
        g_j = None
        for b, pt in zip(babies, row):
            t = o.pmult(L, rotated[b], np.ascontiguousarray(pt[:L]))
            g_j = t if g_j is None else o.hadd(L, g_j, t)
        if G != 1:
            g_j = o.hrotate(L, g_j, keys[G], KQ, G)
        ref = g_j if ref is None else o.hadd(L, ref, g_j)
    assert not np.array_equal(got, ref)
    a, b = sc.decrypt(got, L), sc.decrypt(ref, L)
    assert max(abs(x - y) for x, y in zip(a, b)) < 2 * noise_bound(N, len(babies), len(giants))
