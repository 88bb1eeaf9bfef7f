"""CPU tests of the double-hoisted rotation sum's oracle definition (tests/orc_rotsum.py, the reference for
hml_hrotate_sum_hoisted).  With real keys (test_oracle_semantics.Scheme) the sum decrypts to sum_i pt_i * sigma_i(m); with
n = 1 and pt = 1 it is the hoisted rotation bit for bit; for n >= 2 it is not the sum of the weighted hoisted rotations, which
is why it has a definition of its own."""
import numpy as np
import pytest

from orc_rotsum import hrotate_sum_hoisted
from test_oracle_semantics import CASES, Scheme, automorph_coeff, negacyclic_mul


def small_pt(sc):
    return [sc.rnd.randint(-2, 2) for _ in range(sc.N)]


def setup(N, ML, L, A, KQ, seed, n_pt=4):
    sc = Scheme(N, ML, A, seed=seed)
    gs = [5, 25, 2 * N - 1, 1][:n_pt]
    rks = [sc.switch_key(automorph_coeff(sc.s, g, N), KQ) for g in gs]
    msg = [(1 << 20) * sc.rnd.randint(-8, 8) for _ in range(N)]   # sum_i pt_i * sigma_i(m) stays below q_0 / 2 at L = 1
    ct = sc.encrypt(msg, L)
    polys = [small_pt(sc) for _ in gs]
    ext = list(range(KQ)) + [ML + j for j in range(A)]   # plaintexts laid out for level KQ: Q-limbs, then the P-limbs
    pts = [sc.to_eval(p, ext) for p in polys]
    return sc, gs, rks, msg, ct, polys, pts


@pytest.mark.parametrize("N,ML,L,A,KQ", CASES + [(64, 4, 1, 2, 1)])
def test_rotation_sum_decrypts_to_the_weighted_automorphisms(N, ML, L, A, KQ):
    """decrypt(sum op) ~ sum_i pt_i * sigma_i(m), galois elements 5, 25, 2N - 1 and 1.  Noise: every rotation's key-switch
    noise (< 64 N, test_oracle_semantics) times a plaintext with coefficients in [-2, 2] (|pt|_1 <= 2N), plus pt times the fresh
    noise; far below the 2^20-scaled signal."""
    sc, gs, rks, msg, ct, polys, pts = setup(N, ML, L, A, KQ, seed=4000 + N + 7 * L + A)
    got = sc.decrypt(hrotate_sum_hoisted(sc.o, L, ct, rks, KQ, gs, pts, KQ), L)
    want = [0] * N
    for g, p in zip(gs, polys):
        want = [x + y for x, y in zip(want, negacyclic_mul(p, automorph_coeff(msg, g, N), N))]
    err = max(abs(got[k] - want[k]) for k in range(N))
    assert max(abs(v) for v in want) > 2 ** 24
    assert err < len(gs) * 2 * N * 64 * N, err


def test_negative_control_plaintexts_without_p_limbs_do_not_decrypt():
    """the bound above is meaningful: with the plaintexts' P-limbs zeroed the accumulators are no longer consistent over Q*P
    and the ModDown result is garbage of the size of Q"""
    N, ML, L, A, KQ = 64, 4, 4, 2, 4
    sc, gs, rks, msg, ct, polys, pts = setup(N, ML, L, A, KQ, seed=41)
    for p in pts:
        p[KQ:] = 0
    got = sc.decrypt(hrotate_sum_hoisted(sc.o, L, ct, rks, KQ, gs, pts, KQ), L)
    want = [0] * N
    for g, p in zip(gs, polys):
        want = [x + y for x, y in zip(want, negacyclic_mul(p, automorph_coeff(msg, g, N), N))]
    assert max(abs(got[k] - want[k]) for k in range(N)) > 2 ** 60


@pytest.mark.parametrize("N,ML,L,A,KQ", [(64, 4, 4, 2, 4), (64, 5, 3, 2, 5), (128, 6, 6, 3, 6), (64, 4, 1, 2, 1)])
@pytest.mark.parametrize("g_of", [lambda N: 5, lambda N: 2 * N - 1, lambda N: 1])
def test_one_rotation_with_unit_plaintext_is_the_hoisted_rotation(N, ML, L, A, KQ, g_of):
    sc = Scheme(N, ML, A, seed=42 + N + L)
    g = g_of(N)
    rk = sc.switch_key(automorph_coeff(sc.s, g, N), KQ)
    ct = sc.encrypt([(1 << 30) * sc.rnd.randint(-8, 8) for _ in range(N)], L)
    ones = np.ones((KQ + A, N), dtype=np.uint64)
    got = hrotate_sum_hoisted(sc.o, L, ct, [rk], KQ, [g], [ones], KQ)
    assert np.array_equal(got, sc.o.hrotate_hoisted(L, ct, [rk], KQ, [g])[0])


@pytest.mark.parametrize("N,ML,L,A,KQ", [(64, 4, 4, 2, 4), (128, 6, 6, 3, 6)])
def test_sum_is_not_the_sum_of_weighted_hoisted_rotations(N, ML, L, A, KQ):
    sc, gs, rks, msg, ct, polys, pts = setup(N, ML, L, A, KQ, seed=43 + N)
    for n in (2, 4):
        got = hrotate_sum_hoisted(sc.o, L, ct, rks[:n], KQ, gs[:n], pts[:n], KQ)
        outs = sc.o.hrotate_hoisted(L, ct, rks[:n], KQ, gs[:n])
        ref = sc.o.pmult(L, outs[0], np.ascontiguousarray(pts[0][:L]))
        for out, pt in zip(outs[1:], pts[1:n]):
            ref = sc.o.hadd(L, ref, sc.o.pmult(L, out, np.ascontiguousarray(pt[:L])))
        assert not np.array_equal(got, ref)
        # ... yet both decrypt to the same message (within the noise): equally valid results
        a, b = sc.decrypt(got, L), sc.decrypt(ref, L)
        assert max(abs(x - y) for x, y in zip(a, b)) < n * 2 * N * 64 * N
