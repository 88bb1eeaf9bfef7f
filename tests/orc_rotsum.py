"""TEST INFRASTRUCTURE ONLY: the oracle definition of the double-hoisted rotation sum (hml_hrotate_sum_hoisted), composed from
the scalar C oracle's exported stages (tests/orc.py), so the shared ModUp and ModDown are the oracle's own code:

    t        = orc_modup(c1)                                                     K1..K4, once
    acc_c[m] = sum_i pt_i[m] * ( sum_j sigma_i(t_j)[m] * rk_i[j][c][m] )  mod m,  m in E = (q_0..q_{L-1}, p_0..p_{alpha-1})
    z[l]     = sum_i pt_i[l] * sigma_i(c0)[l]                             mod q_l, l < L
    out      = ( z + ModDown(acc_0), ModDown(acc_1) )                            K6..K10, once

sigma_i is orc_automorph_eval's permutation, applied to every digit limb (own-digit limbs included) exactly as
orc_hrotate_hoisted applies it.  ModDown is orc_keyswitch_digits run on digits that make its K5 the identity (digit 0 = 1 on
every limb, the others 0, the accumulators in the key's digit-0 slots), so K6..K10 are the oracle's own.  The element-wise
products are exact numpy arithmetic for moduli below 2^36 (the rings of the tests)."""
import numpy as np

from orc import _p, lib


def mulmod(a, b, m):
    """a * b mod m for uint64 arrays with a, b < m < 2^36: b is split into 18-bit halves so that no product exceeds 2^55"""
    hi = (a * (b >> np.uint64(18))) % m
    return ((hi << np.uint64(18)) + a * (b & np.uint64(0x3FFFF))) % m


def moddown(o, L, acc):
    """K6..K10 of the oracle's key switch on given accumulators acc [2][L + alpha][N] -> (out0, out1) [L][N]"""
    A, N = o.alpha, o.N
    beta = -(-L // A)
    t = np.zeros((beta, L + A, N), dtype=np.uint64)
    t[0] = 1
    key = np.zeros((beta, 2, L + A, N), dtype=np.uint64)
    key[0] = acc
    out = np.empty((2, L, N), dtype=np.uint64)
    lib().orc_keyswitch_digits(o.h, L, _p(t), _p(key), L, _p(out[0]), _p(out[1]))
    return out


def hrotate_sum_hoisted(o, L, ct, rotkeys, evk_q_limbs, galois, pts, pt_q_limbs):
    """ct [2][L][N]; rotkeys[i] [beta][2][evk_q_limbs + alpha][N]; pts[i] [pt_q_limbs + alpha][N] (P-limb j at row
    pt_q_limbs + j); returns [2][L][N]"""
    A, N, ML = o.alpha, o.N, o.max_level
    assert o.word_bits <= 36 and L <= pt_q_limbs <= ML and L <= evk_q_limbs <= ML
    E, beta = L + A, -(-L // A)
    m = np.array([o.moduli[i] for i in o.ext_mod_idx(L)], dtype=np.uint64)[:, None]
    key_rows = list(range(L)) + [evk_q_limbs + j for j in range(A)]
    pt_rows = list(range(L)) + [pt_q_limbs + j for j in range(A)]
    t = o.modup(L, np.ascontiguousarray(ct[1]))
    acc = np.zeros((2, E, N), dtype=np.uint64)
    z = np.zeros((L, N), dtype=np.uint64)
    for rk, g, pt in zip(rotkeys, galois, pts):
        perm = o.automorph_index(int(g))  # sigma: out[k] = in[perm[k]]
        w = pt[pt_rows] % m
        for c in range(2):
            s = np.zeros((E, N), dtype=np.uint64)
            for j in range(beta):
                s = (s + mulmod(t[j][:, perm], rk[j, c][key_rows] % m, m)) % m
            acc[c] = (acc[c] + mulmod(s, w, m)) % m
        z = (z + mulmod(ct[0][:, perm], w[:L], m[:L])) % m[:L]
    out = moddown(o, L, acc)
    out[0] = (out[0] + z) % m[:L]
    return out
