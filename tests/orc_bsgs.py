"""TEST INFRASTRUCTURE ONLY: the oracle definition of the double-hoisted baby-step / giant-step linear transform
(hml_hrotate_bsgs_hoisted), composed from the oracle stages tests/orc_rotsum.py uses: o.modup, o.automorph_index and
orc_rotsum's moddown / mulmod.  With IP_g(c) = sum_d sigma_g(ModUp(c)_d) * rk_g[d] over E = (q_0..q_{L-1}, p_0..p_{alpha-1}):

    acc_j = sum_{b_i != 1} pt_{j,i} * IP_{b_i}(c1)     z0_j = sum_i pt_{j,i} * sigma_{b_i}(c0)     z1_j = sum_{b_i = 1} pt_{j,i} * c1
    ct_j  = (ModDown(acc_j, 0) + z0_j, ModDown(acc_j, 1) + z1_j)                                    G_j != 1
    A     = sum_{G_j = 1} acc_j + sum_{G_j != 1} IP_{G_j}(ct_j.c1)
    Z0    = sum_{G_j = 1} z0_j  + sum_{G_j != 1} sigma_{G_j}(ct_j.c0)          Z1 = sum_{G_j = 1} z1_j
    out   = (ModDown(A, 0) + Z0, ModDown(A, 1) + Z1)

Identity elements (g = 1 mod 2N) use no key.  sigma is orc_automorph_eval's permutation, applied to every digit limb as
orc_hrotate_hoisted applies it."""
import numpy as np

from orc_rotsum import moddown, mulmod


def is_identity(o, g):
    return int(g) % (2 * o.N) == 1


def hrotate_bsgs_hoisted(o, L, ct, baby_galois, baby_keys, giant_galois, giant_keys, evk_q_limbs, pts, pt_q_limbs):
    """ct [2][L][N]; keys [beta][2][evk_q_limbs + alpha][N] (None allowed for identity elements); pts n2 lists of n1
    plaintexts [pt_q_limbs + alpha][N] (P-limb m at row pt_q_limbs + m); returns [2][L][N]"""
    A, N, ML = o.alpha, o.N, o.max_level
    assert o.word_bits <= 36 and L <= pt_q_limbs <= ML and L <= evk_q_limbs <= ML
    E, beta = L + A, -(-L // A)
    m = np.array([o.moduli[i] for i in o.ext_mod_idx(L)], dtype=np.uint64)[:, None]
    mq = m[:L]
    key_rows = list(range(L)) + [evk_q_limbs + j for j in range(A)]
    pt_rows = list(range(L)) + [pt_q_limbs + j for j in range(A)]

    def ip(t, rk, g):
        """IP_g for digits t = ModUp(c): [2][E][N]"""
        perm = o.automorph_index(int(g))
        out = np.zeros((2, E, N), dtype=np.uint64)
        for c in range(2):
            for d in range(beta):
                out[c] = (out[c] + mulmod(t[d][:, perm], rk[d, c][key_rows] % m, m)) % m
        return out

    t = o.modup(L, np.ascontiguousarray(ct[1]))
    acc_all = np.zeros((2, E, N), dtype=np.uint64)
    z_all = np.zeros((2, L, N), dtype=np.uint64)
    for j, G in enumerate(giant_galois):
        acc = np.zeros((2, E, N), dtype=np.uint64)
        z = np.zeros((2, L, N), dtype=np.uint64)
        for b, rk, pt in zip(baby_galois, baby_keys, pts[j]):
            w = pt[pt_rows] % m
            if is_identity(o, b):
                z[0] = (z[0] + mulmod(ct[0], w[:L], mq)) % mq
                z[1] = (z[1] + mulmod(ct[1], w[:L], mq)) % mq
                continue
            s = ip(t, rk, b)
            for c in range(2):
                acc[c] = (acc[c] + mulmod(s[c], w, m)) % m
            z[0] = (z[0] + mulmod(ct[0][:, o.automorph_index(int(b))], w[:L], mq)) % mq
        if is_identity(o, G):
            acc_all = (acc_all + acc) % m
            z_all = (z_all + z) % mq
            continue
        ct_j = (moddown(o, L, acc) + z) % mq
        acc_all = (acc_all + ip(o.modup(L, np.ascontiguousarray(ct_j[1])), giant_keys[j], G)) % m
        z_all[0] = (z_all[0] + ct_j[0][:, o.automorph_index(int(G))]) % mq
    return (moddown(o, L, acc_all) + z_all) % mq
