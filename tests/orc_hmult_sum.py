"""TEST INFRASTRUCTURE ONLY: the oracle definition of the lazily relinearised sum of products (hml_hmult_sum), composed from the
scalar C oracle's exported stages (tests/orc.py), so the key switch and the rescale are the oracle's own code, the stages
orc_hmult runs after its tensor product:

    D0 = sum_i a_i0 * b_i0,   D1 = sum_i (a_i0 * b_i1 + a_i1 * b_i0),   D2 = sum_i a_i1 * b_i1     mod q_l, l < L
    (o0, o1) = orc_keyswitch(D2)
    out      = ( orc_rescale(D0 + o0), orc_rescale(D1 + o1) )

With one term this is orc_hmult bit for bit.  The element-wise products are exact numpy arithmetic for moduli below 2^36 (the
rings of the tests)."""
import numpy as np

from orc_rotsum import mulmod


def hmult_sum(o, L, cts_a, cts_b, evk, evk_q_limbs):
    """cts_a[i], cts_b[i] [2][L][N]; evk [beta][2][evk_q_limbs + alpha][N]; returns [2][L-1][N]"""
    assert o.word_bits <= 36 and len(cts_a) == len(cts_b) >= 1
    m = np.array(o.moduli[:L], dtype=np.uint64)[:, None]
    d = np.zeros((3, L, o.N), dtype=np.uint64)
    for a, b in zip(cts_a, cts_b):
        a0, a1, b0, b1 = a[0] % m, a[1] % m, b[0] % m, b[1] % m
        d[0] = (d[0] + mulmod(a0, b0, m)) % m
        d[1] = (d[1] + mulmod(a0, b1, m) + mulmod(a1, b0, m)) % m
        d[2] = (d[2] + mulmod(a1, b1, m)) % m
    o0, o1 = o.keyswitch(L, np.ascontiguousarray(d[2]), np.ascontiguousarray(evk), evk_q_limbs)
    out = np.empty((2, L - 1, o.N), dtype=np.uint64)
    out[0] = o.rescale(L, np.ascontiguousarray((d[0] + o0) % m))
    out[1] = o.rescale(L, np.ascontiguousarray((d[1] + o1) % m))
    return out
