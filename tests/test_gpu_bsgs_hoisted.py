"""GPU parity of the double-hoisted BSGS linear transform (hml_hrotate_bsgs_hoisted, Context.hrotate_bsgs_hoisted): bit-exact
against the oracle definition in tests/orc_bsgs.py on single-pass and two-pass rings and at the north star, the corner case
that is the rotation sum, executed counts, rejections."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import homulator_b200 as hml  # noqa: E402
from gpu_common import to_dev, to_host  # noqa: E402
from orc import Oracle, uniform_limbs  # noqa: E402
from orc_bsgs import hrotate_bsgs_hoisted  # noqa: E402
from test_gpu_rotsum_hoisted import SHAPES  # noqa: E402

# (n1, n2, packed key, evk_q_limbs is maxLevel, pt_q_limbs is maxLevel, giant steps include the identity)
RUNS = [(1, 1, False, False, False, False), (3, 2, True, True, False, True), (4, 4, False, False, True, False),
        (4, 4, True, False, False, True), (17, 2, True, True, True, True), (2, 17, False, True, False, False)]


def steps(N, n1, n2, giant_identity):
    """baby steps 1, 5, 25, ... (always the identity first); giant steps 5^n1, 5^(2 n1), ... (and 2N - 1), after 1 if asked"""
    babies = [pow(5, i, 2 * N) for i in range(n1)]
    giants = [pow(5, n1 * j, 2 * N) for j in range(1, n2 + 1)]
    giants[-1] = 2 * N - 1
    if giant_identity:
        giants = [1] + giants[:n2 - 1]
    return babies, giants


def operands(o, L, babies, giants, evk_q, pt_q, seed):
    """ct [2][L][N]; one key per non-identity galois element (None for the identity); n2 x n1 plaintexts cycled over 7"""
    N, ML, A = o.N, o.max_level, o.alpha
    beta = -(-L // A)
    ct = uniform_limbs(o.moduli[:L], N, seed, lead=(2,))
    gs = sorted(set(babies) | set(giants))
    keys = {g: None if g == 1 else uniform_limbs(o.moduli[:evk_q] + o.moduli[ML:], N, seed + 1 + k, lead=(beta, 2)) for k, g in enumerate(gs)}
    pool = [uniform_limbs(o.moduli[:pt_q] + o.moduli[ML:], N, seed + 100 + k) for k in range(7)]
    pts = [[pool[(j * len(babies) + i) % 7] for i in range(len(babies))] for j in range(len(giants))]
    return ct, keys, pts


def device_call(ctx, L, ct, babies, giants, keys, pts, evk_q, pt_q, packed):
    dk = {g: None if k is None else to_dev(k) for g, k in keys.items()}
    if packed:
        dk = {g: None if k is None else ctx.key_pack(k) for g, k in dk.items()}
    dp = {id(p): to_dev(p) for row in pts for p in row}
    return ctx.hrotate_bsgs_hoisted(L, to_dev(ct), babies, [dk[g] for g in babies], giants, [dk[g] for g in giants],
                                    [[dp[id(p)] for p in row] for row in pts], evk_q_limbs=evk_q | (hml.KEY_PACKED if packed else 0),
                                    pt_q_limbs=pt_q)


@pytest.mark.parametrize("N,ML,L,A", SHAPES)
def test_bsgs_matches_oracle(N, ML, L, A):
    ctx, o = hml.Context(N=N, max_level=ML, alpha=A), Oracle(N, 36, ML, A)
    for n1, n2, packed, kq_max, pq_max, gid in RUNS:
        evk_q, pt_q = ML if kq_max else L, ML if pq_max else L
        babies, giants = steps(N, n1, n2, gid)
        ct, keys, pts = operands(o, L, babies, giants, evk_q, pt_q, 7000 + n1 + 31 * n2)
        want = hrotate_bsgs_hoisted(o, L, ct, babies, [keys[g] for g in babies], giants, [keys[g] for g in giants], evk_q, pts, pt_q)
        got = device_call(ctx, L, ct, babies, giants, keys, pts, evk_q, pt_q, packed)
        assert np.array_equal(to_host(got), want), (n1, n2, packed, evk_q, pt_q, gid)


def test_bsgs_north_star():
    """BASELINE.json's config (N = 2^16, maxLevel 45, L 35, alpha 15), 4 x 4 with the identity giant step, word and packed keys"""
    N, ML, L, A = 65536, 45, 35, 15
    Oracle.set_threads(0)
    ctx, o = hml.Context(N=N, max_level=ML, alpha=A), Oracle(N, 36, ML, A)
    babies, giants = steps(N, 4, 4, True)
    ct, keys, pts = operands(o, L, babies, giants, L, L, 7100)
    want = hrotate_bsgs_hoisted(o, L, ct, babies, [keys[g] for g in babies], giants, [keys[g] for g in giants], L, pts, L)
    got = device_call(ctx, L, ct, babies, giants, keys, pts, L, L, False)
    assert np.array_equal(to_host(got), want)
    got_p = device_call(ctx, L, ct, babies, giants, keys, pts, L, L, True)
    assert torch.equal(got_p, got)
    Oracle.set_threads(1)


@pytest.mark.parametrize("N,ML,L,A", [(256, 7, 7, 3), (8192, 9, 8, 3)])
def test_one_identity_giant_step_is_the_rotation_sum(N, ML, L, A):
    """n2 = 1, G = 1 and non-identity baby steps: hrotate_sum_hoisted bit for bit, across two groups of 16"""
    ctx = hml.Context(N=N, max_level=ML, alpha=A)
    beta = -(-L // A)
    ct = ctx.uniform(list(range(L)), 1, lead=(2,))
    for n in (3, 17):
        gs = [pow(5, r, 2 * N) for r in range(1, n + 1)]
        keys = [ctx.uniform(ctx.ext_mod_idx(L), 10 + r, lead=(beta, 2)) for r in range(n)]
        pts = [ctx.uniform(ctx.ext_mod_idx(L), 40 + r) for r in range(n)]
        got = ctx.hrotate_bsgs_hoisted(L, ct, gs, keys, [1], [None], [pts])
        assert torch.equal(got, ctx.hrotate_sum_hoisted(L, ct, keys, gs, pts)), n


def test_executed_counts():
    """With k non-identity giant steps the transforms and conversions are (k + 1) times those of a one-rotation
    hrotate_sum_hoisted, whatever the number of baby steps"""
    N, ML, L, A = 8192, 9, 8, 3
    ctx = hml.Context(N=N, max_level=ML, alpha=A)
    beta = -(-L // A)
    ct = ctx.uniform(list(range(L)), 1, lead=(2,))
    key = ctx.uniform(ctx.ext_mod_idx(L), 2, lead=(beta, 2))
    pt = ctx.uniform(ctx.ext_mod_idx(L), 3)

    def counts(fn):
        fn()  # warm: per-level tables exist
        ctx.exec_counts(reset=True)
        fn()
        torch.cuda.synchronize()
        return ctx.exec_counts()

    one = counts(lambda: ctx.hrotate_sum_hoisted(L, ct, [key], [5], [pt]))
    for gid in (True, False):
        for n2 in (1, 2, 4):
            per_n1 = []
            for n1 in (1, 3, 17):
                babies, giants = steps(N, n1, n2, gid)
                bk = [None if b == 1 else key for b in babies]
                gk = [None if g == 1 else key for g in giants]
                c = counts(lambda: ctx.hrotate_bsgs_hoisted(L, ct, babies, bk, giants, gk, [[pt] * n1 for _ in giants]))
                k = sum(1 for g in giants if g != 1)
                for name in ("ntt_limbs", "intt_limbs", "bconv_limb_macs"):
                    assert c[name] == (k + 1) * one[name], (gid, n2, n1, name)
                per_n1.append(c)
            for name in ("ntt_limbs", "intt_limbs", "bconv_limb_macs"):
                assert per_n1[0][name] == per_n1[1][name] == per_n1[2][name]


def test_rejections():
    N, ML, L, A = 1024, 5, 4, 2
    ctx = hml.Context(N=N, max_level=ML, alpha=A)
    beta = -(-L // A)
    ct = ctx.uniform(list(range(L)), 1, lead=(2,))
    key = ctx.uniform(ctx.ext_mod_idx(L), 2, lead=(beta, 2))
    pt = ctx.uniform(ctx.ext_mod_idx(L), 3)
    lib, C = ctx.lib, hml.api.C
    out = ctx.empty(2, L, N)
    k, p, o = key.data_ptr(), pt.data_ptr(), out.data_ptr()

    def arr(t, v):
        return (t * max(len(v), 1))(*v)

    def call(bg, bk, gg, gk, pts, out=o, evk_q=L, pt_q=L, src=ct.data_ptr(), level=L, n1=None, n2=None):
        n1 = len(bg) if n1 is None else n1
        n2 = len(gg) if n2 is None else n2
        return lib.hml_hrotate_bsgs_hoisted(ctx.h, level, src, n1, arr(C.c_uint64, bg), arr(C.c_void_p, bk), n2, arr(C.c_uint64, gg),
                                            arr(C.c_void_p, gk), evk_q, arr(C.c_void_p, pts), pt_q, out, None)

    ok = ([1, 5], [None, k], [1, 25], [None, k], [p] * 4)
    assert call(*ok) == 0
    invalid = [
        call([], [], [1], [None], [p], n1=0),                     # n1 = 0
        call([1], [None], [], [], [p], n2=0),                     # n2 = 0
        call([1, 5], [None, None], [1], [None], [p, p]),          # null key for a non-identity baby step
        call([1], [None], [1, 25], [None, None], [p, p]),         # null key for a non-identity giant step
        call(*ok[:4], [p, p, None, p]),                           # null plaintext
        call(*ok, out=None),                                      # null output
        call([1, 6], [None, k], [1, 25], [None, k], [p] * 4),     # even baby galois element
        call([1, 5], [None, k], [2, 25], [None, k], [p] * 4),     # even giant galois element
        call(*ok, out=ct.data_ptr()),                             # output == input
        call(*ok, out=ct.data_ptr() + 8 * N),                     # output overlapping the input
        call(*ok, evk_q=L - 1),                                   # evk_q_limbs below L
        call(*ok, evk_q=ML + 1),                                  # ... above maxLevel
        call(*ok, pt_q=L - 1),                                    # pt_q_limbs below L
        call(*ok, pt_q=ML + 1),                                   # ... above maxLevel
        call(*ok, level=ML + 1),                                  # level above maxLevel
        call(*ok, src=None),                                      # null input
    ]
    assert invalid == [1] * len(invalid)                          # HML_ERR_INVALID
    one, pa = arr(C.c_uint64, [1]), arr(C.c_void_p, [p])
    nulls = [lib.hml_hrotate_bsgs_hoisted(ctx.h, L, ct.data_ptr(), 1, None, None, 1, one, None, L, pa, L, o, None),   # baby galois
             lib.hml_hrotate_bsgs_hoisted(ctx.h, L, ct.data_ptr(), 1, one, None, 1, None, None, L, pa, L, o, None),   # giant galois
             lib.hml_hrotate_bsgs_hoisted(ctx.h, L, ct.data_ptr(), 1, one, None, 1, one, None, L, None, L, o, None)]  # plaintexts
    assert nulls == [1, 1, 1]
    # the key arrays themselves may be null when every element is the identity
    assert lib.hml_hrotate_bsgs_hoisted(ctx.h, L, ct.data_ptr(), 1, one, None, 1, one, None, L, pa, L, o, None) == 0
    # more than 8 digits: unsupported, as for every other key switch
    c9 = hml.Context(N=1024, max_level=9, alpha=1)
    ct9, key9, pt9 = c9.uniform(list(range(9)), 1, lead=(2,)), c9.uniform(c9.ext_mod_idx(9), 2, lead=(9, 2)), c9.uniform(c9.ext_mod_idx(9), 3)
    with pytest.raises(hml.HmlError) as e:
        c9.hrotate_bsgs_hoisted(9, ct9, [1, 5], [None, key9], [1], [None], [[pt9, pt9]])
    assert e.value.code == 4                                      # HML_ERR_UNSUPPORTED
    # the rejected calls enqueued nothing: the context still computes the same result
    want = ctx.hrotate_bsgs_hoisted(L, ct, [1, 5], [None, key], [1, 25], [None, key], [[pt, pt], [pt, pt]])
    assert call(*ok) == 0 and torch.equal(out, want)
