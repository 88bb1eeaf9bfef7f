"""GPU parity of the lazily relinearised sum of products (hml_hmult_sum, Context.hmult_sum) and of the replay flag that selects
it (HML_REPLAY_HMULT_SUM, Replay(..., hmult_sum=True)): bit-exact against the oracle definition in tests/orc_hmult_sum.py on a
single-pass and a two-pass ring and at the north star, one term against hml_hmult / hml_hmult_batch, executed counts,
rejections."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import homulator_b200 as hml  # noqa: E402
from gpu_common import to_dev, to_host  # noqa: E402
from homulator_b200.replay import dot_trace  # noqa: E402
from orc import Oracle, uniform_limbs  # noqa: E402
from orc_hmult_sum import hmult_sum  # noqa: E402

# (N, maxLevel, alpha) and levels: one digit, two digits with a short last one, three digits with a short last one, three full
RINGS = {"n4096": ((4096, 9, 3), (3, 5, 8, 9)), "n8192": ((8192, 9, 3), (3, 5, 8, 9))}
# (n_terms, n_out, packed key, evk_q_limbs is maxLevel, term kinds)
RUNS = [(1, 1, False, False, "products"), (1, 3, True, True, "squares"), (2, 1, True, False, "mixed"), (2, 3, False, True, "products"),
        (16, 1, False, True, "squares"), (16, 3, True, False, "mixed"), (17, 1, True, True, "products"), (17, 3, False, False, "mixed"),
        (33, 1, False, False, "mixed"), (33, 3, True, True, "products")]


@pytest.fixture(scope="module", params=list(RINGS))
def ring(request):
    (N, ML, A), levels = RINGS[request.param]
    Oracle.set_threads(0)  # all host cores for the checker
    ctx, o = hml.Context(N=N, max_level=ML, alpha=A), Oracle(N, 36, ML, A)
    yield ctx, o, levels
    ctx.close()
    Oracle.set_threads(1)


def _key(o, L, evk_q, seed):
    beta = -(-L // o.alpha)
    return uniform_limbs(o.moduli[:evk_q] + o.moduli[o.max_level:], o.N, seed, lead=(beta, 2))


def _terms(o, L, n, n_out, kinds, seed, k=5):
    """a pool of k ciphertext batches [n_out][2][L][N] (host and device) and n terms over it: products of two different pool
    entries, squares (the same tensor twice), or both alternating"""
    pool = [uniform_limbs(o.moduli[:L], o.N, seed + i, lead=(n_out, 2)) for i in range(k)]
    dev = [to_dev(p) for p in pool]
    ia = [i % k for i in range(n)]
    sq = [kinds == "squares" or (kinds == "mixed" and i % 2 == 0) for i in range(n)]
    ib = [a if s else (a + 1 + i // k) % k for i, (a, s) in enumerate(zip(ia, sq))]
    return [pool[i] for i in ia], [pool[i] for i in ib], [dev[i] for i in ia], [dev[i] for i in ib]


def _check(ctx, o, L, n, n_out, packed, kq, kinds, seed):
    ha, hb, da, db = _terms(o, L, n, n_out, kinds, seed)
    evk = _key(o, L, kq, seed + 100)
    K = to_dev(evk)
    if packed:
        K = ctx.key_pack(K)
    got = to_host(ctx.hmult_sum(L, da, db, K, evk_q_limbs=kq | (hml.KEY_PACKED if packed else 0)))
    assert got.shape == (n_out, 2, L - 1, o.N)
    for k in range(n_out):
        want = hmult_sum(o, L, [a[k] for a in ha], [b[k] for b in hb], evk, kq)
        assert np.array_equal(got[k], want), (L, n, n_out, packed, kq, kinds, k)


@pytest.mark.parametrize("li", range(4))
def test_sum_matches_oracle(ring, li):
    ctx, o, levels = ring
    L = levels[li]
    for n, n_out, packed, kq_max, kinds in RUNS:
        _check(ctx, o, L, n, n_out, packed, o.max_level if kq_max else L, kinds, 6000 + 37 * n + n_out)


def test_sum_north_star():
    """BASELINE.json's config (N = 2^16, maxLevel 45, L 35, alpha 15): 16 and 17 terms, word and packed keys"""
    N, ML, L, A = 65536, 45, 35, 15
    Oracle.set_threads(0)
    ctx, o = hml.Context(N=N, max_level=ML, alpha=A), Oracle(N, 36, ML, A)
    _check(ctx, o, L, 16, 1, False, L, "mixed", 6100)
    _check(ctx, o, L, 17, 1, True, L, "products", 6200)
    ctx.close()
    Oracle.set_threads(1)


@pytest.mark.parametrize("n_out", [1, 5, 65, 70])
def test_one_term_is_hmult(ring, n_out):
    """n = 1 is hml_hmult (n_out = 1) and hml_hmult_batch (n_out > 1; chunks of 64, 65 and 70 leave partial last chunks) bit for
    bit, for a product and a square.  On the two-pass ring the batches take the stored tensor-product path."""
    ctx, o, levels = ring
    L = levels[2]
    _, _, (a, b), _ = _terms(o, L, 2, n_out, "products", 6300)
    K = to_dev(_key(o, L, L, 6400))
    for x, y in ((a, b), (a, a)):
        got = ctx.hmult_sum(L, [x], [y], K)
        if n_out == 1:
            assert torch.equal(got, ctx.hmult(L, x[0], y[0], K).unsqueeze(0))
            assert torch.equal(ctx.hmult_sum(L, [x[0]], [y[0]], K), got[0])   # [2][L][N] terms give one [2][L-1][N] output
        else:
            assert torch.equal(got, ctx.hmult_batch(L, x, y, K))


def test_executed_counts(ring):
    """Transforms and conversions are those of hml_hmult / hml_hmult_batch whatever the number of terms; ewe_limbs grows by 3L
    per term and output; one more launch per further group of 16 terms and chunk of outputs."""
    ctx, o, levels = ring
    L = levels[2]
    K = to_dev(_key(o, L, L, 6500))

    def counts(fn):
        fn()  # warm: per-level tables exist
        torch.cuda.synchronize()
        ctx.exec_counts(reset=True)
        fn()
        torch.cuda.synchronize()
        return ctx.exec_counts()

    for n_out in (1, 3, 70):
        _, _, da, db = _terms(o, L, 33, n_out, "mixed", 6600)
        ref = counts(lambda: ctx.hmult_batch(L, da[0], db[0], K) if n_out > 1 else ctx.hmult(L, da[0][0], db[0][0], K))
        c = {n: counts(lambda: ctx.hmult_sum(L, da[:n], db[:n], K)) for n in (1, 2, 16, 17, 33)}
        chunks = -(-n_out // 64)
        for n in c:
            for k in ("ntt_limbs", "intt_limbs", "bconv_limb_macs", "automorph_limbs"):
                assert c[n][k] == ref[k], (n_out, n, k)
            assert c[n]["ewe_limbs"] - c[1]["ewe_limbs"] == 3 * L * (n - 1) * n_out, (n_out, n)
            assert c[n]["kernel_launches"] - c[1]["kernel_launches"] == (-(-n // 16) - 1) * chunks, (n_out, n)
        if n_out == 1:
            assert c[1] == ref


def test_rejections():
    N, ML, L, A = 1024, 5, 4, 2
    ctx = hml.Context(N=N, max_level=ML, alpha=A)
    beta = -(-L // A)
    a = ctx.uniform(list(range(L)), 1, lead=(2, 2))
    b = ctx.uniform(list(range(L)), 2, lead=(2, 2))
    key = ctx.uniform(ctx.ext_mod_idx(L), 3, lead=(beta, 2))
    lib, C = ctx.lib, hml.api.C
    out = ctx.empty(2, 2, L - 1, N)
    k, o = key.data_ptr(), out.data_ptr()

    def call(pa, pb, out_ptr, n_out=2, key_ptr=k, kq=L, level=L):
        n = len(pa)
        aa = (C.c_void_p * max(n, 1))(*pa)
        ba = (C.c_void_p * max(n, 1))(*pb)
        return lib.hml_hmult_sum(ctx.h, level, n, aa, ba, n_out, key_ptr, kq, out_ptr, None)

    A_, B_ = a.data_ptr(), b.data_ptr()
    assert call([A_], [B_], o) == 0
    invalid = [
        call([A_], [B_], o, level=1),                              # L < 2
        call([A_], [B_], o, level=ML + 1),                         # level above maxLevel
        call([], [], o),                                           # no term
        call([None], [B_], o),                                     # null entry
        call([A_, A_], [B_, None], o),                             # ... in a later term
        call([A_], [B_], o, key_ptr=None),                         # null key
        call([A_], [B_], None),                                    # null output
        call([A_], [B_], A_),                                      # output == an input
        call([A_, A_], [A_, B_], B_ + 8 * N * (2 * L - 1)),        # output overlapping the last limb of the second term's b
        call([A_], [B_], o, kq=L - 1),                             # evk_q_limbs below L
        call([A_], [B_], o, kq=ML + 1),                            # ... above maxLevel
    ]
    assert invalid == [1] * len(invalid)                          # HML_ERR_INVALID
    assert lib.hml_hmult_sum(ctx.h, L, 1, None, None, 2, k, L, o, None) == 1   # null arrays
    # an empty batch is a no-op whatever the pointers are
    before = out.clone()
    assert lib.hml_hmult_sum(ctx.h, L, 0, None, None, 0, None, 0, None, None) == 0
    assert call([A_], [B_], o, n_out=0) == 0
    torch.cuda.synchronize()
    assert torch.equal(out, before)
    # more than 8 digits: unsupported, as for every other key switch
    c9 = hml.Context(N=1024, max_level=9, alpha=1)
    a9, k9 = c9.uniform(list(range(9)), 1, lead=(2,)), c9.uniform(c9.ext_mod_idx(9), 2, lead=(9, 2))
    with pytest.raises(hml.HmlError) as e:
        c9.hmult_sum(9, [a9], [a9], k9)
    assert e.value.code == 4                                      # HML_ERR_UNSUPPORTED
    # the rejected calls enqueued nothing: the context still computes the same result
    want = ctx.hmult_sum(L, [a], [b], key)
    assert call([A_], [B_], o) == 0 and torch.equal(out, want)


def _dot_operands(ctx, o, L, n):
    N, A = o.N, o.alpha
    beta = -(-L // A)
    x = to_dev(uniform_limbs(o.moduli[:L], N, 1, lead=(2,)))
    keys = {r: to_dev(uniform_limbs(o.moduli[:L] + o.moduli[o.max_level:], N, 200 + r, lead=(beta, 2))) for r in range(1, n)}
    evk = to_dev(uniform_limbs(o.moduli[:L] + o.moduli[o.max_level:], N, 300, lead=(beta, 2)))
    return x, keys, evk


@pytest.mark.parametrize("n", [5, 17])
def test_replay_dot_trace(n):
    """dot_trace(n) with hmult_sum=True, as launches and as a graph run twice, with and without hoisted rotations: y equals the
    rotations followed by Context.hmult_sum called directly, and differs from the replay without the flag; a shard refuses it."""
    N, ML, A, L = 8192, 7, 3, 7
    ctx, o = hml.Context(N=N, max_level=ML, alpha=A), Oracle(N, 36, ML, A)
    x, keys, evk = _dot_operands(ctx, o, L, n)
    trace = dot_trace(n)
    gs = [pow(5, r, 2 * N) for r in range(1, n)]
    for hoist in (False, True):
        rots = ctx.hrotate_hoisted(L, x, [keys[r] for r in range(1, n)], gs) if hoist else \
            [ctx.hrotate(L, x, keys[r], g) for r, g in zip(range(1, n), gs)]
        want = ctx.hmult_sum(L, [x] * n, [x] + rots, evk)
        plain = hml.Replay(ctx, L, trace, hoist=hoist).bind(x, [], keys, evk)
        assert not torch.equal(plain.run().result("y"), want)
        plain.close()
        for graph in (False, True):
            rp = hml.Replay(ctx, L, trace, graph=graph, hoist=hoist, hmult_sum=True).bind(x, [], keys, evk)
            for _ in range(2 if graph else 1):
                rp.run()
                assert torch.equal(rp.result("y"), want), (graph, hoist)
            rp.close()
    sh = hml.Shard(ctx, L, 0, 1)
    with pytest.raises(hml.HmlError) as e:
        hml.Replay(ctx, L, trace, shard=sh, hmult_sum=True)
    assert e.value.code == 4                                      # HML_ERR_UNSUPPORTED
    sh.close()
    ctx.close()


def test_replay_hmult_sum_conditions():
    """Chains that do not qualify run as without the flag: a temporary read after the chain, and a temporary whose earlier
    content is a source of the chain's first product.  A product of the chain cannot read y, nor run at another level: the
    trace's level rule (the sources of hadd at one level) already refuses such traces, with the flag or without.  The other
    flags combine with this one, and a qualifying chain written as hadd(y, t, y) is fused."""
    N, ML, A, L = 4096, 5, 2, 4
    ctx = hml.Context(N=N, max_level=ML, alpha=A)
    beta = -(-L // A)
    x = ctx.uniform(list(range(L)), 1, lead=(2,))
    keys = {r: ctx.uniform(ctx.ext_mod_idx(L), 200 + r, lead=(beta, 2)) for r in (1, 2, 3)}
    evk = ctx.uniform(ctx.ext_mod_idx(L), 300, lead=(beta, 2))
    rot = [("hrotate", "r1", "x", 1), ("hrotate", "r2", "x", 2), ("hrotate", "r3", "x", 3)]
    chain = [("hmult", "y", "x", "r1"), ("hmult", "m", "x", "r2"), ("hadd", "y", "y", "m"), ("hmult", "m", "r3", "x"), ("hadd", "y", "m", "y")]
    t_live = rot + chain + [("hadd", "w", "m", "y")]
    t_source = rot + [("padd", "m", "r3", 0), ("hmult", "y", "x", "m"), ("hmult", "m", "x", "r2"), ("hadd", "y", "y", "m")]
    pt = [ctx.uniform(list(range(L)), 400)]
    for tr, names in ((t_live, ("y", "w")), (t_source, ("y",))):
        for graph in (False, True):
            for hoist in (False, True):
                ref = hml.Replay(ctx, L, tr, graph=graph, hoist=hoist).bind(x, pt, keys, evk)
                rp = hml.Replay(ctx, L, tr, graph=graph, hoist=hoist, hoist_sum=True, hmult_sum=True).bind(x, pt, keys, evk)
                ref.run()
                rp.run()
                for name in names:
                    assert torch.equal(rp.result(name), ref.result(name)), (name, graph, hoist)
                rp.close()
                ref.close()
    y_source = rot + [("hmult", "y", "x", "r1"), ("hmult", "m", "y", "y"), ("hadd", "y", "y", "m")]
    mixed = rot + [("hmult", "u", "x", "r3"), ("hmult", "y", "x", "r1"), ("hmult", "m", "u", "u"), ("hadd", "y", "y", "m")]
    for tr in (y_source, mixed):
        for flag in (False, True):
            with pytest.raises(hml.HmlError) as e:
                hml.Replay(ctx, L, tr, hmult_sum=flag)
            assert e.value.code == 1                              # HML_ERR_INVALID: sources of one hadd at two levels
    rp = hml.Replay(ctx, L, rot + chain, hmult_sum=True).bind(x, [], keys, evk)
    got = rp.run().result("y").clone()
    rp.close()
    r = [ctx.hrotate(L, x, keys[i], pow(5, i, 2 * N)) for i in (1, 2, 3)]
    assert torch.equal(got, ctx.hmult_sum(L, [x, x, r[2]], [r[0], r[1], x], evk))
    ctx.close()
