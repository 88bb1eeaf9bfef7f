"""GPU parity of the double-hoisted rotation sum (hml_hrotate_sum_hoisted, Context.hrotate_sum_hoisted) and of the replay flag
that selects it (HML_REPLAY_HOIST_SUM, Replay(..., hoist_sum=True)): bit-exact against the oracle definition in
tests/orc_rotsum.py on single-pass and two-pass rings and at the north star, executed counts, rejections."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import homulator_b200 as hml  # noqa: E402
from gpu_common import to_dev, to_host  # noqa: E402
from homulator_b200.replay import bsgs_trace, rotsum_trace  # noqa: E402
from orc import Oracle, uniform_limbs  # noqa: E402
from orc_rotsum import hrotate_sum_hoisted  # noqa: E402

# (N, maxLevel, L, alpha): the shapes of test_gpu_ops.SMALL (beta = 1, L % alpha != 0, L < alpha, L = 1, several digits) and
# two-pass rings (N = 8192)
SHAPES = [(16, 6, 6, 2), (16, 6, 5, 2), (16, 5, 2, 3), (64, 4, 4, 4), (256, 7, 7, 3), (1024, 3, 1, 2), (4096, 9, 8, 3),
          (8192, 9, 8, 3), (8192, 6, 5, 2), (8192, 4, 1, 2)]
# (n_rot, packed key, evk_q_limbs is maxLevel, pt_q_limbs is maxLevel)
RUNS = [(1, False, False, False), (3, True, True, False), (16, False, False, True), (17, True, True, True), (33, False, True, False)]


def galois_pool(N):
    return [1, 2 * N - 1] + [pow(5, r, 2 * N) for r in range(1, 6)]


def operands(o, L, n, evk_q, pt_q, seed):
    """ct [2][L][N]; n keys and plaintexts cycled over a few distinct ones; galois elements cycled over galois_pool"""
    N, ML, A = o.N, o.max_level, o.alpha
    beta = -(-L // A)
    ct = uniform_limbs(o.moduli[:L], N, seed, lead=(2,))
    keys = [uniform_limbs(o.moduli[:evk_q] + o.moduli[ML:], N, seed + 1 + k, lead=(beta, 2)) for k in range(5)]
    pts = [uniform_limbs(o.moduli[:pt_q] + o.moduli[ML:], N, seed + 10 + k) for k in range(7)]
    gp = galois_pool(N)
    return ct, [keys[i % 5] for i in range(n)], [gp[i % len(gp)] for i in range(n)], [pts[i % 7] for i in range(n)]


@pytest.mark.parametrize("N,ML,L,A", SHAPES)
def test_rotation_sum_matches_oracle(N, ML, L, A):
    ctx, o = hml.Context(N=N, max_level=ML, alpha=A), Oracle(N, 36, ML, A)
    for n, packed, kq_max, pq_max in RUNS:
        evk_q, pt_q = ML if kq_max else L, ML if pq_max else L
        ct, keys, gs, pts = operands(o, L, n, evk_q, pt_q, 5000 + n)
        want = hrotate_sum_hoisted(o, L, ct, keys, evk_q, gs, pts, pt_q)
        dk = {id(k): to_dev(k) for k in keys}
        if packed:
            dk = {i: ctx.key_pack(k) for i, k in dk.items()}
        dp = {id(p): to_dev(p) for p in pts}
        got = ctx.hrotate_sum_hoisted(L, to_dev(ct), [dk[id(k)] for k in keys], gs, [dp[id(p)] for p in pts],
                                      evk_q_limbs=evk_q | (hml.KEY_PACKED if packed else 0), pt_q_limbs=pt_q)
        assert np.array_equal(to_host(got), want), (n, packed, evk_q, pt_q)


def test_rotation_sum_north_star():
    """BASELINE.json's config (N = 2^16, maxLevel 45, L 35, alpha 15): 16 rotations in one group, word and packed keys"""
    N, ML, L, A = 65536, 45, 35, 15
    Oracle.set_threads(0)
    ctx, o = hml.Context(N=N, max_level=ML, alpha=A), Oracle(N, 36, ML, A)
    ct, keys, gs, pts = operands(o, L, 16, L, L, 5100)
    want = hrotate_sum_hoisted(o, L, ct, keys, L, gs, pts, L)
    dk = {id(k): to_dev(k) for k in keys}
    dp = [to_dev(p) for p in pts]
    got = ctx.hrotate_sum_hoisted(L, to_dev(ct), [dk[id(k)] for k in keys], gs, dp)
    assert np.array_equal(to_host(got), want)
    pk = {i: ctx.key_pack(k) for i, k in dk.items()}
    got_p = ctx.hrotate_sum_hoisted(L, to_dev(ct), [pk[id(k)] for k in keys], gs, dp, evk_q_limbs=L | hml.KEY_PACKED)
    assert torch.equal(got_p, got)
    Oracle.set_threads(1)


@pytest.mark.parametrize("N,ML,L,A", [(256, 7, 7, 3), (8192, 9, 8, 3)])
def test_one_rotation_with_unit_plaintext_is_the_hoisted_rotation(N, ML, L, A):
    ctx = hml.Context(N=N, max_level=ML, alpha=A)
    beta = -(-L // A)
    ct = ctx.uniform(list(range(L)), 1, lead=(2,))
    key = ctx.uniform(ctx.ext_mod_idx(L), 2, lead=(beta, 2))
    ones = torch.ones(L + A, N, dtype=torch.int64, device=ctx.device)
    for g in (5, 2 * N - 1, 1):
        got = ctx.hrotate_sum_hoisted(L, ct, [key], [g], [ones])
        assert torch.equal(got, ctx.hrotate_hoisted(L, ct, [key], [g])[0]), g


def test_executed_counts():
    """The transforms and conversions do not grow with the number of rotations; each extra group of 16 rotations costs one
    launch (the later group adds to the stored sums)."""
    N, ML, L, A = 8192, 9, 8, 3
    ctx = hml.Context(N=N, max_level=ML, alpha=A)
    beta, E = -(-L // A), L + A
    ct = ctx.uniform(list(range(L)), 1, lead=(2,))
    key = ctx.uniform(ctx.ext_mod_idx(L), 2, lead=(beta, 2))
    pt = ctx.uniform(ctx.ext_mod_idx(L), 3)
    counts = {}
    for n in (2, 16, 17, 33):
        gs = [pow(5, r, 2 * N) for r in range(1, n + 1)]
        ctx.hrotate_sum_hoisted(L, ct, [key] * n, gs, [pt] * n)  # warm: per-level tables exist
        ctx.exec_counts(reset=True)
        ctx.hrotate_sum_hoisted(L, ct, [key] * n, gs, [pt] * n)
        torch.cuda.synchronize()
        counts[n] = ctx.exec_counts()
    for k in ("ntt_limbs", "intt_limbs", "bconv_limb_macs"):
        assert counts[2][k] == counts[16][k] == counts[33][k], k
    assert counts[17]["kernel_launches"] == counts[16]["kernel_launches"] + 1
    assert counts[33]["kernel_launches"] == counts[16]["kernel_launches"] + 2
    assert counts[16]["kernel_launches"] == counts[2]["kernel_launches"]
    for n in (2, 16, 33):
        assert counts[n]["ewe_limbs"] - counts[2]["ewe_limbs"] == (n - 2) * (2 * beta * E + 2 * E + L)
        assert counts[n]["automorph_limbs"] == n * L


def test_rejections():
    N, ML, L, A = 1024, 5, 4, 2
    ctx = hml.Context(N=N, max_level=ML, alpha=A)
    beta = -(-L // A)
    ct = ctx.uniform(list(range(L)), 1, lead=(2,))
    key = ctx.uniform(ctx.ext_mod_idx(L), 2, lead=(beta, 2))
    pt = ctx.uniform(ctx.ext_mod_idx(L), 3)
    lib, C = ctx.lib, hml.api.C

    def call(n, keys, gs, pts, out, evk_q=L, pt_q=L, src=ct, level=L):
        ka = (C.c_void_p * max(n, 1))(*keys)
        pa = (C.c_void_p * max(n, 1))(*pts)
        ga = (C.c_uint64 * max(n, 1))(*gs)
        return lib.hml_hrotate_sum_hoisted(ctx.h, level, src.data_ptr(), n, ka, evk_q, ga, pa, pt_q, out, None)

    out = ctx.empty(2, L, N)
    k, p, o = key.data_ptr(), pt.data_ptr(), out.data_ptr()
    assert call(1, [k], [5], [p], o) == 0
    invalid = [
        call(0, [], [], [], o),                                   # no rotation
        call(1, [None], [5], [p], o),                             # null key
        call(1, [k], [5], [None], o),                             # null plaintext
        call(1, [k], [5], [p], None),                             # null output
        call(2, [k, k], [5, 6], [p, p], o),                       # even galois element
        call(1, [k], [5], [p], ct.data_ptr()),                    # output == input
        call(1, [k], [5], [p], ct.data_ptr() + 8 * N),            # output overlapping the input
        call(1, [k], [5], [p], o, evk_q=L - 1),                   # evk_q_limbs below L
        call(1, [k], [5], [p], o, evk_q=ML + 1),                  # ... above maxLevel
        call(1, [k], [5], [p], o, pt_q=L - 1),                    # pt_q_limbs below L
        call(1, [k], [5], [p], o, pt_q=ML + 1),                   # ... above maxLevel
        call(1, [k], [5], [p], o, level=ML + 1),                  # level above maxLevel
    ]
    assert invalid == [1] * len(invalid)                          # HML_ERR_INVALID
    assert lib.hml_hrotate_sum_hoisted(ctx.h, L, ct.data_ptr(), 1, None, L, None, None, L, o, None) == 1   # null arrays
    # more than 8 digits: unsupported, as for every other key switch
    c9 = hml.Context(N=1024, max_level=9, alpha=1)
    ct9, key9, pt9 = c9.uniform(list(range(9)), 1, lead=(2,)), c9.uniform(c9.ext_mod_idx(9), 2, lead=(9, 2)), c9.uniform(c9.ext_mod_idx(9), 3)
    with pytest.raises(hml.HmlError) as e:
        c9.hrotate_sum_hoisted(9, ct9, [key9], [5], [pt9])
    assert e.value.code == 4                                      # HML_ERR_UNSUPPORTED
    # the rejected calls enqueued nothing: the context still computes the same result
    want = ctx.hrotate_sum_hoisted(L, ct, [key], [5], [pt])
    assert call(1, [k], [5], [p], o) == 0 and torch.equal(out, want)


def _fused_oracle(o, L, trace, x, pts, keys, evk):
    """y of rotsum_trace with the run of rotations and its accumulation chain as one double-hoisted sum, z = hmult(y, y)"""
    N = o.N
    rots = [op for op in trace if op[0] == "hrotate"]
    weight = {op[2]: op[3] for op in trace if op[0] == "pmult"}
    y = hrotate_sum_hoisted(o, L, x, [keys[op[3]] for op in rots], L, [pow(5, op[3], 2 * N) for op in rots],
                            [pts[weight[op[1]]] for op in rots], L)
    return {"y": y, "z": o.hmult(L, y, y, evk, L)}


@pytest.mark.parametrize("n", [5, 17])
def test_replay_hoist_sum(n):
    """rotsum_trace(n) with hoist_sum=True, as launches and as a graph run twice: y and z against the oracle with the fused
    sum, and different from the hoisted replay; a trace without the pattern is unchanged by the flag; a shard refuses it."""
    N, ML, A, L = 8192, 7, 3, 7
    ctx, o = hml.Context(N=N, max_level=ML, alpha=A), Oracle(N, 36, ML, A)
    Oracle.set_threads(0)
    beta = -(-L // A)
    trace = rotsum_trace(n)
    x = uniform_limbs(o.moduli[:L], N, 1, lead=(2,))
    pts = {i: uniform_limbs(o.moduli[:L] + o.moduli[ML:], N, 100 + i) for i in range(max(n, 6))}   # bsgs_trace(3, 2) uses 6
    keys = {r: uniform_limbs(o.moduli[:L] + o.moduli[ML:], N, 200 + r, lead=(beta, 2)) for r in range(1, n + 1)}
    evk = uniform_limbs(o.moduli[:L] + o.moduli[ML:], N, 300, lead=(beta, 2))
    dx, dp, dk, de = to_dev(x), {k: to_dev(v) for k, v in pts.items()}, {k: to_dev(v) for k, v in keys.items()}, to_dev(evk)
    want = _fused_oracle(o, L, trace, x, pts, keys, evk)
    hoisted = hml.Replay(ctx, L, trace, hoist=True).bind(dx, dp, dk, de)
    h = {k: to_host(hoisted.run().result(k)) for k in ("y", "z")}
    hoisted.close()
    assert not np.array_equal(h["y"], want["y"]) and not np.array_equal(h["z"], want["z"])
    for graph in (False, True):
        for hoist in (False, True):
            rp = hml.Replay(ctx, L, trace, graph=graph, hoist=hoist, hoist_sum=True).bind(dx, dp, dk, de)
            for _ in range(2 if graph else 1):
                rp.run()
                assert np.array_equal(to_host(rp.result("y")), want["y"]), (graph, hoist)
                assert np.array_equal(to_host(rp.result("z")), want["z"]), (graph, hoist)
            rp.close()
    # bsgs_trace(3, 2) has no run of rotations followed by an accumulation of all their outputs: bit-identical without the flag
    tr = bsgs_trace(3, 2)
    for graph in (False, True):
        for hoist in (False, True):
            ref = hml.Replay(ctx, L, tr, graph=graph, hoist=hoist).bind(dx, dp, dk, de)
            rp = hml.Replay(ctx, L, tr, graph=graph, hoist=hoist, hoist_sum=True).bind(dx, dp, dk, de)
            for _ in range(2 if graph else 1):
                ref.run()
                rp.run()
            for name in ("y", "z"):
                assert torch.equal(rp.result(name), ref.result(name)), (graph, hoist, name)
            rp.close()
            ref.close()
    sh = hml.Shard(ctx, L, 0, 1)
    with pytest.raises(hml.HmlError) as e:
        hml.Replay(ctx, L, trace, shard=sh, hoist=True, hoist_sum=True)
    assert e.value.code == 4                                      # HML_ERR_UNSUPPORTED
    sh.close()
    Oracle.set_threads(1)


def test_replay_hoist_sum_conditions():
    """Chains that do not qualify run as without the flag: a rotation output read again later, and an accumulator that is a
    rotation output.  A qualifying chain written as hadd(y, t, y) is fused."""
    N, ML, A, L = 4096, 5, 2, 4
    ctx = hml.Context(N=N, max_level=ML, alpha=A)
    beta = -(-L // A)
    x = ctx.uniform(list(range(L)), 1, lead=(2,))
    pts = {i: ctx.uniform(ctx.ext_mod_idx(L), 100 + i) for i in range(3)}
    keys = {r: ctx.uniform(ctx.ext_mod_idx(L), 200 + r, lead=(beta, 2)) for r in (1, 2, 3)}
    rot = [("hrotate", "r0", "x", 1), ("hrotate", "r1", "x", 2), ("hrotate", "r2", "x", 3)]
    chain = [("pmult", "y", "r2", 0), ("pmult", "m", "r0", 1), ("hadd", "y", "m", "y"), ("pmult", "m", "r1", 2), ("hadd", "y", "y", "m")]
    live = rot + chain + [("hadd", "w", "r1", "y")]
    own_acc = rot + [("pmult", "r0", "r0", 0), ("pmult", "m", "r1", 1), ("hadd", "r0", "r0", "m"), ("pmult", "m", "r2", 2),
                     ("hadd", "r0", "r0", "m")]
    for tr, names in ((live, ("y", "w")), (own_acc, ("r0",))):
        for hoist in (False, True):
            ref = hml.Replay(ctx, L, tr, hoist=hoist).bind(x, pts, keys, None)
            rp = hml.Replay(ctx, L, tr, hoist=hoist, hoist_sum=True).bind(x, pts, keys, None)
            ref.run()
            rp.run()
            for name in names:
                assert torch.equal(rp.result(name), ref.result(name)), (name, hoist)
            rp.close()
            ref.close()
    rp = hml.Replay(ctx, L, rot + chain, hoist_sum=True).bind(x, pts, keys, None)
    got = rp.run().result("y").clone()
    rp.close()
    want = ctx.hrotate_sum_hoisted(L, x, [keys[1], keys[2], keys[3]], [5, 25, 125], [pts[1], pts[2], pts[0]])
    assert torch.equal(got, want)
