"""GPU parity of hoisted rotations on limb-sharded ciphertexts (hml_hrotate_hoisted_sharded / hml_group_hrotate_hoisted).

One ModUp of c1 serves every rotation of the op; groups of up to max_rot rotations share one inner-product launch, one P-limb
INTT and one exchange.  On one GPU the ranks are emulated (a context per rank, one stream, separate signal / wait launches);
the assembled owned rows must equal the oracle's hoisted definition and the single-GPU hoisted rotation bit for bit.  With >= 2
GPUs the one-process-per-GPU path (tests/mp_sharded_hoisted.py) runs as well."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import homulator_b200 as hml  # noqa: E402
from gpu_common import to_dev, to_host  # noqa: E402
from homulator_b200.replay import bsgs_trace, rotsum_trace, shard_operands  # noqa: E402
from orc import Oracle, uniform_limbs  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SHAPES = [(256, 7, 7, 3, 2), (256, 7, 7, 3, 3), (1024, 6, 5, 2, 4), (4096, 4, 4, 4, 8), (8192, 9, 8, 3, 2), (8192, 9, 9, 3, 8)]
NORTH_STAR = [(65536, 45, 35, 15, w) for w in (2, 4, 8)]


def galois_elts(N):
    return [5, 25, 2 * N - 1, 1, pow(5, 7, 2 * N)]


_CASES = {}


def oracle_case(N, ML, L, A):
    """seeded operands and every oracle result the parity test needs, computed once per shape for the whole module"""
    key = (N, ML, L, A)
    if key not in _CASES:
        o = Oracle(N, 36, ML, A)
        Oracle.set_threads(0)
        beta = -(-L // A)
        ct = uniform_limbs(o.moduli[:L], N, 3100 + L, lead=(2,))
        b = uniform_limbs(o.moduli[:L], N, 3101 + L, lead=(2,))
        gs = galois_elts(N)
        rks = [uniform_limbs(o.moduli[:L] + o.moduli[ML:], N, 3110 + i, lead=(beta, 2)) for i in range(len(gs))]
        want = o.hrotate_hoisted(L, ct, rks, L, gs)
        after = {"keyswitch": o.keyswitch(L, ct[1], rks[0], L), "hrotate": o.hrotate(L, ct, rks[0], L, 25),
                 "hmult": o.hmult(L, ct, b, rks[0], L), "rescale": np.stack([o.rescale(L, b[0]), o.rescale(L, b[1])])}
        Oracle.set_threads(1)
        _CASES[key] = (o, ct, b, rks, gs, want, after)
    return _CASES[key]


def split(L, A, world, a, keys):
    """every rank's owned rows of a ciphertext-like array [.., L, N] (a 1-limb zero placeholder where it owns none) and of
    each key [beta][2][E][N] (None where the rank owns no extended limb)"""
    N = a.shape[-1]
    own = [list(range(r, L, world)) for r in range(world)]
    own_e = [[e for e in range(L + A) if e % world == r] for r in range(world)]
    a_own = [to_dev(a[..., own[r], :]) if own[r] else to_dev(np.zeros(a.shape[:-2] + (1, N), dtype=np.uint64)) for r in range(world)]
    k_own = [[to_dev(k[:, :, own_e[r]]) if own_e[r] else None for k in keys] for r in range(world)]
    return own, a_own, k_own


def assemble(outs, idx, shape):
    got = np.zeros(shape, dtype=np.uint64)
    for r, rows in enumerate(idx):
        if rows:
            got[..., rows, :] = to_host(outs[r])[..., :len(rows), :]
    return got


@pytest.mark.parametrize("N,ML,L,A,world", SHAPES + NORTH_STAR)
def test_group_hoisted_rotations_emulated_ranks(N, ML, L, A, world):
    """group_hrotate_hoisted against orc_hrotate_hoisted and the single-GPU hoisted rotation, with several groups per op
    (max_rot = 2: the extra exchange before a later group rewrites gather buffer 2) and with one group (max_rot = n_rot); each
    twice (epoch reuse).  Then the textbook sharded ops on the same group must still match the oracle: the new exchanges keep
    the buffer reuse of later ops ordered."""
    o, ct, b, rks, gs, want, after = oracle_case(N, ML, L, A)
    ctxs = [hml.Context(N=N, max_level=ML, alpha=A) for _ in range(world)]
    single = ctxs[0].hrotate_hoisted(L, to_dev(ct), [to_dev(k) for k in rks], gs)
    for w, s in zip(want, single):
        assert np.array_equal(to_host(s), w)
    del single
    R = range(world)
    own, ct_own, k_own = split(L, A, world, ct, rks)
    _, b_own, _ = split(L, A, world, b, [])
    keep = [[i for i in own[r] if i < L - 1] for r in R]
    for max_rot in (2, len(gs)):
        group = hml.Shard.local_group(ctxs, L, max_rot=max_rot)
        for sh in group:
            sh.prepare(L)
        for _ in range(2):
            outs = hml.group_hrotate_hoisted(group, L, ct_own, k_own, gs)
            for i, w in enumerate(want):
                assert np.array_equal(assemble([outs[r][i] for r in R], own, (2, L, N)), w), (max_rot, i)
        evk_own = [k[0] for k in k_own]
        nq = [max(len(own[r]), 1) for r in R]
        o0, o1 = [ctxs[r].empty(nq[r], N) for r in R], [ctxs[r].empty(nq[r], N) for r in R]
        hml.group_op(group, "keyswitch", L, [x[1].contiguous() for x in ct_own], key=evk_own, out0=o0, out1=o1)
        assert np.array_equal(assemble(o0, own, (L, N)), after["keyswitch"][0]) and np.array_equal(assemble(o1, own, (L, N)), after["keyswitch"][1])
        rot = [ctxs[r].empty(2, nq[r], N) for r in R]
        hml.group_op(group, "hrotate", L, ct_own, key=evk_own, out0=rot, galois_elt=25)
        assert np.array_equal(assemble(rot, own, (2, L, N)), after["hrotate"])
        mul = [ctxs[r].empty(2, max(len(keep[r]), 1), N) for r in R]
        hml.group_op(group, "hmult", L, ct_own, b=b_own, key=evk_own, out0=mul)
        assert np.array_equal(assemble(mul, keep, (2, L - 1, N)), after["hmult"])
        rs = [ctxs[r].empty(2, max(len(keep[r]), 1), N) for r in R]
        hml.group_op(group, "rescale", L, b_own, out0=rs)
        assert np.array_equal(assemble(rs, keep, (2, L - 1, N)), after["rescale"])
        # a hoisted op straight after a rescale, then a rescale again (rescale buffer ordering across the new op)
        outs = hml.group_hrotate_hoisted(group, L, ct_own, [k[:3] for k in k_own], gs[:3])
        for i in range(3):
            assert np.array_equal(assemble([outs[r][i] for r in R], own, (2, L, N)), want[i])
        hml.group_op(group, "rescale", L, b_own, out0=rs)
        assert np.array_equal(assemble(rs, keep, (2, L - 1, N)), after["rescale"])
        for sh in group:
            sh.check()
            sh.close()


def test_hoisted_work_is_shared():
    """Executed counts of n_rot = 2 against n_rot = 6 in ONE group on a two-pass ring: every extra rotation adds only its
    ModDown (one base conversion of the alpha P-limbs to the owned Q-limbs for both accumulators, and its forward NTT with the
    fused epilogue: 3 launches); the ModUp, the inner product, the P-limb INTT and the exchanges are shared."""
    N, ML, L, A, world = 8192, 9, 8, 3, 2
    beta = -(-L // A)
    o = Oracle(N, 36, ML, A)
    ct = uniform_limbs(o.moduli[:L], N, 3300, lead=(2,))
    gs = [pow(5, r, 2 * N) for r in range(1, 7)]
    rks = [uniform_limbs(o.moduli[:L] + o.moduli[ML:], N, 3310 + i, lead=(beta, 2)) for i in range(6)]
    ctxs = [hml.Context(N=N, max_level=ML, alpha=A) for _ in range(world)]
    group = hml.Shard.local_group(ctxs, L, max_rot=6)
    for sh in group:
        sh.prepare(L)
    own, ct_own, k_own = split(L, A, world, ct, rks)
    counts = {}
    for n in (2, 6):
        hml.group_hrotate_hoisted(group, L, ct_own, [k[:n] for k in k_own], gs[:n])  # warm: plans and tables exist
        for c in ctxs:
            c.exec_counts(reset=True)
        hml.group_hrotate_hoisted(group, L, ct_own, [k[:n] for k in k_own], gs[:n])
        torch.cuda.synchronize()
        counts[n] = [c.exec_counts() for c in ctxs]
    for r in range(world):
        nq, np_ = len(own[r]), len([j for j in range(A) if (L + j) % world == r])
        c2, c6 = counts[2][r], counts[6][r]
        assert c6["bconv_limb_macs"] - c2["bconv_limb_macs"] == 4 * 2 * A * nq
        assert c6["ntt_limbs"] - c2["ntt_limbs"] == 4 * 2 * nq
        assert c6["intt_limbs"] - c2["intt_limbs"] == 4 * 2 * np_   # the P-limb INTT grows, inside its one launch
        # 3 launches per extra rotation and not one more: the exchange launches (signal + wait) do not grow either
        assert c6["kernel_launches"] - c2["kernel_launches"] == 4 * 3
    for sh in group:
        sh.check()
        sh.close()


def test_hoisted_sharded_rejections():
    N, ML, L, A, world = 256, 7, 7, 3, 2
    beta = -(-L // A)
    o = Oracle(N, 36, ML, A)
    ct = uniform_limbs(o.moduli[:L], N, 3400, lead=(2,))
    rk = uniform_limbs(o.moduli[:L] + o.moduli[ML:], N, 3401, lead=(beta, 2))
    ctxs = [hml.Context(N=N, max_level=ML, alpha=A) for _ in range(world)]
    for bad in (0, 17):
        with pytest.raises(hml.HmlError):
            hml.Shard(ctxs[0], L, 0, world, max_rot=bad)
    mixed = [hml.Shard(ctxs[0], L, 0, world, max_rot=2), hml.Shard(ctxs[1], L, 1, world, max_rot=3)]
    arr = (hml.api.C.c_void_p * world)(*[g.h for g in mixed])
    assert ctxs[0].lib.hml_shard_connect_local(arr, world) != 0
    for sh in mixed:
        sh.close()
    group = hml.Shard.local_group(ctxs, L, max_rot=2)
    for sh in group:
        sh.prepare(L)
    own, ct_own, k_own = split(L, A, world, ct, [rk, rk])
    gs = [5, 25]
    # n_rot = 0 is a no-op, even with nothing to work on
    assert hml.group_hrotate_hoisted(group, L, ct_own, [[] for _ in group], []) == [[] for _ in group]
    sh0, c0 = group[0], ctxs[0]
    assert c0.lib.hml_hrotate_hoisted_sharded(sh0.h, L, None, 0, None, None, None, None) == 0
    with pytest.raises(hml.HmlError):  # null input
        hml.group_hrotate_hoisted(group, L, [None, ct_own[1]], k_own, gs)
    with pytest.raises(hml.HmlError):  # null output
        po = (hml.api.C.c_void_p * 2)(None, None)
        keys = (hml.api.C.c_void_p * 2)(*[k.data_ptr() for k in k_own[0]])
        g = (hml.api.C.c_uint64 * 2)(*gs)
        c0._chk(c0.lib.hml_hrotate_hoisted_sharded(sh0.h, L, ct_own[0].data_ptr(), 2, keys, g, po, None))
    with pytest.raises(hml.HmlError):  # an output aliasing the input
        sh0.hrotate_hoisted(L, ct_own[0], k_own[0], gs, outs=[ct_own[0], c0.empty(*ct_own[0].shape)])
    with pytest.raises(hml.HmlError):  # even galois element
        hml.group_hrotate_hoisted(group, L, ct_own, k_own, [5, 6])
    with pytest.raises(hml.HmlError):  # level above the shard's maximum
        hml.group_hrotate_hoisted(group, L + 1, ct_own, k_own, gs)
    with pytest.raises(hml.HmlError):  # null key on a rank that owns extended limbs
        hml.group_hrotate_hoisted(group, L, ct_own, [k_own[0], [k_own[1][0], None]], gs)
    # a rank without Q-limbs still owns P-limbs: its key is required too (world 8, L 4: ranks 4..7 own P-limbs only)
    N8, ML8, L8, A8, w8 = 4096, 4, 4, 4, 8
    o8 = Oracle(N8, 36, ML8, A8)
    ct8 = uniform_limbs(o8.moduli[:L8], N8, 3402, lead=(2,))
    rk8 = uniform_limbs(o8.moduli[:L8] + o8.moduli[ML8:], N8, 3403, lead=(1, 2))
    ctx8 = [hml.Context(N=N8, max_level=ML8, alpha=A8) for _ in range(w8)]
    g8 = hml.Shard.local_group(ctx8, L8)
    for sh in g8:
        sh.prepare(L8)
    _, ct8_own, k8_own = split(L8, A8, w8, ct8, [rk8])
    k8_bad = [list(k) for k in k8_own]
    k8_bad[5] = [None]
    with pytest.raises(hml.HmlError):
        hml.group_hrotate_hoisted(g8, L8, ct8_own, k8_bad, [5])
    # the rejected calls enqueued nothing: the groups still work
    outs = hml.group_hrotate_hoisted(group, L, ct_own, k_own, gs)
    want = o.hrotate_hoisted(L, ct, [rk, rk], L, gs)
    for i in range(2):
        assert np.array_equal(assemble([outs[r][i] for r in range(world)], own, (2, L, N)), want[i])
    for sh in group + g8:
        sh.check()
        sh.close()


@pytest.mark.parametrize("N,ML,L,A", [(8192, 9, 8, 3), (65536, 45, 35, 15)])
def test_hoisted_replay_over_a_one_rank_shard(N, ML, L, A):
    """A world-1 shard runs the real fused exchange on one GPU.  rotsum_trace(6) and bsgs_trace(4, 4) with hoisted rotations,
    as launches and as a graph, must equal the unsharded hoisted replay bit for bit (tests/test_gpu_ops.py ties that one to the
    oracle)."""
    ctx = hml.Context(N=N, max_level=ML, alpha=A)
    beta = -(-L // A)
    q = list(range(L))
    x = ctx.uniform(q, 1, lead=(2,))
    evk = ctx.uniform(ctx.ext_mod_idx(L), 3, lead=(beta, 2))
    pts = {i: ctx.uniform(q, 200 + i) for i in range(16)}
    for tr in (rotsum_trace(6), bsgs_trace(4, 4)):
        rots = sorted({op[3] for op in tr if op[0] == "hrotate"})
        keys = {r: ctx.uniform(ctx.ext_mod_idx(L), 100 + r, lead=(beta, 2)) for r in rots}
        one = hml.Replay(ctx, L, tr, hoist=True).bind(x, pts, keys, evk)
        ref = one.run().result("z").clone()
        for max_rot in (1, 4):
            sh = hml.Shard(ctx, L, 0, 1, max_rot=max_rot)
            sh.prepare(L)
            x_own, pts_own, keys_own, evk_own = shard_operands(sh, L, x, pts, keys, evk)
            for graph in (False, True):
                rp = hml.Replay(ctx, L, tr, shard=sh, graph=graph, hoist=True).bind(x_own, pts_own, keys_own, evk_own)
                for _ in range(2):
                    got = rp.run().result("z")
                    torch.cuda.synchronize()
                    assert torch.equal(got, ref), (len(tr), max_rot, graph)
                rp.close()
            sh.check()
            sh.close()
        one.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_hoisted_sharded_over_nvlink():
    n = min(torch.cuda.device_count(), 8)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
           "--master-port", "29547", os.path.join(ROOT, "tests", "mp_sharded_hoisted.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "SHARDED_HOISTED_OK" in r.stdout
