"""GPU parity of the double-hoisted rotation sum and the lazily relinearised product sum on limb-sharded ciphertexts
(hml_hrotate_sum_hoisted_sharded / hml_group_hrotate_sum_hoisted, hml_hmult_sum_sharded / hml_group_hmult_sum).

On one GPU the ranks are emulated (a context per rank, one stream, separate signal / wait launches); the owned rows of every
rank must equal the one-GPU ops (hml_hrotate_sum_hoisted with pt_q_limbs = L, hml_hmult_sum with one output) bit for bit, and
at the small shapes the oracle definitions (tests/orc_rotsum.py, tests/orc_hmult_sum.py).  A world-1 shard runs the real fused
exchange, directly and as a captured CUDA graph.  With >= 2 GPUs the one-process-per-GPU path (tests/mp_sharded_sums.py) runs
as well."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import homulator_b200 as hml  # noqa: E402
from gpu_common import to_host  # noqa: E402
from homulator_b200.replay import shard_plaintexts  # noqa: E402
from orc import Oracle  # noqa: E402
from orc_hmult_sum import hmult_sum as orc_hmult_sum  # noqa: E402
from orc_rotsum import hrotate_sum_hoisted as orc_rotsum  # noqa: E402
from test_gpu_sharded_hoisted import NORTH_STAR, SHAPES  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def galois_elts(N, n):
    """n odd galois elements starting with 1, 2N - 1 and 5^7 (17 entries: two inner-product groups)"""
    g = [1, 2 * N - 1, pow(5, 7, 2 * N)] + [pow(5, r, 2 * N) for r in (1, 2, 3, 4, 5, 6, 8, 9, 10, 11, 12, 13, 14, 15)]
    return g[:n]


class Operands:
    """seeded device operands of one shape: ct, keys, extended-basis plaintexts, product terms, and the evaluation key"""

    def __init__(self, ctx, L, n_max=17):
        beta = ctx.beta(L)
        q, ext = list(range(L)), ctx.ext_mod_idx(L)
        self.ct = ctx.uniform(q, 1, lead=(2,))
        self.keys = [ctx.uniform(ext, 100 + i, lead=(beta, 2)) for i in range(n_max)]
        self.pts = [ctx.uniform(ext, 200 + i) for i in range(n_max)]
        self.a = [ctx.uniform(q, 300 + i, lead=(2,)) for i in range(n_max)]
        self.b = [ctx.uniform(q, 400 + i, lead=(2,)) for i in range(n_max)]
        self.evk = ctx.uniform(ext, 3, lead=(beta, 2))


def rows(t, idx, N):
    """rows idx of dim -2 of t (a one-limb zero placeholder when idx is empty), contiguous on t's device"""
    if not idx:
        return torch.zeros(t.shape[:-2] + (1, N), dtype=t.dtype, device=t.device)
    return t[..., idx, :].contiguous()


def own_rows(L, A, world):
    own = [list(range(r, L, world)) for r in range(world)]
    own_e = [[e for e in range(L + A) if e % world == r] for r in range(world)]
    keep = [[i for i in own[r] if i < L - 1] for r in range(world)]
    return own, own_e, keep


def owned_equal(outs, idx, want):
    """every rank's output rows equal rows idx[r] of the full result"""
    return all(torch.equal(outs[r][:, :len(i)], want[:, i]) for r, i in enumerate(idx) if i)


def shard_key(k, own_e):
    return k[:, :, own_e].contiguous() if own_e else None


@pytest.mark.parametrize("N,ML,L,A,world", SHAPES + NORTH_STAR)
def test_group_sums_emulated_ranks(N, ML, L, A, world):
    """both sums at n in {5, 17} rotations and {1, 4 with a square, 17} terms, each twice (epoch reuse), against the one-GPU ops
    (and the oracle at the small shapes); n_terms = 1 is hml_hmult_sharded.  Then the textbook sharded key switch, hrotate, hmult
    and rescale on the same group must still match: the sums keep the buffer reuse of later ops ordered."""
    ctxs = [hml.Context(N=N, max_level=ML, alpha=A) for _ in range(world)]
    ctx, R = ctxs[0], range(world)
    op = Operands(ctx, L)
    own, own_e, keep = own_rows(L, A, world)
    small = N <= 8192
    o = Oracle(N, 36, ML, A) if small else None
    group = hml.Shard.local_group(ctxs, L, max_rot=2)
    for sh in group:
        sh.prepare(L)
    ct_own = [rows(op.ct, own[r], N) for r in R]
    for n in (5, 17):
        gs = galois_elts(N, n)
        want = ctx.hrotate_sum_hoisted(L, op.ct, op.keys[:n], gs, op.pts[:n])
        if small:
            h = lambda ts: [to_host(t) for t in ts]  # noqa: E731
            assert np.array_equal(to_host(want), orc_rotsum(o, L, to_host(op.ct), h(op.keys[:n]), L, gs, h(op.pts[:n]), L)), n
        keys = [[shard_key(k, own_e[r]) for k in op.keys[:n]] for r in R]
        pts = [shard_plaintexts(sh, L, op.pts[:n]) for sh in group]
        for _ in range(2):
            outs = hml.group_hrotate_sum_hoisted(group, L, ct_own, keys, gs, pts)
            torch.cuda.synchronize()
            assert owned_equal(outs, own, want), ("rotation sum", n)
    evk_own = [shard_key(op.evk, own_e[r]) for r in R]
    for n, sq in ((1, None), (4, 2), (17, None)):
        a, b = op.a[:n], list(op.b[:n])
        if sq is not None:
            b[sq] = a[sq]
        want = ctx.hmult_sum(L, a, b, op.evk)
        if small:
            assert np.array_equal(to_host(want), orc_hmult_sum(o, L, [to_host(t) for t in a], [to_host(t) for t in b], to_host(op.evk), L)), n
        a_own = [[rows(t, own[r], N) for t in a] for r in R]
        b_own = [[a_own[r][k] if k == sq else rows(t, own[r], N) for k, t in enumerate(b)] for r in R]
        for _ in range(2):
            outs = hml.group_hmult_sum(group, L, a_own, b_own, evk_own)
            torch.cuda.synchronize()
            assert owned_equal(outs, keep, want), ("product sum", n)
        if n == 1:
            mul = [ctxs[r].empty(2, max(len(keep[r]), 1), N) for r in R]
            hml.group_op(group, "hmult", L, [x[0] for x in a_own], b=[x[0] for x in b_own], key=evk_own, out0=mul)
            assert all(torch.equal(mul[r][:, :len(k)], outs[r][:, :len(k)]) for r, k in enumerate(keep) if k)
    # the textbook sharded ops after the sums, against the one-GPU ops
    b_own = [rows(op.b[0], own[r], N) for r in R]
    nq = [max(len(own[r]), 1) for r in R]
    w0, w1 = ctx.keyswitch(L, op.ct[1].contiguous(), op.evk)
    o0, o1 = [ctxs[r].empty(nq[r], N) for r in R], [ctxs[r].empty(nq[r], N) for r in R]
    hml.group_op(group, "keyswitch", L, [x[1].contiguous() for x in ct_own], key=evk_own, out0=o0, out1=o1)
    assert owned_equal([x[None] for x in o0], own, w0[None]) and owned_equal([x[None] for x in o1], own, w1[None])
    rot = [ctxs[r].empty(2, nq[r], N) for r in R]
    hml.group_op(group, "hrotate", L, ct_own, key=evk_own, out0=rot, galois_elt=25)
    assert owned_equal(rot, own, ctx.hrotate(L, op.ct, op.evk, 25))
    mul = [ctxs[r].empty(2, max(len(keep[r]), 1), N) for r in R]
    hml.group_op(group, "hmult", L, ct_own, b=b_own, key=evk_own, out0=mul)
    assert owned_equal(mul, keep, ctx.hmult(L, op.ct, op.b[0], op.evk))
    rs = [ctxs[r].empty(2, max(len(keep[r]), 1), N) for r in R]
    hml.group_op(group, "rescale", L, b_own, out0=rs)
    assert owned_equal(rs, keep, torch.stack([ctx.rescale(L, op.b[0][0].contiguous()), ctx.rescale(L, op.b[0][1].contiguous())]))
    for sh in group:
        sh.check()
        sh.close()


def test_sharded_sums_work_is_shared():
    """Executed counts per rank on a two-pass ring.  The rotation sum runs the transforms and conversions of one hoisted sharded
    rotation whatever n; its launches, exchanges included, do not grow from 2 to 6 rotations and grow by one inner-product launch
    from 16 to 17.  The product sum runs hml_hmult_sharded's transforms and conversions whatever n_terms."""
    N, ML, L, A, world = 8192, 9, 8, 3, 2
    ctxs = [hml.Context(N=N, max_level=ML, alpha=A) for _ in range(world)]
    R = range(world)
    op = Operands(ctxs[0], L)
    own, own_e, keep = own_rows(L, A, world)
    group = hml.Shard.local_group(ctxs, L, max_rot=4)
    for sh in group:
        sh.prepare(L)
    ct_own = [rows(op.ct, own[r], N) for r in R]
    keys = [[shard_key(k, own_e[r]) for k in op.keys] for r in R]
    pts = [shard_plaintexts(sh, L, op.pts) for sh in group]
    evk_own = [shard_key(op.evk, own_e[r]) for r in R]
    gs = [pow(5, r, 2 * N) for r in range(1, 18)]

    def counted(fn):
        fn()  # warm: plans and tables exist
        for c in ctxs:
            c.exec_counts(reset=True)
        fn()
        torch.cuda.synchronize()
        return [c.exec_counts() for c in ctxs]

    work = ("ntt_limbs", "intt_limbs", "bconv_limb_macs")
    one = counted(lambda: hml.group_hrotate_hoisted(group, L, ct_own, [k[:1] for k in keys], gs[:1]))
    rot = {n: counted(lambda: hml.group_hrotate_sum_hoisted(group, L, ct_own, [k[:n] for k in keys], gs[:n], [p[:n] for p in pts]))
           for n in (2, 6, 16, 17)}
    for r in R:
        for n in (2, 6, 16, 17):
            assert all(rot[n][r][k] == one[r][k] for k in work), (r, n)
        assert rot[6][r]["kernel_launches"] == rot[2][r]["kernel_launches"]
        assert rot[17][r]["kernel_launches"] == rot[16][r]["kernel_launches"] + 1
    a_own = [[rows(t, own[r], N) for t in op.a] for r in R]
    b_own = [[rows(t, own[r], N) for t in op.b] for r in R]
    out = [ctxs[r].empty(2, max(len(keep[r]), 1), N) for r in R]
    mul = counted(lambda: hml.group_op(group, "hmult", L, [x[0] for x in a_own], b=[x[0] for x in b_own], key=evk_own, out0=out))
    for n in (1, 4, 17):
        got = counted(lambda: hml.group_hmult_sum(group, L, [x[:n] for x in a_own], [x[:n] for x in b_own], evk_own))
        for r in R:
            assert all(got[r][k] == mul[r][k] for k in work), (r, n)
    for sh in group:
        sh.check()
        sh.close()


def test_sharded_sums_rejections():
    """every invalid call raises before anything is enqueued: the group still works afterwards"""
    N, ML, L, A, world = 256, 7, 7, 3, 2
    ctxs = [hml.Context(N=N, max_level=ML, alpha=A) for _ in range(world)]
    R, c0 = range(world), ctxs[0]
    op = Operands(c0, L, n_max=2)
    own, own_e, keep = own_rows(L, A, world)
    group = hml.Shard.local_group(ctxs, L)
    for sh in group:
        sh.prepare(L)
    sh0, lib = group[0], c0.lib
    ct_own = [rows(op.ct, own[r], N) for r in R]
    keys = [[shard_key(k, own_e[r]) for k in op.keys] for r in R]
    pts = [shard_plaintexts(sh, L, op.pts) for sh in group]
    evk_own = [shard_key(op.evk, own_e[r]) for r in R]
    a_own = [[rows(t, own[r], N) for t in op.a] for r in R]
    b_own = [[rows(t, own[r], N) for t in op.b] for r in R]
    gs = [5, 25]
    bad_rot = [
        lambda: hml.group_hrotate_sum_hoisted(group, L, ct_own, [[] for _ in R], [], [[] for _ in R]),    # n_rot = 0
        lambda: hml.group_hrotate_sum_hoisted(group, L, [None, ct_own[1]], keys, gs, pts),                # null input
        lambda: hml.group_hrotate_sum_hoisted(group, L, ct_own, keys, gs, pts, outs=[None, c0.empty(2, 3, N)]),  # null output
        lambda: hml.group_hrotate_sum_hoisted(group, L, ct_own, [keys[0], [keys[1][0], None]], gs, pts),  # null key
        lambda: hml.group_hrotate_sum_hoisted(group, L, ct_own, keys, gs, [pts[0], [None, pts[1][1]]]),   # null plaintext
        lambda: hml.group_hrotate_sum_hoisted(group, L, ct_own, keys, [5, 6], pts),                       # even galois element
        lambda: hml.group_hrotate_sum_hoisted(group, L, ct_own, keys, gs, pts, outs=ct_own),              # output = input
        lambda: hml.group_hrotate_sum_hoisted(group, L + 1, ct_own, keys, gs, pts),                       # level above max
        lambda: c0._chk(lib.hml_hrotate_sum_hoisted_sharded(sh0.h, L, ct_own[0].data_ptr(), 2, (hml.api.C.c_void_p * 2)(
            *[k.data_ptr() for k in keys[0]]), None, (hml.api.C.c_void_p * 2)(*[p.data_ptr() for p in pts[0]]),
            c0.empty(2, 4, N).data_ptr(), None)),                                                        # null galois array
        lambda: sh0.hrotate_sum_hoisted(L, ct_own[0], keys[0], gs, pts[0], out=ct_own[0].view(-1)[N:].view(7, N)),  # overlap
    ]
    outs_alias = [a_own[r][1] for r in R]
    bad_mul = [
        lambda: hml.group_hmult_sum(group, L, [[] for _ in R], [[] for _ in R], evk_own),                 # n_terms = 0
        lambda: hml.group_hmult_sum(group, 1, [x[:1] for x in a_own], [x[:1] for x in b_own], evk_own),   # L < 2
        lambda: hml.group_hmult_sum(group, L + 1, a_own, b_own, evk_own),                                 # level above max
        lambda: hml.group_hmult_sum(group, L, [a_own[0], [a_own[1][0], None]], b_own, evk_own),           # null term
        lambda: hml.group_hmult_sum(group, L, a_own, b_own, [evk_own[0], None]),                          # null key
        lambda: hml.group_hmult_sum(group, L, a_own, b_own, evk_own, outs=[None, c0.empty(2, 3, N)]),     # null output
        lambda: hml.group_hmult_sum(group, L, a_own, b_own, evk_own, outs=outs_alias),                    # output = an input
        lambda: c0._chk(lib.hml_hmult_sum_sharded(sh0.h, L, 2, None, (hml.api.C.c_void_p * 2)(*[t.data_ptr() for t in b_own[0]]),
                                                  evk_own[0].data_ptr(), c0.empty(2, 3, N).data_ptr(), None)),   # null array
    ]
    for call in bad_rot + bad_mul:
        with pytest.raises(hml.HmlError):
            call()
    # a rank without Q-limbs still owns P-limbs: its key and plaintext are required (world 8, L 4: ranks 4..7 own P-limbs only)
    N8, ML8, L8, A8, w8 = 4096, 4, 4, 4, 8
    ctx8 = [hml.Context(N=N8, max_level=ML8, alpha=A8) for _ in range(w8)]
    op8 = Operands(ctx8[0], L8, n_max=1)
    own8, own_e8, _ = own_rows(L8, A8, w8)
    g8 = hml.Shard.local_group(ctx8, L8)
    for sh in g8:
        sh.prepare(L8)
    ct8 = [rows(op8.ct, own8[r], N8) for r in range(w8)]
    k8 = [[shard_key(op8.keys[0], own_e8[r])] for r in range(w8)]
    p8 = [shard_plaintexts(sh, L8, op8.pts[:1]) for sh in g8]
    for bad in ("key", "pt"):
        k, p = [list(x) for x in k8], [list(x) for x in p8]
        (k if bad == "key" else p)[5] = [None]
        with pytest.raises(hml.HmlError):
            hml.group_hrotate_sum_hoisted(g8, L8, ct8, k, [5], p)
    e8 = [shard_key(op8.evk, own_e8[r]) for r in range(w8)]
    e8[6] = None
    a8 = [[rows(op8.a[0], own8[r], N8)] for r in range(w8)]
    with pytest.raises(hml.HmlError):
        hml.group_hmult_sum(g8, L8, a8, a8, e8)
    # nothing was enqueued: both groups still work
    want = c0.hrotate_sum_hoisted(L, op.ct, op.keys, gs, op.pts)
    assert owned_equal(hml.group_hrotate_sum_hoisted(group, L, ct_own, keys, gs, pts), own, want)
    want = c0.hmult_sum(L, op.a, op.b, op.evk)
    assert owned_equal(hml.group_hmult_sum(group, L, a_own, b_own, evk_own), keep, want)
    want8 = ctx8[0].hrotate_sum_hoisted(L8, op8.ct, op8.keys[:1], [5], op8.pts[:1])
    assert owned_equal(hml.group_hrotate_sum_hoisted(g8, L8, ct8, k8, [5], p8), own8, want8)
    for sh in group + g8:
        sh.check()
        sh.close()


@pytest.mark.parametrize("N,ML,L,A", [(8192, 9, 8, 3), (65536, 45, 35, 15)])
def test_sums_over_a_one_rank_shard_and_in_a_graph(N, ML, L, A):
    """A world-1 shard runs the real fused exchange on one GPU: both ops directly, then captured once in a CUDA graph and
    replayed twice, must equal the one-GPU ops (capture fails if an op allocates or synchronises)."""
    ctx = hml.Context(N=N, max_level=ML, alpha=A)
    op = Operands(ctx, L)
    gs = galois_elts(N, 17)
    want_rot = ctx.hrotate_sum_hoisted(L, op.ct, op.keys, gs, op.pts)
    b = list(op.b)
    b[3] = op.a[3]
    want_mul = ctx.hmult_sum(L, op.a, b, op.evk)
    sh = hml.Shard(ctx, L, 0, 1, max_rot=4)
    sh.prepare(L)
    pts = shard_plaintexts(sh, L, op.pts)
    rot = sh.hrotate_sum_hoisted(L, op.ct, op.keys, gs, pts)
    mul = sh.hmult_sum(L, op.a, b, op.evk)
    torch.cuda.synchronize()
    assert torch.equal(rot, want_rot) and torch.equal(mul, want_mul)
    # warm on the capture stream: the context hands its workspace over between streams outside the capture
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        sh.hrotate_sum_hoisted(L, op.ct, op.keys, gs, pts, out=rot)
        sh.hmult_sum(L, op.a, b, op.evk, out=mul)
    torch.cuda.synchronize()
    rot.zero_()
    mul.zero_()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        sh.hrotate_sum_hoisted(L, op.ct, op.keys, gs, pts, out=rot)
        sh.hmult_sum(L, op.a, b, op.evk, out=mul)
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(rot, want_rot) and torch.equal(mul, want_mul)
        rot.zero_()
        mul.zero_()
    del g
    sh.check()
    sh.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_sharded_sums_over_nvlink():
    n = min(torch.cuda.device_count(), 8)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
           "--master-port", "29549", os.path.join(ROOT, "tests", "mp_sharded_sums.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "SHARDED_SUMS_OK" in r.stdout
