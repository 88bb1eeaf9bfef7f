"""Bit-exact parity checks shared by the element-width and extreme-residue tests: every op of the library on given operands
against the scalar oracle (tests/orc.py) and the oracle definitions of the hoisted and summed ops (tests/orc_*.py).  Every
check runs the word key and its packed copy (hml_key_pack) where the op takes a key."""
import numpy as np
import torch

import homulator_b200 as hml
from gpu_common import to_dev, to_host
from orc_bsgs import hrotate_bsgs_hoisted
from orc_hmult_sum import hmult_sum
from orc_rotsum import hrotate_sum_hoisted


def key_variants(ctx, evk, evk_q):
    """(device key, evk_q_limbs argument) for the word key and its packed copy"""
    K = to_dev(evk)
    return [(K, evk_q), (ctx.key_pack(K), evk_q | hml.KEY_PACKED)]


def eq(got, want, what):
    got = to_host(got) if isinstance(got, torch.Tensor) else got
    assert got.shape == want.shape and np.array_equal(got, want), what


def check_core(ctx, o, L, a, b, evk, evk_q, g=5):
    """keyswitch of b1, rescale of a0 and b1, hmult(a, b) (L >= 2) and hrotate(a, g) at level L; returns the oracle's hmult and
    hrotate results for the batched checks"""
    w0, w1 = o.keyswitch(L, np.ascontiguousarray(b[1]), evk, evk_q)
    want_m = o.hmult(L, a, b, evk, evk_q) if L >= 2 else None
    want_r = o.hrotate(L, a, evk, evk_q, g)
    if L >= 2:
        for x in (a[0], b[1]):
            eq(ctx.rescale(L, to_dev(x)), o.rescale(L, np.ascontiguousarray(x)), ("rescale", L))
    for K, kq in key_variants(ctx, evk, evk_q):
        g0, g1 = ctx.keyswitch(L, to_dev(b[1]), K, kq)
        eq(g0, w0, ("keyswitch 0", L, kq))
        eq(g1, w1, ("keyswitch 1", L, kq))
        if L >= 2:
            eq(ctx.hmult(L, to_dev(a), to_dev(b), K, evk_q_limbs=kq), want_m, ("hmult", L, kq))
        eq(ctx.hrotate(L, to_dev(a), K, g, evk_q_limbs=kq), want_r, ("hrotate", L, kq, g))
    return want_m, want_r


def check_batched(ctx, o, L, a, b, evk, evk_q, want_m, want_r, g=5):
    """hmult_batch of (a, b), (b, a), (a, b) (the tensor product is symmetric: every entry is hmult(a, b)) and hrotate_batch of
    (a, b), stand-alone inner product over several ciphertexts, word and packed keys.  want_m / want_r are the oracle's
    hmult(a, b) and hrotate(a, g) for the same g (check_core's results)."""
    want_rb = o.hrotate(L, b, evk, evk_q, g)
    A, B = torch.stack([to_dev(a), to_dev(b), to_dev(a)]), torch.stack([to_dev(b), to_dev(a), to_dev(b)])
    for K, kq in key_variants(ctx, evk, evk_q):
        got = to_host(ctx.hmult_batch(L, A, B, K, evk_q_limbs=kq))
        for i in range(3):
            eq(got[i], want_m, ("hmult_batch", L, kq, i))
        rot = to_host(ctx.hrotate_batch(L, A[:2].contiguous(), K, g, evk_q_limbs=kq))
        eq(rot[0], want_r, ("hrotate_batch", L, kq, 0))
        eq(rot[1], want_rb, ("hrotate_batch", L, kq, 1))


def check_hoisted(ctx, o, L, ct, keys, evk_q, gs):
    """hrotate_hoisted of ct under galois elements gs (keys[i] for gs[i]) against the oracle's hoisted definition"""
    want = o.hrotate_hoisted(L, ct, keys, evk_q, gs)
    dk = [key_variants(ctx, k, evk_q) for k in keys]
    for v in range(2):
        got = ctx.hrotate_hoisted(L, to_dev(ct), [d[v][0] for d in dk], gs, evk_q_limbs=dk[0][v][1])
        for i, (x, w) in enumerate(zip(got, want)):
            eq(x, w, ("hrotate_hoisted", L, v, i))


def check_rotsum(ctx, o, L, ct, keys, evk_q, gs, pts, pt_q):
    """hrotate_sum_hoisted: sum_i pts[i] * rotate(ct, gs[i]) against tests/orc_rotsum.py"""
    want = hrotate_sum_hoisted(o, L, ct, keys, evk_q, gs, pts, pt_q)
    dk = [key_variants(ctx, k, evk_q) for k in keys]
    dp = [to_dev(p) for p in pts]
    for v in range(2):
        got = ctx.hrotate_sum_hoisted(L, to_dev(ct), [d[v][0] for d in dk], gs, dp, evk_q_limbs=dk[0][v][1], pt_q_limbs=pt_q)
        eq(got, want, ("hrotate_sum_hoisted", L, len(gs), v))


def check_bsgs(ctx, o, L, ct, babies, giants, keys, evk_q, pts, pt_q):
    """hrotate_bsgs_hoisted against tests/orc_bsgs.py; keys maps every galois element to its key (None for the identity)"""
    want = hrotate_bsgs_hoisted(o, L, ct, babies, [keys[g] for g in babies], giants, [keys[g] for g in giants], evk_q, pts, pt_q)
    dk = {g: None if k is None else key_variants(ctx, k, evk_q) for g, k in keys.items()}
    dp = {id(p): to_dev(p) for row in pts for p in row}
    for v in range(2):
        pick = {g: None if d is None else d[v][0] for g, d in dk.items()}
        got = ctx.hrotate_bsgs_hoisted(L, to_dev(ct), babies, [pick[g] for g in babies], giants, [pick[g] for g in giants],
                                       [[dp[id(p)] for p in row] for row in pts], evk_q_limbs=evk_q | (hml.KEY_PACKED if v else 0),
                                       pt_q_limbs=pt_q)
        eq(got, want, ("hrotate_bsgs_hoisted", L, len(babies), len(giants), v))


def check_hmult_sum(ctx, o, L, cts_a, cts_b, evk, evk_q):
    """hmult_sum of the terms cts_a[i] * cts_b[i] (the same array twice is a square) against tests/orc_hmult_sum.py"""
    want = hmult_sum(o, L, cts_a, cts_b, evk, evk_q)
    dev = {}
    for x in list(cts_a) + list(cts_b):
        dev.setdefault(id(x), to_dev(x))
    for K, kq in key_variants(ctx, evk, evk_q):
        got = ctx.hmult_sum(L, [dev[id(x)] for x in cts_a], [dev[id(x)] for x in cts_b], K, evk_q_limbs=kq)
        eq(got, want, ("hmult_sum", L, len(cts_a), kq))
