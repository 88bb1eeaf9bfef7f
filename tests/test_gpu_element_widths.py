"""GPU parity at every element width the library accepts below the shipped 36 bits: 20, 24, 28, 32, 33 and 35-bit moduli.

At 36 bits every modulus lies within 0.5 % of 2^36.  At 20-28 bits the moduli of one context spread over 25 % or more, every
residue fits in 32 bits (the high byte of a packed limb is zero), and at 33 and 35 bits bit 32 is set while the fifth byte is
not full.  Each shape below names the dispatch path it selects; every result is compared bit for bit with the scalar oracle at
the same width (or with a one-GPU op that is)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import homulator_b200 as hml  # noqa: E402
from gpu_common import to_dev, to_host  # noqa: E402
from orc import Oracle, uniform_limbs  # noqa: E402
from parity_checks import (check_batched, check_bsgs, check_core, check_hmult_sum, check_hoisted, check_rotsum,  # noqa: E402
                           eq)

# (width, N, maxLevel, alpha, ((L, evk_q_limbs), ...)).  beta = ceil(L / alpha) picks the inner product's digit bound NB in
# {1, 2, 3, 4, 8} (ewe.cu with_max_beta); two-pass rings with beta >= 2 run the HPIP-fused inner product (context.cu
# ks_uses_hpip: logN > NTT_SMALL_LOG && beta >= 2 && one ciphertext), the others k_inner.  Conversions with <= 48 sources and
# targets on N >= 128 run on tcgen05 (ewe.cu launch_bconv: an image exists, bconv_umma.cu bconv_image_shape), larger ones
# on the DMMA kernel.
SHAPES = [
    # single-pass ring (logN 11 <= NTT_SMALL_LOG, ntt.cuh); beta 3 / 2 / 1; tcgen05 conversions; key laid out for maxLevel
    (20, 2048, 12, 4, ((12, 12), (5, 12), (3, 3))),
    # two-pass ring (logN 13 > NTT_SMALL_LOG); beta 2 -> HPIP, beta 1 -> k_inner
    (20, 8192, 3, 2, ((3, 3), (2, 3))),
    # DMMA conversion: L = 70 has 60 + 10 = 70 ModUp targets and 70 ModDown targets (> 48, no tcgen05 image); beta 7 -> NB 8;
    # L = 40: 40 targets, tcgen05 again, beta 4
    (20, 256, 70, 10, ((70, 70), (40, 70))),
    # two-pass ring, HPIP with beta 4 and 3
    (24, 8192, 40, 10, ((40, 40), (23, 40))),
    # hmult's merged ModDown + Rescale with 48 targets plus the fold (bconv_image_shape: NP > 256, no tcgen05 image) and ModUp
    # digit 0 with 49 targets: the DMMA kernel on a two-pass ring, fold pre-pass included; beta 7 (NB 8, HPIP)
    (24, 8192, 49, 7, ((49, 49),)),
    # N = 2^16 at 24 bits: beta 2 (HPIP) and 1
    (24, 65536, 8, 4, ((8, 8), (3, 8))),
    # single-pass ring with beta 8 and 5 (NB 8, padding digits) and 3
    (24, 4096, 16, 2, ((16, 16), (10, 16), (6, 6))),
    # the north-star shape at 28 bits: beta 3 (HPIP, 15-source conversions on tcgen05), beta 2 with a maxLevel key, beta 1
    (28, 65536, 45, 15, ((35, 35), (20, 45), (12, 12))),
    # alpha 5: beta 8 (NB 8, HPIP) and 4
    (28, 65536, 45, 5, ((40, 40), (20, 45))),
    (28, 4096, 16, 2, ((16, 16), (9, 16))),
    # widths above 32 bits (bit 32 set, fifth byte not full): the north-star shape at one level, and single-pass beta 8 / 5
    (32, 65536, 45, 15, ((35, 35),)),
    (32, 4096, 16, 2, ((16, 16), (10, 16), (4, 4))),
    (33, 65536, 45, 15, ((35, 35),)),
    (33, 4096, 16, 2, ((16, 16), (10, 16), (4, 4))),
    (35, 65536, 45, 15, ((35, 35),)),
    (35, 4096, 16, 2, ((16, 16), (10, 16), (4, 4))),
]


@pytest.fixture(scope="module", autouse=True)
def threaded_oracle():
    Oracle.set_threads(0)  # all host cores for the checker; results do not depend on it (tests/test_oracle.py)
    yield
    Oracle.set_threads(1)


def _ctx(w, N, ML, A):
    return hml.Context(N=N, max_level=ML, alpha=A, element_bit_width=w), Oracle(N, w, ML, A)


def _case(o, L, evk_q, seed):
    beta = -(-L // o.alpha)
    a = uniform_limbs(o.moduli[:L], o.N, seed, lead=(2,))
    b = uniform_limbs(o.moduli[:L], o.N, seed + 1, lead=(2,))
    evk = uniform_limbs(o.moduli[:evk_q] + o.moduli[o.max_level:], o.N, seed + 2, lead=(beta, 2))
    return a, b, evk


def _check_primitives(ctx, o, L):
    """ntt / intt / ntt_batch over every modulus, ewe, automorph, bconv and bconv_batch in the ModUp digit-0 and ModDown shapes of
    level L; canonical edges q - 1 and 0 in every limb"""
    N, ML, A = o.N, o.max_level, o.alpha
    idx = list(range(ML + A))
    x = uniform_limbs(o.moduli, N, 31)
    x[:, :2] = np.array(o.moduli, dtype=np.uint64)[:, None] - np.uint64(1)
    x[:, 2] = 0
    want = np.stack([o.ntt(i, x[i]) for i in idx])
    eq(ctx.ntt(to_dev(x), idx), want, "ntt")
    eq(ctx.intt(to_dev(want), idx), x, "ntt round trip")
    eq(ctx.intt(to_dev(x), idx), np.stack([o.intt(i, x[i]) for i in idx]), "intt")
    sub = [0, ML - 1, ML + A - 1]
    xb = np.stack([x[sub], want[sub]])
    eq(ctx.ntt_batch(to_dev(xb), sub), np.stack([np.stack([o.ntt(i, xb[k][r]) for r, i in enumerate(sub)]) for k in range(2)]), "ntt_batch")
    ys = [np.ascontiguousarray(y) for y in (x[sub], want[sub], x[sub][:, ::-1], want[sub][:, ::-1])]
    for sel, neg in (((0, 1, 2, 3), True), ((0, 1, 2, None), False), ((0, None, 2, None), True)):
        got = to_host(ctx.ewe(*[to_dev(ys[s]) if s is not None else None for s in sel], sub, subtract=neg))
        for r, i in enumerate(sub):
            eq(got[r], o.ewe(i, *[np.ascontiguousarray(ys[s][r]) if s is not None else None for s in sel], sub=neg), ("ewe", sel, i))
    for g in (5, 2 * N - 1):
        got = to_host(ctx.automorph(to_dev(x[sub]), g))
        for r, i in enumerate(sub):
            eq(got[r], o.automorph_eval(g, x[i]), ("automorph", g, i))
    digit0 = list(range(min(A, L)))
    up = (digit0, [i for i in range(L) if i not in digit0] + list(range(ML, ML + A)))
    down = (list(range(ML, ML + A)), list(range(L)))
    for src, dst in (up, down):
        if not dst:
            continue
        xs = np.stack([np.stack([x[i] if k == 0 else want[i] for i in src]) for k in range(2)])
        got = to_host(ctx.bconv_batch(to_dev(xs), src, dst))
        one = to_host(ctx.bconv(to_dev(xs[1]), src, dst))
        check = range(len(dst)) if N <= 4096 else (0, len(dst) // 2, len(dst) - 1)
        for t in check:
            for k in range(2):
                eq(got[k, t], o.bconv(src, dst[t], xs[k]), ("bconv_batch", len(src), dst[t], k))
            eq(one[t], o.bconv(src, dst[t], xs[1]), ("bconv", len(src), dst[t]))


@pytest.mark.parametrize("w,N,ML,A,levels", SHAPES, ids=lambda v: str(v) if not isinstance(v, tuple) else "L" + "_".join(str(l[0]) for l in v))
def test_widths_match_oracle(w, N, ML, A, levels):
    """moduli and roots, the primitives, and keyswitch / rescale / hmult / hrotate (word and packed keys) at every level of the
    shape; the batched ops (k_inner over several ciphertexts, the chunked tensor product) at the first level"""
    ctx, o = _ctx(w, N, ML, A)
    assert ctx.moduli == o.moduli and ctx.psi == o.psi
    assert all(q < (1 << w) for q in o.moduli) and max(o.moduli) >= 1 << (w - 1)
    _check_primitives(ctx, o, levels[0][0])
    for k, (L, evk_q) in enumerate(levels):
        a, b, evk = _case(o, L, evk_q, 100 * w + 7 * k)
        want_m, want_r = check_core(ctx, o, L, a, b, evk, evk_q, g=5 if k % 2 == 0 else 2 * N - 1)
        if k == 0:
            check_batched(ctx, o, L, a, b, evk, evk_q, want_m, want_r)
    ctx.close()


# one shape per width for the hoisted and summed ops: (N, maxLevel, alpha, L)
SUM_SHAPES = {20: (8192, 3, 2, 3),      # two-pass, beta 2
              24: (8192, 12, 4, 11),    # two-pass, beta 3, short last digit
              28: (4096, 16, 2, 9),     # single-pass, beta 5 (NB 8)
              32: (8192, 9, 3, 8),      # two-pass, beta 3
              33: (2048, 12, 4, 12),    # single-pass, beta 3
              35: (8192, 6, 2, 5)}      # two-pass, beta 3


@pytest.mark.parametrize("w", sorted(SUM_SHAPES))
def test_hoisted_and_summed_ops(w):
    """hrotate_hoisted, hrotate_sum_hoisted (17 rotations: a full group of 16 and an accumulating one), hrotate_bsgs_hoisted
    (identity baby and giant steps) and hmult_sum (17 terms, squares and products) against the oracle definitions"""
    N, ML, A, L = SUM_SHAPES[w]
    ctx, o = _ctx(w, N, ML, A)
    beta = -(-L // A)
    ct = uniform_limbs(o.moduli[:L], N, 40 + w, lead=(2,))
    keys = [uniform_limbs(o.moduli[:ML] + o.moduli[ML:], N, 50 + w + k, lead=(beta, 2)) for k in range(3)]
    gs = [pow(5, r, 2 * N) for r in range(1, 18)]
    check_hoisted(ctx, o, L, ct, keys, ML, [gs[0], gs[3], 2 * N - 1])
    pts = [uniform_limbs(o.moduli[:L] + o.moduli[ML:], N, 60 + w + k) for k in range(5)]
    check_rotsum(ctx, o, L, ct, [keys[i % 3] for i in range(17)], ML, gs, [pts[i % 5] for i in range(17)], L)
    babies, giants = [1, 5, 25], [1, pow(5, 3, 2 * N), 2 * N - 1]
    bk = {1: None, 5: keys[0], 25: keys[1], pow(5, 3, 2 * N): keys[2], 2 * N - 1: keys[0]}
    check_bsgs(ctx, o, L, ct, babies, giants, bk, ML, [[pts[(j + i) % 5] for i in range(3)] for j in range(3)], L)
    cts = [uniform_limbs(o.moduli[:L], N, 70 + w + k, lead=(2,)) for k in range(4)]
    check_hmult_sum(ctx, o, L, [cts[i % 4] for i in range(17)], [cts[(i * 3) % 4] for i in range(17)], keys[0], ML)
    ctx.close()


def test_hmult_batch_more_than_one_chunk():
    """65 ciphertexts at 20 bits: one full chunk of 64 and a partial one (context.cu: batches run in chunks of 64)"""
    N, ML, A, L, n = 2048, 12, 4, 5, 65
    ctx, o = _ctx(20, N, ML, A)
    a, b, evk = _case(o, L, L, 900)
    pool = [uniform_limbs(o.moduli[:L], N, 910 + k, lead=(2,)) for k in range(3)]
    As = torch.stack([to_dev(pool[i % 3]) for i in range(n)])
    Bs = torch.stack([to_dev(pool[(i + 1) % 3]) for i in range(n)])
    K = to_dev(evk)
    got = to_host(ctx.hmult_batch(L, As, Bs, K))
    want = {k: o.hmult(L, pool[k], pool[(k + 1) % 3], evk, L) for k in range(3)}
    for i in (0, 1, 2, 63, 64):
        eq(got[i], want[i % 3], ("hmult_batch", i))
    rot = to_host(ctx.hrotate_batch(L, As, K, 25))
    for i in (2, 64):
        eq(rot[i], o.hrotate(L, pool[i % 3], evk, L, 25), ("hrotate_batch", i))
    ctx.close()


@pytest.mark.parametrize("w", [28, 33])
def test_host_paths_words_and_packed(w):
    """hml_hmult_host / hml_hmult_host_packed (5 bytes a coefficient over PCIe): at 28 bits the fifth byte is zero, at 33 bits
    bit 32 is set; 11 ciphertexts = one full chunk of 8 and a partial one"""
    N, ML, A, L, n = 65536, 45, 15, 12, 11
    ctx, o = _ctx(w, N, ML, A)
    a, b, evk = _case(o, L, L, 1000 + w)
    want = o.hmult(L, a, b, evk, L)
    want_r = o.hrotate(L, a, evk, L, 5)
    A_ = torch.stack([to_dev(a if i % 2 == 0 else b) for i in range(n)]).cpu().pin_memory()
    B_ = torch.stack([to_dev(b if i % 2 == 0 else a) for i in range(n)]).cpu().pin_memory()
    K = to_dev(evk)
    oh = torch.empty(n, 2, L - 1, N, dtype=torch.int64).pin_memory()
    ctx.hmult_host(L, A_, B_, K, oh)
    for i in (0, 7, 8, 10):
        eq(oh[i].numpy().view(np.uint64), want, ("hmult_host", i))
    ap, bp = ctx.pack_host(A_), ctx.pack_host(B_)
    assert torch.equal(ctx.unpack_host(ap, A_.shape), A_)
    op = torch.empty(n * 2 * (L - 1) * 5 * N, dtype=torch.uint8).pin_memory()
    ctx.hmult_host_packed(L, n, ap, bp, K, op)
    assert torch.equal(ctx.unpack_host(op, oh.shape), oh)
    rp = torch.empty(n * 2 * L * 5 * N, dtype=torch.uint8).pin_memory()
    ctx.hrotate_host_packed(L, n, ap, K, rp, 5)
    rot = ctx.unpack_host(rp, A_.shape)
    for i in (0, 8, 10):
        eq(rot[i].numpy().view(np.uint64), want_r, ("hrotate_host_packed", i))
    ctx.close()


def test_sharded_ops_at_28_bits():
    """world-2 limb-sharded keyswitch, hmult and hrotate (hml_group_op, both ranks emulated on this GPU) at 28 bits against the
    one-GPU ops, which are checked against the oracle here too"""
    from test_gpu_sharded import _split
    N, ML, A, L, world = 65536, 45, 15, 20, 2
    ctxs = [hml.Context(N=N, max_level=ML, alpha=A, element_bit_width=28) for _ in range(world)]
    o = Oracle(N, 28, ML, A)
    a, b, evk = _case(o, L, L, 1100)
    ctx = ctxs[0]
    K = to_dev(evk)
    one_ks = [to_host(t) for t in ctx.keyswitch(L, to_dev(a[1]), K)]
    one_rot = to_host(ctx.hrotate(L, to_dev(a), K, 25))
    one_mul = to_host(ctx.hmult(L, to_dev(a), to_dev(b), K))
    eq(one_mul, o.hmult(L, a, b, evk, L), "one-GPU hmult")
    eq(one_rot, o.hrotate(L, a, evk, L, 25), "one-GPU hrotate")
    group = hml.Shard.local_group(ctxs, L)
    for sh in group:
        sh.prepare(L)
    own, a_own, evk_own = _split(o, L, world, a, evk)
    _, b_own, _ = _split(o, L, world, b, evk)
    keep = [[i for i in own[r] if i < L - 1] for r in range(world)]

    def assemble(outs, idx, shape):
        got = np.zeros(shape, dtype=np.uint64)
        for r in range(world):
            got[..., idx[r], :] = to_host(outs[r])[..., :len(idx[r]), :]
        return got

    o0 = [ctxs[r].empty(len(own[r]), N) for r in range(world)]
    o1 = [ctxs[r].empty(len(own[r]), N) for r in range(world)]
    hml.group_op(group, "keyswitch", L, [x[1].contiguous() for x in a_own], key=evk_own, out0=o0, out1=o1)
    eq(assemble(o0, own, (L, N)), one_ks[0], "sharded keyswitch 0")
    eq(assemble(o1, own, (L, N)), one_ks[1], "sharded keyswitch 1")
    rot = [ctxs[r].empty(2, len(own[r]), N) for r in range(world)]
    hml.group_op(group, "hrotate", L, a_own, key=evk_own, out0=rot, galois_elt=25)
    eq(assemble(rot, own, (2, L, N)), one_rot, "sharded hrotate")
    mul = [ctxs[r].empty(2, len(keep[r]), N) for r in range(world)]
    hml.group_op(group, "hmult", L, a_own, b=b_own, key=evk_own, out0=mul)
    eq(assemble(mul, keep, (2, L - 1, N)), one_mul, "sharded hmult")
    for sh in group:
        sh.check()
        sh.close()
    for c in ctxs:
        c.close()


@pytest.mark.parametrize("w,N,ML,A", [(19, 2048, 4, 2), (37, 2048, 4, 2), (20, 65536, 1, 1), (20, 65536, 2, 1), (20, 4096, 9, 2),
                                      (24, 65536, 60, 20)])
def test_unsupported_widths_and_rings_are_rejected(w, N, ML, A):
    """widths outside [20, 36] and rings without enough primes = 1 (mod 2N) in (2^(w-1), 2^w) fail context creation with an
    HmlError (no crash, no context)"""
    with pytest.raises(hml.HmlError):
        hml.Context(N=N, max_level=ML, alpha=A, element_bit_width=w)
    # the library still works afterwards
    ctx = hml.Context(N=2048, max_level=4, alpha=2, element_bit_width=20)
    assert len(ctx.moduli) == 6
    ctx.close()
