#!/usr/bin/env python3
"""Regenerate tests/golden/exec_counts.json: hml_exec_counts after each op (needs a GPU).

Covers the one-GPU primitives and ops, the batched and host-buffer ops and the limb-sharded ops of local groups of 2 and 3
emulated ranks (hml_group_op, hml_group_hrotate_hoisted and the collective variant of the sharded key switch) on a
single-pass ring (N = 4096), a small two-pass ring (N = 8192) and the north-star ring (N = 2^16, L = 35, alpha = 15).  The
counters depend on the shapes only, so every operand is zero.  tests/test_gpu_exec_counts.py replays the same cases and
compares them with the committed file.

    python tests/golden/gen_exec_counts.py [--profile]

--profile writes nothing; it runs every case inside hml_profile_begin / hml_profile_end and prints a `# <case>` line to
stderr before each, so that with HML_PROFILE_DUMP=1 stderr holds the class of every launch group of every case."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden", "exec_counts.json")
SHAPES = {"n4096": (4096, 6, 5, 2), "n8192": (8192, 9, 8, 3), "north_star": (65536, 45, 35, 15)}
WORLDS = (2, 3)


def _ctx_ops(ctx, L):
    """(name, fn) of every one-GPU case at level L; fn() runs the op once"""
    import torch
    import homulator_b200 as hml
    N, A = ctx.N, ctx.alpha
    beta, E = ctx.beta(L), L + A
    nm = len(ctx.moduli)
    small = N <= 8192
    z = lambda *shape: torch.zeros(*shape, dtype=torch.int64, device=ctx.device)  # noqa: E731
    ct, ct2, evk = z(2, L, N), z(2, L, N), z(beta, 2, E, N)
    keys = [z(beta, 2, E, N) for _ in range(3)]
    gs = [5, 1, 2 * N - 1]
    evk_p = ctx.key_pack(evk)

    def pinned(*shape):
        return torch.zeros(*shape, dtype=torch.int64).pin_memory()

    def packed(n_limbs):
        return torch.zeros(ctx.lib.hml_packed_bytes(ctx.h, n_limbs), dtype=torch.uint8).pin_memory()

    wide = [i % nm for i in range(130)]
    ops = [
        ("ntt", lambda: ctx.ntt(ct[0], list(range(L)))),
        ("intt", lambda: ctx.intt(ct[0], list(range(L)))),
        ("ntt_130_limbs", lambda: ctx.ntt(z(130, N), wide)),
        ("intt_130_limbs", lambda: ctx.intt(z(130, N), wide)),
        ("ntt_batch", lambda: ctx.ntt_batch(z(3, L, N), list(range(L)))),
        ("intt_batch", lambda: ctx.ntt_batch(z(3, L, N), list(range(L)), inverse=True)),
        ("keyswitch", lambda: ctx.keyswitch(L, ct[1], evk)),
        ("keyswitch_packed_key", lambda: ctx.keyswitch(L, ct[1], evk_p, L | hml.KEY_PACKED)),
        ("rescale", lambda: ctx.rescale(L, ct[0])),
        ("hmult", lambda: ctx.hmult(L, ct, ct2, evk)),
        ("hmult_packed_key", lambda: ctx.hmult(L, ct, ct2, evk_p, L | hml.KEY_PACKED)),
        ("hrotate", lambda: ctx.hrotate(L, ct, evk, 5)),
        ("hrotate_g1", lambda: ctx.hrotate(L, ct, evk, 1)),
        ("hrotate_in_place", lambda: ctx.hrotate(L, ct2, evk, 5, out=ct2)),
        ("hrotate_hoisted", lambda: ctx.hrotate_hoisted(L, ct, keys, gs)),
        ("hmult_batch_3", lambda: ctx.hmult_batch(L, z(3, 2, L, N), z(3, 2, L, N), evk)),
        ("hmult_batch_6", lambda: ctx.hmult_batch(L, z(6, 2, L, N), z(6, 2, L, N), evk)),
        ("hrotate_batch_3", lambda: ctx.hrotate_batch(L, z(3, 2, L, N), evk, 5)),
        ("hrotate_batch_6", lambda: ctx.hrotate_batch(L, z(6, 2, L, N), evk, 5)),
        ("hmult_host_3", lambda: ctx.hmult_host(L, pinned(3, 2, L, N), pinned(3, 2, L, N), evk, pinned(3, 2, L - 1, N))),
        ("hrotate_host_3", lambda: ctx.hrotate_host(L, pinned(3, 2, L, N), evk, pinned(3, 2, L, N), 5)),
        ("hmult_host_packed_3", lambda: ctx.hmult_host_packed(L, 3, packed(6 * L), packed(6 * L), evk, packed(6 * (L - 1)))),
        ("hrotate_host_packed_3", lambda: ctx.hrotate_host_packed(L, 3, packed(6 * L), evk, packed(6 * L), 5)),
    ]
    if small:  # batches that cross a chunk boundary (transform: 16384 limbs per launch; ops: 64 ciphertexts)
        ops += [("ntt_batch_chunked", lambda: ctx.ntt_batch(z(130, 128, N), list(range(nm)) * (128 // nm) + list(range(128 % nm)))),
                ("hmult_batch_70", lambda: ctx.hmult_batch(L, z(70, 2, L, N), z(70, 2, L, N), evk)),
                ("hrotate_batch_70", lambda: ctx.hrotate_batch(L, z(70, 2, L, N), evk, 5))]
    return ops


def _group_ops(ctxs, L, world):
    """(name, fn) of every sharded case of one emulated group"""
    import torch
    import homulator_b200 as hml
    N, A = ctxs[0].N, ctxs[0].alpha
    beta = ctxs[0].beta(L)
    R = range(world)
    own = [list(range(r, L, world)) for r in R]
    own_e = [[e for e in range(L + A) if e % world == r] for r in R]
    nq = [max(len(own[r]), 1) for r in R]
    z = lambda *shape: torch.zeros(*shape, dtype=torch.int64, device=ctxs[0].device)  # noqa: E731
    ct = [z(2, nq[r], N) for r in R]
    d = [z(nq[r], N) for r in R]
    evk = [z(beta, 2, len(own_e[r]), N) if own_e[r] else None for r in R]
    gs = [5, 1, 2 * N - 1]
    keys = [[z(beta, 2, len(own_e[r]), N) if own_e[r] else None for _ in gs] for r in R]
    g1 = hml.Shard.local_group(ctxs, L)
    g2 = hml.Shard.local_group(ctxs, L, max_rot=2)
    for sh in g1 + g2:
        sh.prepare(L)

    def collective_keyswitch():  # hml_keyswitch_shard_begin / _mid / _end, the all-gathers done as device copies
        st = torch.cuda.current_stream().cuda_stream
        lays = [hml.shard_layout(L, A, r, world) for r in R]
        b1 = [z(world, lays[r]["gather1_slots"], N) for r in R]
        b2 = [z(world, 2, lays[r]["gather2_slots"], N) for r in R]
        for r, c in enumerate(ctxs):
            c._chk(c.lib.hml_keyswitch_shard_begin(c.h, L, r, world, d[r].data_ptr(), b1[r].data_ptr(), st))
        for r in R:
            for s in R:
                b1[r][s].copy_(b1[s][s])
        for r, c in enumerate(ctxs):
            if evk[r] is not None:
                c._chk(c.lib.hml_keyswitch_shard_mid(c.h, L, r, world, d[r].data_ptr(), b1[r].data_ptr(), evk[r].data_ptr(),
                                                     b2[r].data_ptr(), st))
        for r in R:
            for s in R:
                b2[r][s].copy_(b2[s][s])
        for r, c in enumerate(ctxs):
            o0, o1 = z(nq[r], N), z(nq[r], N)
            c._chk(c.lib.hml_keyswitch_shard_end(c.h, L, r, world, b2[r].data_ptr(), o0.data_ptr(), o1.data_ptr(), st))

    return [
        ("keyswitch", lambda: hml.group_op(g1, "keyswitch", L, d, key=evk, out0=[z(nq[r], N) for r in R], out1=[z(nq[r], N) for r in R])),
        ("hrotate", lambda: hml.group_op(g1, "hrotate", L, ct, key=evk, out0=[z(2, nq[r], N) for r in R], galois_elt=25)),
        ("hrotate_g1", lambda: hml.group_op(g1, "hrotate", L, ct, key=evk, out0=[z(2, nq[r], N) for r in R], galois_elt=1)),
        ("hmult", lambda: hml.group_op(g1, "hmult", L, ct, b=ct, key=evk, out0=[z(2, nq[r], N) for r in R])),
        ("rescale", lambda: hml.group_op(g1, "rescale", L, ct, out0=[z(2, nq[r], N) for r in R])),
        ("hrotate_hoisted", lambda: hml.group_hrotate_hoisted(g1, L, ct, keys, gs)),
        ("hrotate_hoisted_max_rot_2", lambda: hml.group_hrotate_hoisted(g2, L, ct, keys, gs)),
        ("keyswitch_collective", collective_keyswitch),
    ], g1 + g2


def run_shape(shape, profile=False):
    """{case: counts} for one shape; counts is one dict for a one-GPU case and a list of one dict per rank for a group"""
    import torch
    import homulator_b200 as hml
    N, ML, L, A = SHAPES[shape]
    res = {}

    def once(name, ctxs, fn):
        for c in ctxs:
            c.exec_counts(reset=True)
        if profile:
            print("# %s" % name, file=sys.stderr, flush=True)
            for c in ctxs:
                c._chk(c.lib.hml_profile_begin(c.h, c._stream()))
        fn()
        torch.cuda.synchronize()
        if profile:
            from homulator_b200.api import _Profile
            import ctypes as C
            for c in ctxs:
                pr = _Profile()
                c._chk(c.lib.hml_profile_end(c.h, C.byref(pr)))
            sys.stderr.flush()
        got = [c.exec_counts() for c in ctxs]
        res[name] = got[0] if len(ctxs) == 1 else got

    ctx = hml.Context(N=N, max_level=ML, alpha=A)
    for n, fn in _ctx_ops(ctx, L):
        once("%s/%s" % (shape, n), [ctx], fn)
    ctx.close()
    for w in WORLDS:
        ctxs = [hml.Context(N=N, max_level=ML, alpha=A) for _ in range(w)]
        ops, group = _group_ops(ctxs, L, w)
        for n, fn in ops:
            once("%s/w%d/%s" % (shape, w, n), ctxs, fn)
        for sh in group:
            sh.check()
            sh.close()
        for c in ctxs:
            c.close()
    torch.cuda.empty_cache()
    return res


def main():
    profile = "--profile" in sys.argv[1:]
    res = {}
    for shape in SHAPES:
        res.update(run_shape(shape, profile))
    if profile:
        return
    with open(GOLDEN, "w") as f:
        json.dump(res, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote %d cases to %s" % (len(res), GOLDEN))


if __name__ == "__main__":
    main()
