"""Double-hoisted BSGS linear transforms on one GPU at BASELINE.json's north star (N = 2^16, maxLevel 45, L 35, alpha 15):
bsgs_trace(n1, n2) for (n1, n2) in (4, 4), (8, 8), (16, 4), with word and with packed keys, timed in two arms:
  replay_hoist  Replay(bsgs_trace(n1, n2), graph=True, hoist=True): one ModUp for the n1 - 1 baby rotations and one ModDown
                per baby rotation, n1 * n2 pmult / hadd passes, n2 - 1 textbook giant rotations, then the trace's hmult(y, y)
  bsgs_op       hml_hrotate_bsgs_hoisted (one ModUp for every baby step, one per giant rotation, one ModDown per giant rotation
                and one at the end), then the same hmult(y, y), issued as launches
The trace's j = 0 step is y = g0 + g0, one extra add that does not change the work.  `bsgs_op_alone_us` is the op without the
hmult.  The arms alternate inside every repetition after a warm-up; each entry is the median over repetitions of the
CUDA-event time of `iters` back-to-back runs, per run.  The rotation keys (18 x 157 MB for 16 x 4) and plaintexts are far
larger than the L2.  exec_counts are those of one run of each arm (the replay run as launches: a graph replays the same ones).
Prints ONE JSON line with the card name, power limit and SM clocks read in the same run.
Run as: python profiles/bsgs_hoisted.py [--reps R] [--iters I]"""
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

import torch  # noqa: E402

import homulator_b200 as hml  # noqa: E402
from homulator_b200.replay import bsgs_trace  # noqa: E402
from sharded_hoisted import card  # noqa: E402

SHAPES = [(4, 4), (8, 8), (16, 4)]
COUNTS = ("kernel_launches", "ntt_limbs", "intt_limbs", "bconv_limb_macs", "ewe_limbs", "automorph_limbs")


def main():
    reps = int(sys.argv[sys.argv.index("--reps") + 1]) if "--reps" in sys.argv else 7
    iters = int(sys.argv[sys.argv.index("--iters") + 1]) if "--iters" in sys.argv else 10
    N, ML, L, A = 65536, 45, 35, 15
    ctx = hml.Context(N=N, max_level=ML, alpha=A)
    beta = -(-L // A)
    x = ctx.uniform(list(range(L)), 1, lead=(2,))
    evk_w = ctx.uniform(ctx.ext_mod_idx(L), 3, lead=(beta, 2))

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) * 1e3 / iters

    def compare(fns):
        """{name: median us per run}, the arms alternating inside every repetition"""
        for fn in fns.values():
            for _ in range(3):
                fn()
        torch.cuda.synchronize()
        t = {k: [] for k in fns}
        for _ in range(reps):
            for k, fn in fns.items():
                t[k].append(timed(fn))
        return {k: round(statistics.median(v), 1) for k, v in t.items()}

    def counts(fn):
        torch.cuda.synchronize()
        ctx.exec_counts(reset=True)
        fn()
        torch.cuda.synchronize()
        c = ctx.exec_counts()
        return {k: c[k] for k in COUNTS}

    res = {}
    for n1, n2 in SHAPES:
        trace = bsgs_trace(n1, n2)
        rots = sorted({op[3] for op in trace if op[0] == "hrotate"})
        keys_w = {r: ctx.uniform(ctx.ext_mod_idx(L), 100 + r, lead=(beta, 2)) for r in rots}
        pts = {k: ctx.uniform(ctx.ext_mod_idx(L), 1000 + k) for k in range(n1 * n2)}  # the extended basis serves both arms
        babies = [pow(5, i, 2 * N) for i in range(n1)]
        giants = [pow(5, n1 * j, 2 * N) for j in range(n2)]
        rows = [[pts[j * n1 + i] for i in range(n1)] for j in range(n2)]
        y, z = ctx.empty(2, L, N), ctx.empty(2, L - 1, N)
        for kind in ("word", "packed"):
            if kind == "word":
                keys, evk, kq = keys_w, evk_w, L
            else:
                keys, evk, kq = {r: ctx.key_pack(k) for r, k in keys_w.items()}, ctx.key_pack(evk_w), L | hml.KEY_PACKED
            bk = [None] + [keys[i] for i in range(1, n1)]
            gk = [None] + [keys[n1 * j] for j in range(1, n2)]

            def op():
                ctx.hrotate_bsgs_hoisted(L, x, babies, bk, giants, gk, rows, evk_q_limbs=kq, out=y)

            def op_hmult():
                op()
                ctx.hmult(L, y, y, evk, evk_q_limbs=kq, out=z)

            # the op's workspace is the largest at this level: size it before the replay captures a graph that points into it
            op()
            torch.cuda.synchronize()
            rp = hml.Replay(ctx, L, trace, graph=True, hoist=True).bind(x, pts, keys, evk, evk_q_limbs=kq)
            name = "bsgs_%dx%d_%s" % (n1, n2, kind)
            res[name + "_us"] = compare({"replay_hoist": rp.run, "bsgs_op": op_hmult})
            res[name + "_op_alone_us"] = compare({"bsgs_op": op})["bsgs_op"]
            rp.close()
            if kind == "word":
                launches = hml.Replay(ctx, L, trace, hoist=True).bind(x, pts, keys, evk, evk_q_limbs=kq)
                launches.run()
                res["bsgs_%dx%d_exec_counts" % (n1, n2)] = {"replay_hoist": counts(launches.run), "bsgs_op": counts(op_hmult)}
                launches.close()
    line = {**card(), "N": N, "maxLevel": ML, "L": L, "alpha": A, "reps": reps, "iters": iters,
            "timing": "CUDA events, median over repetitions of the per-run time of `iters` back-to-back runs; arms alternate"}
    line.update(res)
    print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
