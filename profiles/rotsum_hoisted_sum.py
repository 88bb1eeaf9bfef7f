"""Double-hoisted rotation sums on one GPU: rotsum_trace(16) and rotsum_trace(32) at BASELINE.json's north star (N = 2^16,
maxLevel 45, L 35, alpha 15), each replayed as one CUDA graph in three modes:
  textbook   every rotation is its own key switch, then pmult / hadd (the pmult_add peephole)
  hoist      HML_REPLAY_HOIST: one ModUp per run of rotations, one ModDown per rotation, then the same accumulation
  hoist_sum  HML_REPLAY_HOIST_SUM: the run and its accumulation are one hml_hrotate_sum_hoisted (one ModUp, one ModDown)
and the op alone for n = 16: hml_hrotate_sum_hoisted against hml_hrotate_hoisted followed by the weighted sum of its 16
outputs (one hml_pmult, 15 hml_pmult_add: what the replay runs).
Operands are uniform residues (Context.uniform); plaintexts span the extended basis (ext_mod_idx(L)), as hoist_sum binds them.
The modes alternate inside every repetition; each entry is the median over repetitions of the CUDA-event time of `iters`
back-to-back runs, per run.  The working set (2.4 GB of rotation keys for 16 rotations) is far larger than the L2.
Prints ONE JSON line with the card name, power limit and SM clocks read in the same run.
Run as: python profiles/rotsum_hoisted_sum.py [--reps R] [--iters I]"""
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

import torch  # noqa: E402

import homulator_b200 as hml  # noqa: E402
from homulator_b200.replay import rotsum_trace  # noqa: E402
from sharded_hoisted import card  # noqa: E402


def main():
    reps = int(sys.argv[sys.argv.index("--reps") + 1]) if "--reps" in sys.argv else 7
    iters = int(sys.argv[sys.argv.index("--iters") + 1]) if "--iters" in sys.argv else 10
    N, ML, L, A = 65536, 45, 35, 15
    ctx = hml.Context(N=N, max_level=ML, alpha=A)
    beta = -(-L // A)
    x = ctx.uniform(list(range(L)), 1, lead=(2,))
    evk = ctx.uniform(ctx.ext_mod_idx(L), 3, lead=(beta, 2))
    pts = {i: ctx.uniform(ctx.ext_mod_idx(L), 200 + i) for i in range(32)}
    keys = {r: ctx.uniform(ctx.ext_mod_idx(L), 100 + r, lead=(beta, 2)) for r in range(1, 33)}

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) * 1e3 / iters

    def compare(fns):
        """{name: median us per run}, the candidates alternating inside every repetition"""
        for fn in fns.values():
            for _ in range(3):
                fn()
        torch.cuda.synchronize()
        t = {k: [] for k in fns}
        for _ in range(reps):
            for k, fn in fns.items():
                t[k].append(timed(fn))
        return {k: round(statistics.median(v), 1) for k, v in t.items()}

    res = {}
    modes = {"textbook": {}, "hoist": {"hoist": True}, "hoist_sum": {"hoist_sum": True}}
    for n in (16, 32):
        rps = {m: hml.Replay(ctx, L, rotsum_trace(n), graph=True, **kw).bind(x, pts, keys, evk) for m, kw in modes.items()}
        res["rotsum_%d_graph_us" % n] = compare({m: rp.run for m, rp in rps.items()})
        for rp in rps.values():
            rp.close()

    # the op alone, n = 16
    n = 16
    gs = [pow(5, r, 2 * N) for r in range(1, n + 1)]
    ks, ps = [keys[r] for r in range(1, n + 1)], [pts[i] for i in range(n)]
    outs = [ctx.empty(2, L, N) for _ in range(n)]
    acc, y = ctx.empty(2, L, N), ctx.empty(2, L, N)

    def hoisted_then_pmult_add():
        ctx.hrotate_hoisted(L, x, ks, gs, outs=outs)
        ctx.pmult(L, outs[0], ps[0], out=acc)
        for i in range(1, n):
            ctx.pmult_add(L, outs[i], ps[i], acc, out=acc)

    res["op_16_us"] = compare({"hrotate_hoisted_then_weighted_sum": hoisted_then_pmult_add,
                               "hrotate_sum_hoisted": lambda: ctx.hrotate_sum_hoisted(L, x, ks, gs, ps, out=y)})
    line = {**card(), "N": N, "maxLevel": ML, "L": L, "alpha": A, "reps": reps, "iters": iters,
            "timing": "CUDA events, median over repetitions of the per-run time of `iters` back-to-back runs; modes alternate"}
    line.update(res)
    print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
