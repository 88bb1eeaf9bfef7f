"""Lazily relinearised sums of products on one GPU at BASELINE.json's north star (N = 2^16, maxLevel 45, L 35, alpha 15):
  op_<n>_us          n in {4, 16, 64} products, one output: hml_hmult_sum against n hml_hmult + (n - 1) hml_hadd
  op_16_squares_us   the same for 16 squares (each term's two ciphertexts are one tensor, read once by hml_hmult_sum)
  op_16x32_us        16 products for each of 32 outputs: hml_hmult_sum (n_out = 32) against the 512 products through 16
                     hml_hmult_batch calls of 32, each followed by 32 hml_hadd into the running sums
  dot_16_graph_us    dot_trace(16) replayed as one CUDA graph with hoisted rotations, without and with hmult_sum=True
Operands are uniform residues (Context.uniform); every term reads its own ciphertexts (4.7 GB for 64 products), so the inputs
are far larger than the L2.  The candidates alternate inside every repetition; each entry is the median over repetitions of
the CUDA-event time of `iters` back-to-back runs, per run.  Prints ONE JSON line with the card name, power limit and SM clocks
read in the same run.
Run as: python profiles/hmult_sum.py [--reps R] [--iters I] > profiles/hmult_sum_1gpu.json"""
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

import torch  # noqa: E402

import homulator_b200 as hml  # noqa: E402
from homulator_b200.replay import dot_trace  # noqa: E402
from sharded_hoisted import card  # noqa: E402


def main():
    reps = int(sys.argv[sys.argv.index("--reps") + 1]) if "--reps" in sys.argv else 5
    iters = int(sys.argv[sys.argv.index("--iters") + 1]) if "--iters" in sys.argv else 5
    N, ML, L, A = 65536, 45, 35, 15
    ctx = hml.Context(N=N, max_level=ML, alpha=A)
    beta = -(-L // A)
    q = list(range(L))
    evk = ctx.uniform(ctx.ext_mod_idx(L), 3, lead=(beta, 2))
    cts = [ctx.uniform(q, 1000 + i, lead=(2,)) for i in range(128)]

    def timed(fn, n_iter):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_iter):
            fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) * 1e3 / n_iter

    def compare(fns, n_iter=None):
        """{name: median us per run}, the candidates alternating inside every repetition"""
        n_iter = n_iter or iters
        for fn in fns.values():
            for _ in range(2):
                fn()
        torch.cuda.synchronize()
        t = {k: [] for k in fns}
        for _ in range(reps):
            for k, fn in fns.items():
                t[k].append(timed(fn, n_iter))
        return {k: round(statistics.median(v), 1) for k, v in t.items()}

    def hmults_then_hadds(a, b, y, t):
        def run():
            ctx.hmult(L, a[0], b[0], evk, out=y)
            for x0, x1 in zip(a[1:], b[1:]):
                ctx.hmult(L, x0, x1, evk, out=t)
                ctx.hadd(L - 1, y, t, out=y)
        return run

    res = {}
    y, t, s = ctx.empty(2, L - 1, N), ctx.empty(2, L - 1, N), ctx.empty(2, L - 1, N)
    for n in (4, 16, 64):
        a, b = cts[:n], cts[n:2 * n]
        res["op_%d_us" % n] = compare({"hmult_then_hadd": hmults_then_hadds(a, b, y, t),
                                       "hmult_sum": lambda: ctx.hmult_sum(L, a, b, evk, out=s)})
    a = cts[:16]
    res["op_16_squares_us"] = compare({"hmult_then_hadd": hmults_then_hadds(a, a, y, t),
                                       "hmult_sum": lambda: ctx.hmult_sum(L, a, a, evk, out=s)})
    del cts

    # 16 products for each of 32 outputs
    n, n_out = 16, 32
    ba = [ctx.uniform(q, 2000 + i, lead=(n_out, 2)) for i in range(n)]
    bb = [ctx.uniform(q, 3000 + i, lead=(n_out, 2)) for i in range(n)]
    ys, ts, ss = (ctx.empty(n_out, 2, L - 1, N) for _ in range(3))

    def batches_then_hadds():
        ctx.hmult_batch(L, ba[0], bb[0], evk, out=ys)
        for x0, x1 in zip(ba[1:], bb[1:]):
            ctx.hmult_batch(L, x0, x1, evk, out=ts)
            for k in range(n_out):
                ctx.hadd(L - 1, ys[k], ts[k], out=ys[k])

    res["op_16x32_us"] = compare({"hmult_batch_then_hadd": batches_then_hadds,
                                  "hmult_sum": lambda: ctx.hmult_sum(L, ba, bb, evk, out=ss)}, n_iter=2)
    del ba, bb, ys, ts, ss

    # dot_trace(16): 15 hoisted rotations of x, then the chain of 16 products
    x = ctx.uniform(q, 1, lead=(2,))
    keys = {r: ctx.uniform(ctx.ext_mod_idx(L), 100 + r, lead=(beta, 2)) for r in range(1, 16)}
    rps = {m: hml.Replay(ctx, L, dot_trace(16), graph=True, hoist=True, hmult_sum=m == "hmult_sum").bind(x, [], keys, evk)
           for m in ("hoist", "hmult_sum")}
    res["dot_16_graph_us"] = compare({m: rp.run for m, rp in rps.items()})
    for rp in rps.values():
        rp.close()
    line = {**card(), "N": N, "maxLevel": ML, "L": L, "alpha": A, "reps": reps, "iters": iters,
            "timing": "CUDA events, median over repetitions of the per-run time of `iters` back-to-back runs (2 for op_16x32); "
                      "candidates alternate"}
    line.update(res)
    print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
