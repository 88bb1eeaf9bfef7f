"""Double-hoisted rotation sums and lazily relinearised product sums on a limb-sharded ciphertext, at BASELINE.json's north star
(N = 2^16, maxLevel 45, L 35, alpha 15), on a world-1 shard (the real fused exchange on one GPU):
  rotsum_16_us    sum_i pt_i * rotate(ct, g_i), 16 rotations:
                    sum_sharded      hml_hrotate_sum_hoisted_sharded
                    hoisted_ew       hml_hrotate_hoisted_sharded (one group of 16) + 16 hml_ew_sharded pmult passes (kind 1, then 3)
                    one_gpu          hml_hrotate_sum_hoisted
  hmult_sum_16_us sum_i a_i * b_i, 16 products:
                    sum_sharded      hml_hmult_sum_sharded
                    hmult_hadd       16 hml_hmult_sharded + 15 hml_ew_sharded hadds
                    one_gpu          hml_hmult_sum
Operands are uniform residues (Context.uniform): 16 rotation keys (2.5 GB) and 32 ciphertexts (1.1 GB), far larger than the L2.
The arms alternate inside every repetition; each entry is the median over repetitions of the CUDA-event time of `iters`
back-to-back runs, per run.  With >= 2 visible GPUs, tests/mp_sharded_sums.py runs under torchrun over 2, 4 and 8 of them and
its timing lines are added; otherwise the multi-GPU entry says "not measured".  Prints ONE JSON line with the card name, power
limit and SM clocks read in the same run.
Run as: python profiles/sharded_sums.py [--reps R] [--iters I] > profiles/sharded_sums_1gpu.json"""
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

import torch  # noqa: E402

import homulator_b200 as hml  # noqa: E402
from homulator_b200.replay import shard_plaintexts  # noqa: E402
from sharded_hoisted import card  # noqa: E402


def multi_gpu():
    g = torch.cuda.device_count()
    if g < 2:
        return "not measured (%d GPU visible)" % g
    lines = []
    for w in (2, 4, 8):
        if w > g:
            break
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(w), "--master-addr", "127.0.0.1",
               "--master-port", "29551", os.path.join(ROOT, "tests", "mp_sharded_sums.py")]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=1800)
        lines += [json.loads(s.split(" ", 1)[1]) for s in r.stdout.splitlines() if s.startswith("SHARDED_SUMS_TIME ")]
    return lines


def main():
    reps = int(sys.argv[sys.argv.index("--reps") + 1]) if "--reps" in sys.argv else 5
    iters = int(sys.argv[sys.argv.index("--iters") + 1]) if "--iters" in sys.argv else 5
    N, ML, L, A = 65536, 45, 35, 15
    n = 16
    ctx = hml.Context(N=N, max_level=ML, alpha=A)
    q, ext, beta = list(range(L)), ctx.ext_mod_idx(L), ctx.beta(L)
    ct = ctx.uniform(q, 1, lead=(2,))
    keys = [ctx.uniform(ext, 100 + i, lead=(beta, 2)) for i in range(n)]
    pts = [ctx.uniform(ext, 200 + i) for i in range(n)]
    gs = [pow(5, r, 2 * N) for r in range(1, n + 1)]
    a = [ctx.uniform(q, 300 + i, lead=(2,)) for i in range(n)]
    b = [ctx.uniform(q, 400 + i, lead=(2,)) for i in range(n)]
    evk = ctx.uniform(ext, 3, lead=(beta, 2))
    sh = hml.Shard(ctx, L, 0, 1, max_rot=16)
    sh.prepare(L)
    pts_ext = shard_plaintexts(sh, L, pts)          # world 1: every row, [L + alpha][N]
    pts_q = [p[:L].contiguous() for p in pts]       # the element-wise passes read the Q-limbs only
    lib, st = ctx.lib, ctx._stream

    def timed(fn, n_iter):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_iter):
            fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) * 1e3 / n_iter

    def compare(fns):
        """{name: median us per run}, the arms alternating inside every repetition"""
        for fn in fns.values():
            for _ in range(2):
                fn()
        torch.cuda.synchronize()
        t = {k: [] for k in fns}
        for _ in range(reps):
            for k, fn in fns.items():
                t[k].append(timed(fn, iters))
        return {k: round(statistics.median(v), 1) for k, v in t.items()}

    rot_outs = [ctx.empty(2, L, N) for _ in range(n)]
    y, s1, s2 = ctx.empty(2, L, N), ctx.empty(2, L, N), ctx.empty(2, L, N)

    def hoisted_ew():
        sh.hrotate_hoisted(L, ct, keys, gs, outs=rot_outs)
        for i in range(n):
            ctx._chk(lib.hml_ew_sharded(sh.h, L, 1 if i == 0 else 3, rot_outs[i].data_ptr(), pts_q[i].data_ptr(), y.data_ptr(), st()))

    res = {"rotsum_16_us": compare({"sum_sharded": lambda: sh.hrotate_sum_hoisted(L, ct, keys, gs, pts_ext, out=s1),
                                    "hoisted_ew": hoisted_ew,
                                    "one_gpu": lambda: ctx.hrotate_sum_hoisted(L, ct, keys, gs, pts, out=s2)})}
    # every arm computes its own function: the sum against the one-GPU op bit for bit
    torch.cuda.synchronize()
    assert torch.equal(s1, s2)
    del rot_outs

    m, t, m1, m2 = (ctx.empty(2, L - 1, N) for _ in range(4))

    def hmult_hadd():
        sh.hmult(L, a[0], b[0], evk, out=m)
        for x0, x1 in zip(a[1:], b[1:]):
            sh.hmult(L, x0, x1, evk, out=t)
            ctx._chk(lib.hml_ew_sharded(sh.h, L - 1, 0, m.data_ptr(), t.data_ptr(), m.data_ptr(), st()))

    res["hmult_sum_16_us"] = compare({"sum_sharded": lambda: sh.hmult_sum(L, a, b, evk, out=m1),
                                      "hmult_hadd": hmult_hadd,
                                      "one_gpu": lambda: ctx.hmult_sum(L, a, b, evk, out=m2)})
    torch.cuda.synchronize()
    assert torch.equal(m1, m2)
    sh.check()
    sh.close()
    line = {**card(), "N": N, "maxLevel": ML, "L": L, "alpha": A, "world": 1, "reps": reps, "iters": iters,
            "timing": "CUDA events, median over repetitions of the per-run time of `iters` back-to-back runs; arms alternate"}
    line.update(res)
    line["multi_gpu"] = multi_gpu()
    print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
