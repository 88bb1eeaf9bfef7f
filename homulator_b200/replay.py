"""Op-sequence traces (BASELINE.json configs[4]; SURVEY.md 8f rank 3) and a thin front end to the C ABI's replay object.

The reference simulates ONE operation per run and explicitly does not chain them ("NotSuppotr the continuous operation
simulate", reference src/Operation.cpp:636,675,714); its repository contains no application trace.  A trace here is a list of
tuples over the five operations the reference's CLI accepts (reference bench_test/bench_micro24.cpp:29-48):
    ("hrotate", dst, src, r)        dst = rotate(src, 5^r)            (rotation key bound for amount r)
    ("pmult",   dst, src, pt)       dst = src * plaintext[pt]
    ("hadd",    dst, a, b)          dst = a + b
    ("padd",    dst, src, pt)       dst = src + plaintext[pt]
    ("hmult",   dst, a, b)          dst = rescale(relin(a * b))       (drops one level; final)
Execution lives in the library (homulator_b200/csrc/replay.cu: hml_replay_*): plain launches or one captured CUDA graph,
textbook, hoisted or (one GPU) double-hoisted rotation sums and lazily relinearised product sums, one GPU or limb-sharded over a group.  This module only defines the synthetic traces and maps
names to slots (homulator_b200.api.Replay).
"""
from collections import Counter


def bsgs_trace(n1=4, n2=4):
    """Baby-step/giant-step matrix-vector product (the inner loop of CKKS bootstrapping's CoeffToSlot): n1 - 1 baby rotations of
    x, n1 * n2 plaintext multiplications and additions, n2 - 1 giant rotations, then one hmult."""
    t = []
    for i in range(1, n1):                       # baby steps: rot_i = rotate(x, i)
        t.append(("hrotate", "b%d" % i, "x", i))
    for j in range(n2):                          # giant steps
        acc = None
        for i in range(n1):
            src = "x" if i == 0 else "b%d" % i
            if acc is None:
                acc = "g%d" % j
                t.append(("pmult", acc, src, j * n1 + i))
            else:
                t.append(("pmult", "m", src, j * n1 + i))
                t.append(("hadd", acc, acc, "m"))
        if j:
            t.append(("hrotate", acc, acc, n1 * j))
            t.append(("hadd", "y", "y", acc))
        else:
            t.append(("hadd", "y", acc, acc))
    t.append(("hmult", "z", "y", "y"))
    return t


def rotsum_trace(n=16):
    """The shape SURVEY.md 8d suggests for configs[4]: y = sum_i plaintext_i * rotate(x, i + 1) over n rotations of ONE
    ciphertext (n hrotate + n pmult + n - 1 hadd), then one hmult.  Every rotation reads x: fully hoistable."""
    t = [("hrotate", "r%d" % i, "x", i + 1) for i in range(n)]
    for i in range(n):
        if i == 0:
            t.append(("pmult", "y", "r0", 0))
        else:
            t.append(("pmult", "m", "r%d" % i, i))
            t.append(("hadd", "y", "y", "m"))
    t.append(("hmult", "z", "y", "y"))
    return t


def dot_trace(n=16):
    """y = sum_{i<n} x * rotate(x, i): n - 1 hoistable rotations of x, then the chain of products summed as they are formed
    (one square x * x, n - 1 products and n - 1 hadd).  The rotation-plus-product shape of an encrypted inner product; with
    hmult_sum=True the chain is one hml_hmult_sum."""
    t = [("hrotate", "r%d" % i, "x", i) for i in range(1, n)]
    t.append(("hmult", "y", "x", "x"))
    for i in range(1, n):
        t.append(("hmult", "m", "x", "r%d" % i))
        t.append(("hadd", "y", "y", "m"))
    return t


def trace_counts(trace):
    return dict(Counter(op[0] for op in trace))


def replay(ctx, L, trace, x, plaintexts, rot_keys, evk, graph=False, hoist=False, hoist_sum=False, names=("y", "z")):
    """Run `trace` once at level L through hml_replay_* and return {name: tensor} for `names` (copies).  With hoist_sum=True
    the plaintexts are [L + alpha][N] (see homulator_b200.api.Replay)."""
    from .api import Replay
    rp = Replay(ctx, L, trace, graph=graph, hoist=hoist, hoist_sum=hoist_sum).bind(x, plaintexts, rot_keys, evk)
    rp.run()
    out = {n: rp.result(n).clone() for n in names if n in rp.names}
    rp.close()
    return out


def shard_operands(sh, L, x, plaintexts, rot_keys, evk):
    """This rank's slices of full-size operands: ciphertext [2][nq][N], plaintexts [nq][N], keys [beta][2][n_own_ext][N]."""
    import torch
    oi = torch.tensor(sh.own_q(L), device=x.device, dtype=torch.long)
    oe = torch.tensor(sh.own_ext(L), device=x.device, dtype=torch.long)
    cut = lambda k: k[:, :, oe].contiguous() if k is not None else None  # noqa: E731
    return (x[:, oi].contiguous(), {i: p[oi].contiguous() for i, p in plaintexts.items()}, {r: cut(k) for r, k in rot_keys.items()}, cut(evk))


def shard_plaintexts(sh, L, plaintexts):
    """This rank's slices of extended-basis plaintexts [L + alpha][N] (P-limb j at row L + j), as the sharded rotation sum takes
    them: the owned rows in own_ext(L) order, [nq + np][N]; None where the rank owns no extended limb."""
    import torch
    own = sh.own_ext(L)
    if not own:
        return [None for _ in plaintexts]
    oe = torch.tensor(own, device=plaintexts[0].device, dtype=torch.long) if plaintexts else None
    return [p[oe].contiguous() for p in plaintexts]
