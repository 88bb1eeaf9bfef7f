"""Child process of tests/test_gpu_ops.py::test_alternative_kernel_paths: the library reads its switches once per process
(HML_BCONV_UMMA, HML_PDL, HML_BATCH_CHUNK), so every setting is proven in a process of its own: hmult / hrotate / keyswitch /
rescale / batched ops against the oracle on a two-pass ring, and batched transforms small enough for the 128-thread column
pass and large enough for the 256-thread one."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import homulator_b200 as hml  # noqa: E402
from gpu_common import to_dev, to_host  # noqa: E402
from orc import Oracle, uniform_limbs  # noqa: E402


def main():
    Oracle.set_threads(0)
    for N, ML, A, L in ((8192, 7, 3, 7), (16384, 6, 2, 5)):
        ctx, o = hml.Context(N=N, max_level=ML, alpha=A), Oracle(N, 36, ML, A)
        beta = -(-L // A)
        a = uniform_limbs(o.moduli[:L], N, 1, lead=(2,))
        b = uniform_limbs(o.moduli[:L], N, 2, lead=(2,))
        evk = uniform_limbs(o.moduli[:L] + o.moduli[ML:], N, 3, lead=(beta, 2))
        K = to_dev(evk)
        want_m, want_r = o.hmult(L, a, b, evk, L), o.hrotate(L, a, evk, L, 25)
        assert np.array_equal(to_host(ctx.hmult(L, to_dev(a), to_dev(b), K)), want_m)
        assert np.array_equal(to_host(ctx.hrotate(L, to_dev(a), K, 25)), want_r)
        w0, w1 = o.keyswitch(L, b[1], evk, L)
        g0, g1 = ctx.keyswitch(L, to_dev(b[1]), K, L)
        assert np.array_equal(to_host(g0), w0) and np.array_equal(to_host(g1), w1)
        assert np.array_equal(to_host(ctx.rescale(L, to_dev(a[0]))), o.rescale(L, a[0]))
        A3, B3 = torch.stack([to_dev(a), to_dev(b), to_dev(a)]), torch.stack([to_dev(b), to_dev(b), to_dev(a)])
        got = ctx.hmult_batch(L, A3, B3, K)
        assert np.array_equal(to_host(got[0]), want_m) and np.array_equal(to_host(got[1]), o.hmult(L, b, b, evk, L))
        rot = ctx.hrotate_batch(L, A3, K, 25)
        assert np.array_equal(to_host(rot[2]), want_r)
        idx = list(range(L))
        # 3 x L limbs: 128-thread column CTAs.  256 x L limbs is at least 18 32 KB tiles per SM (3584 tiles at N = 8192,
        # 5120 at N = 16384): 256-thread column CTAs
        for lead, seed, j in (((3,), 9, 1), ((256,), 10, 200)):
            x = ctx.uniform(idx, seed, lead=lead)
            fwd = ctx.ntt_batch(x, idx)
            assert torch.equal(ctx.ntt_batch(fwd, idx, inverse=True), x)
            for i in range(L):
                assert np.array_equal(to_host(fwd[j, i]), o.ntt(i, to_host(x[j, i])))
    print("ENV_PATHS_OK")


if __name__ == "__main__":
    main()
