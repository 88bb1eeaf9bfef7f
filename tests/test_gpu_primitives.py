"""GPU parity, primitives: every kernel class against the scalar oracle, bit-exact, through the C ABI."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import homulator_b200 as hml  # noqa: E402
from gpu_common import to_dev, to_host  # noqa: E402
from orc import Oracle, uniform_limbs  # noqa: E402


@pytest.fixture(scope="module")
def big():
    """north-star parameter set: N=2^16, 36-bit words, maxLevel 45, alpha 15"""
    return hml.Context(N=65536, max_level=45, alpha=15), Oracle(65536, 36, 45, 15)


def test_moduli_and_roots_match_oracle(big):
    ctx, o = big
    assert ctx.moduli == o.moduli
    assert ctx.psi == o.psi


@pytest.mark.parametrize("logN", [4, 5, 8, 11, 12, 13, 14, 15, 16])
def test_ntt_intt_all_sizes(logN):
    N = 1 << logN
    ml, al = 5, 3
    ctx, o = hml.Context(N=N, max_level=ml, alpha=al), Oracle(N, 36, ml, al)
    assert ctx.moduli == o.moduli
    idx = list(range(ml + al))
    x = uniform_limbs(o.moduli, N, 100 + logN)
    # edge values: zeros, q-1, 1
    x[0, :4] = 0
    x[1, :4] = o.moduli[1] - 1
    x[2, :] = o.moduli[2] - 1
    want = np.stack([o.ntt(i, x[i]) for i in idx])
    got = to_host(ctx.ntt(to_dev(x), idx))
    assert np.array_equal(got, want)
    back = to_host(ctx.intt(to_dev(want), idx))
    assert np.array_equal(back, x)
    want_i = np.stack([o.intt(i, x[i]) for i in idx])
    assert np.array_equal(to_host(ctx.intt(to_dev(x), idx)), want_i)
    # in place
    d = to_dev(x)
    ctx.ntt(d, idx, out=d)
    assert np.array_equal(to_host(d), want)


def test_ntt_north_star_all_60_moduli(big):
    ctx, o = big
    idx = list(range(60))
    x = uniform_limbs(o.moduli, 65536, 7)
    got = to_host(ctx.ntt(to_dev(x), idx))
    for i in (0, 1, 17, 34, 44, 45, 59):
        assert np.array_equal(got[i], o.ntt(i, x[i])), i
    # every limb: round trip + Horner spot check of the definition a(psi^(2 brv(k)+1)) on random slots
    assert np.array_equal(to_host(ctx.intt(to_dev(got), idx)), x)
    rng = np.random.default_rng(1)
    for i in idx:
        m, psi = o.moduli[i], o.psi[i]
        for k in rng.integers(0, 65536, 2):
            brv = int(format(int(k), "016b")[::-1], 2)
            pt = pow(psi, 2 * brv + 1, m)
            acc = 0
            for c in x[i][::-1]:
                acc = (acc * pt + int(c)) % m
            assert int(got[i][k]) == acc


def test_ntt_repeated_moduli_and_more_than_128_limbs():
    N = 256
    ctx, o = hml.Context(N=N, max_level=4, alpha=2), Oracle(N, 36, 4, 2)
    idx = [i % 6 for i in range(300)]
    x = np.stack([uniform_limbs([o.moduli[i]], N, 1000 + k)[0] for k, i in enumerate(idx)])
    got = to_host(ctx.ntt(to_dev(x), idx))
    for k in (0, 127, 128, 255, 256, 299):
        assert np.array_equal(got[k], o.ntt(idx[k], x[k]))


@pytest.mark.parametrize("logN,nb", [(8, 3), (13, 5), (16, 9), (16, 1)])
def test_ntt_batch_matches_oracle(logN, nb):
    """hml_ntt_batch / hml_intt_batch: one launch pair for [n_batch][n_limbs][N], twiddles reused across the batch"""
    N = 1 << logN
    ctx, o = hml.Context(N=N, max_level=4, alpha=2), Oracle(N, 36, 4, 2)
    idx = [5, 0, 3]
    x = np.stack([np.stack([uniform_limbs([o.moduli[i]], N, 700 + 10 * b + i)[0] for i in idx]) for b in range(nb)])
    want = np.stack([np.stack([o.ntt(i, x[b][r]) for r, i in enumerate(idx)]) for b in range(nb)])
    got = to_host(ctx.ntt_batch(to_dev(x), idx))
    assert np.array_equal(got, want)
    assert np.array_equal(to_host(ctx.ntt_batch(to_dev(want), idx, inverse=True)), x)
    d = to_dev(x)
    ctx.ntt_batch(d, idx, out=d)  # in place
    assert np.array_equal(to_host(d), want)


@pytest.mark.parametrize("N", [16, 4096, 65536])
def test_ewe_variants(N):
    ctx, o = hml.Context(N=N, max_level=4, alpha=2), Oracle(N, 36, 4, 2)
    idx = [0, 3, 5]
    xs = [np.stack([uniform_limbs([o.moduli[i]], N, 200 + 10 * k + i)[0] for i in idx]) for k in range(4)]
    xs[0][0, :3] = 0
    xs[1][1, :3] = o.moduli[3] - 1
    d = [to_dev(x) for x in xs]
    cases = [((0, 1, 2, 3), False), ((0, 1, 2, 3), True), ((0, None, 2, None), False), ((0, None, 2, None), True),
             ((0, 1, None, None), False), ((0, 1, 2, None), False), ((0, None, None, None), False)]
    for sel, sub in cases:
        args = [d[s] if s is not None else None for s in sel]
        got = to_host(ctx.ewe(*args, idx, subtract=sub))
        for r, i in enumerate(idx):
            hargs = [xs[s][r] if s is not None else None for s in sel]
            assert np.array_equal(got[r], o.ewe(i, *hargs, sub=sub)), (sel, sub, i)


@pytest.mark.parametrize("N,g", [(16, 5), (4096, 25), (65536, 5), (65536, 2 * 65536 - 1), (65536, pow(5, 77, 2 * 65536))])
def test_automorphism(N, g):
    ctx, o = hml.Context(N=N, max_level=3, alpha=1), Oracle(N, 36, 3, 1)
    x = uniform_limbs(o.moduli, N, 300)
    got = to_host(ctx.automorph(to_dev(x), g))
    for i in range(4):
        assert np.array_equal(got[i], o.automorph_eval(g, x[i]))
    # against the coefficient-domain definition, through the GPU NTT
    idx = list(range(4))
    coeff = np.stack([o.automorph_coeff(i, g, x[i]) for i in idx])
    a = to_host(ctx.automorph(ctx.ntt(to_dev(x), idx), g))
    b = to_host(ctx.ntt(to_dev(coeff), idx))
    assert np.array_equal(a, b)


@pytest.mark.parametrize("N,ml,al,src,dst", [
    (16, 6, 3, [1, 2, 4], [0, 3, 5, 6, 7, 8]),
    (4096, 6, 3, [0], [1, 2, 3, 4, 5, 6, 7, 8]),
    (65536, 45, 15, list(range(15)), list(range(15, 35)) + list(range(45, 60))),  # ModUp digit 0 at L=35
    (65536, 45, 15, list(range(30, 35)), list(range(30)) + list(range(45, 60))),  # short last digit
    (65536, 45, 15, list(range(45, 60)), list(range(35))),                        # ModDown
    (32768, 28, 28, list(range(28)), list(range(28, 56))),                        # parameter set A: 28 sources
])
def test_bconv(N, ml, al, src, dst):
    ctx, o = hml.Context(N=N, max_level=ml, alpha=al), Oracle(N, 36, ml, al)
    x = np.stack([uniform_limbs([o.moduli[i]], N, 400 + i)[0] for i in src])
    x[0, :2] = o.moduli[src[0]] - 1
    got = to_host(ctx.bconv(to_dev(x), src, dst))
    check = range(len(dst)) if N <= 4096 else (0, 1, len(dst) // 2, len(dst) - 1)
    for t in check:
        assert np.array_equal(got[t], o.bconv(src, dst[t], x)), dst[t]


@pytest.mark.parametrize("N,ml,al,src,dst,nb", [
    (128, 50, 48, list(range(50, 98)), list(range(48)), 3),            # 48 -> 48: the largest shape of the tcgen05 kernel, one tile per batch
    (256, 20, 10, list(range(17)), list(range(17, 30)), 5),            # two 16-source slabs, ragged targets
    (1024, 12, 5, [0, 2, 4, 6, 8], list(range(9, 17)), 7),             # strided sources, more batches than SMs-per-tile
    (512, 60, 20, list(range(33)), list(range(33, 80)), 2),            # three slabs, 47 targets
    (256, 70, 20, list(range(10)), list(range(10, 70)), 2),            # 60 targets: above the tcgen05 limit -> FP64 tensor-core kernel
    (65536, 45, 15, list(range(45, 60)), list(range(35)), 3),          # ModDown shape, 1536 tiles on 148 persistent CTAs
])
def test_bconv_batch(N, ml, al, src, dst, nb):
    """hml_bconv_batch against the oracle: every batch, every target on the small rings (tail tiles, padding targets and
    sources, the 2- and 3-slab kernels), sampled targets at N = 2^16."""
    ctx, o = hml.Context(N=N, max_level=ml, alpha=al), Oracle(N, 36, ml, al)
    x = np.stack([np.stack([uniform_limbs([o.moduli[i]], N, 900 + 31 * b + i)[0] for i in src]) for b in range(nb)])
    x[0, 0, :2] = o.moduli[src[0]] - 1
    x[nb - 1, :, N - 1] = [o.moduli[i] - 1 for i in src]
    got = to_host(ctx.bconv_batch(to_dev(x), src, dst))
    assert got.shape == (nb, len(dst), N)
    check = range(len(dst)) if N <= 4096 else (0, 17, len(dst) - 1)
    for b in range(nb):
        for t in check:
            assert np.array_equal(got[b, t], o.bconv(src, dst[t], x[b])), (b, dst[t])


def test_bconv_tensor_core_kernels_agree_in_a_subprocess():
    """HML_BCONV_UMMA is read once per process: the same batched conversions and one hmult on the FP64 tensor-core kernel
    (child process, HML_BCONV_UMMA=0) must be bit-identical to the tcgen05 kernel's results here."""
    _tensor_core_kernels_agree(36)


def test_bconv_tensor_core_kernels_agree_in_a_subprocess_at_28_bits():
    """the same comparison with 28-bit moduli: every residue is below 2^32, so the fifth byte plane of the tcgen05 operands is
    zero"""
    _tensor_core_kernels_agree(28)


def _tensor_core_kernels_agree(w):
    """batched conversions, hmult_batch and hrotate_batch at element width w, run once with the tcgen05 conversion and once
    with the FP64 tensor-core conversion (one child process each): the results must be bit-identical"""
    import os
    import subprocess
    import sys
    import tempfile
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    body = (
        "import sys; sys.path.insert(0, %r)\n"
        "import torch, homulator_b200 as hml\n"
        "ctx = hml.Context(N=8192, max_level=12, alpha=4, element_bit_width=%d)\n"
        "L = 11\n"
        "src, dst = list(range(12, 16)), list(range(L))\n"
        "x = ctx.uniform(src, 5, lead=(6,))\n"
        "y = ctx.bconv_batch(x, src, dst)\n"
        "evk = ctx.uniform(ctx.ext_mod_idx(L), 3, lead=(ctx.beta(L), 2))\n"
        "a = ctx.uniform(list(range(L)), 1, lead=(3, 2)); b = ctx.uniform(list(range(L)), 2, lead=(3, 2))\n"
        "h = ctx.hmult_batch(L, a, b, evk); r = ctx.hrotate_batch(L, a, evk, 5)\n"
        "torch.save([y.cpu(), h.cpu(), r.cpu()], sys.argv[1])\n" % (root, w))
    outs = []
    with tempfile.TemporaryDirectory() as d:
        for flag in ("1", "0"):
            path = os.path.join(d, "o%s.pt" % flag)
            r = subprocess.run([sys.executable, "-c", body, path], env=dict(os.environ, HML_BCONV_UMMA=flag), capture_output=True,
                               text=True, timeout=600)
            assert r.returncode == 0, r.stdout + r.stderr
            outs.append(torch.load(path))
    for u, v in zip(*outs):
        assert torch.equal(u, v)


def test_errors_are_reported_not_raised_across_the_abi(big):
    ctx, _ = big
    x = ctx.empty(1, 65536)
    with pytest.raises(hml.HmlError):
        ctx.ntt(x, [60])  # modulus index out of range
    with pytest.raises(hml.HmlError):
        ctx.automorph(x, 4)  # even galois element
    with pytest.raises(hml.HmlError):
        ctx.hmult(1, x, x, x)  # L < 2
    with pytest.raises(hml.HmlError):
        ctx.hmult(46, x, x, x)  # L > maxLevel


def test_full_size_properties_without_the_oracle(big):
    """Size-independent properties at N = 2^16 over all 60 moduli: linearity of the transform, the convolution theorem on
    a monomial (multiplying by X^s is a negacyclic shift), and the batched launch shape against the single-limb one."""
    ctx, o = big
    N, idx = 65536, list(range(60))
    q = torch.tensor(o.moduli, dtype=torch.int64, device="cuda").view(60, 1)
    a, b = ctx.uniform(idx, 11), ctx.uniform(idx, 12)
    fa, fb = ctx.ntt(a, idx), ctx.ntt(b, idx)
    assert torch.equal(ctx.ntt((a + b) % q, idx), (fa + fb) % q)                      # linearity, exact mod q
    s = 12345
    mono = torch.zeros(60, N, dtype=torch.int64, device="cuda")
    mono[:, s] = 1
    prod = ctx.intt(ctx.ewe(ctx.ntt(mono, idx), fb, None, None, idx), idx)              # X^s * b in Z_q[X]/(X^N + 1)
    want = torch.cat([(q - b[:, N - s:]) % q, b[:, :N - s]], dim=1)
    assert torch.equal(prod, want)
    batch = torch.stack([a, b, (a + b) % q])
    fbatch = ctx.ntt_batch(batch[:, :50].contiguous(), idx[:50])
    assert torch.equal(fbatch[0], fa[:50]) and torch.equal(fbatch[1], fb[:50])
    assert torch.equal(ctx.ntt_batch(fbatch, idx[:50], inverse=True), batch[:, :50])
