"""Batched hmult on two-pass rings, where the tensor product runs inside the key switch: d2 = a1 * b1 is formed on the
ModUp transform's load, and the inner product forms d0 = a0 * b0, d1 = a0 * b1 + a1 * b0 itself and folds them into its
accumulators as d_c * P.  Checked bit-exactly against the oracle and against the one-ciphertext path, which still stores
d0, d1 and d2, at levels with one, two and three digits (full and short last digits), across chunk boundaries, with packed
keys and keys of a higher level, and through the host-buffer entry points."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import homulator_b200 as hml  # noqa: E402
from gpu_common import to_dev, to_host  # noqa: E402
from orc import Oracle, uniform_limbs  # noqa: E402

# (N, maxLevel, alpha) and levels: one digit, two digits with a short last one, three digits with a short last one, three full
RINGS = {"n8192": ((8192, 9, 3), (3, 5, 8, 9)), "north_star": ((65536, 45, 15), (15, 16, 35, 45))}


@pytest.fixture(scope="module", params=list(RINGS))
def ring(request):
    (N, ML, A), levels = RINGS[request.param]
    Oracle.set_threads(0)  # all host cores for the checker
    ctx, o = hml.Context(N=N, max_level=ML, alpha=A), Oracle(N, 36, ML, A)
    yield ctx, o, levels
    ctx.close()
    Oracle.set_threads(1)


def _pool(o, L, seed, k=4):
    """k distinct seeded ciphertexts, host [k][2][L][N]"""
    return np.stack([uniform_limbs(o.moduli[:L], o.N, seed + i, lead=(2,)) for i in range(k)])


def _key(o, L, evk_q, seed):
    beta = -(-L // o.alpha)
    return uniform_limbs(o.moduli[:evk_q] + o.moduli[o.max_level:], o.N, seed, lead=(beta, 2))


def _pairs(pool_dev, n):
    """n ciphertext pairs from the pool (neighbours in the batch differ)"""
    k = pool_dev.shape[0]
    ia = [i % k for i in range(n)]
    ib = [(i + 1 + i // k) % k for i in range(n)]
    return pool_dev[ia], pool_dev[ib], ia, ib


def _singles(ctx, L, A, B, K, idx, kq=None):
    return torch.stack([ctx.hmult(L, A[i], B[i], K, evk_q_limbs=kq) for i in idx])


@pytest.mark.parametrize("li", range(4))
def test_batch_vs_oracle_and_single(ring, li):
    ctx, o, levels = ring
    L = levels[li]
    pool = _pool(o, L, 2000 + L)
    evk = _key(o, L, L, 2100 + L)
    P, K = to_dev(pool), to_dev(evk)
    A, B, ia, ib = _pairs(P, 5)
    got = ctx.hmult_batch(L, A, B, K)
    assert torch.equal(got, _singles(ctx, L, A, B, K, range(5)))
    for i in (0, 3):
        assert np.array_equal(to_host(got[i]), o.hmult(L, pool[ia[i]], pool[ib[i]], evk, L)), (L, i)


@pytest.mark.parametrize("n", [65, 70])
def test_partial_last_chunk(ring, n):
    """chunks of 64: 65 leaves one ciphertext for the last chunk (the one-ciphertext schedule), 70 leaves six"""
    ctx, o, levels = ring
    L = levels[2]
    pool = _pool(o, L, 2200)
    K = to_dev(_key(o, L, L, 2300))
    A, B, _, _ = _pairs(to_dev(pool), n)
    got = ctx.hmult_batch(L, A, B, K)
    idx = [0, 1, 62, 63, 64, n - 1]
    assert torch.equal(got[idx], _singles(ctx, L, A, B, K, idx))


def test_packed_and_higher_level_keys(ring):
    """a key generated for maxLevel (evk_q_limbs > L), as words and packed"""
    ctx, o, levels = ring
    L, ML = levels[2], o.max_level
    pool = _pool(o, L, 2400)
    evk = _key(o, L, ML, 2500)
    K = to_dev(evk)
    A, B, ia, ib = _pairs(to_dev(pool), 4)
    got = ctx.hmult_batch(L, A, B, K, evk_q_limbs=ML)
    assert torch.equal(got, _singles(ctx, L, A, B, K, range(4), ML))
    assert np.array_equal(to_host(got[1]), o.hmult(L, pool[ia[1]], pool[ib[1]], evk, ML))
    assert torch.equal(ctx.hmult_batch(L, A, B, ctx.key_pack(K), evk_q_limbs=ML | hml.KEY_PACKED), got)


def test_host_entry_points(ring):
    """hml_hmult_host and hml_hmult_host_packed run the batched schedule per chunk"""
    ctx, o, levels = ring
    L, N, n = levels[2], o.N, 11
    A, B, _, _ = _pairs(to_dev(_pool(o, L, 2600)), n)
    K = to_dev(_key(o, L, L, 2700))
    want = ctx.hmult_batch(L, A, B, K).cpu()
    assert torch.equal(want[[0, 5, 10]], _singles(ctx, L, A, B, K, (0, 5, 10)).cpu())
    ah, bh = A.cpu().pin_memory(), B.cpu().pin_memory()
    oh = torch.empty(n, 2, L - 1, N, dtype=torch.int64).pin_memory()
    ctx.hmult_host(L, ah, bh, K, oh)
    assert torch.equal(oh, want)
    op = torch.empty(n * 2 * (L - 1) * 5 * N, dtype=torch.uint8).pin_memory()
    ctx.hmult_host_packed(L, n, ctx.pack_host(ah), ctx.pack_host(bh), K, op)
    assert torch.equal(ctx.unpack_host(op, oh.shape), want)
