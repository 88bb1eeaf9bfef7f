"""GPU parity on structured extreme operands.  Uniform random residues almost never drive a lazy sum to its worst case; these
operands do.  Per limb i, with h_i = (q_i - 1) / 2, every coefficient holds one of

    0, 1, q_i - 1, h_i, h_i + 1, alternating q_i - 1 / 0, alternating h_i / h_i + 1

either as given (evaluation domain) or as the forward NTT of that polynomial ("ntt:" families): then the key switch's ModUp
INTT hands the same constant to every coefficient of every conversion source (q - 1 everywhere for ntt:q-1).  A product
h * 1 reduces to +h and (h + 1) * 1 to -h, so sums of such products reach the one-signed maximum of the lazy accumulators:
k_tensor_sum's 16-pair sums, rot_sum_body's weighted sums, the HPIP row-pass accumulators, the tcgen05 epilogue's
< 2^52 shift-add at every coefficient of every tile, the DMMA conversion's 16-source folds and the row pass's centring at
(q - 1) / 2.  Ciphertexts, keys (word and packed) and plaintexts all take these families; every result is compared bit for
bit with the scalar oracle or the oracle definitions in tests/orc_*.py."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import homulator_b200 as hml  # noqa: E402
from orc import Oracle  # noqa: E402
from parity_checks import check_batched, check_bsgs, check_core, check_hmult_sum, check_hoisted, check_rotsum  # noqa: E402

# (width, N, maxLevel, alpha, L)
SHAPES = {
    # single-pass ring (logN 12 <= NTT_SMALL_LOG, ntt.cuh), beta 3: k_inner for every inner product, tcgen05 conversions
    "w36_n4096": (36, 4096, 9, 3, 8),
    # two-pass ring, beta 3: HPIP-fused inner product (context.cu ks_uses_hpip), hmult's merged ModDown + Rescale (fold)
    "w36_n8192": (36, 8192, 7, 3, 7),
    # the north star: N = 2^16, maxLevel 45, alpha 15, L 35 (HPIP, 15-source conversions with 35 targets on tcgen05)
    "w36_n65536": (36, 65536, 45, 15, 35),
    "w28_n65536": (28, 65536, 45, 15, 35),
    # alpha 20 > 16 sources at N = 256: ModUp digit 0 converts to 70 targets, the DMMA kernel, whose main loop and the hmult
    # fold reduce every 16 sources (ewe.cu k_bconv_mma)
    "w36_dmma": (36, 256, 70, 20, 70),
    # two-pass ring with 48 + 1 merged ModDown + Rescale targets (no tcgen05 image: bconv_image_shape's NP > 256): the DMMA
    # kernel with hmult's fold pre-pass; beta 7
    "w36_dmma_fold": (36, 8192, 49, 7, 49),
}

# (ciphertext a, ciphertext b and plaintexts, keys)
SCENARIOS = [
    ("h", "1", "1"),                                  # every product h * 1 = +h: one-signed maximum of every lazy sum
    ("h+1", "h+1", "1"),                              # (h + 1) * 1 = -h: the same at the negative end
    ("q-1", "q-1", "q-1"),
    ("ntt:q-1", "1", "h"),                            # c1 and d2 are NTT(q - 1): every conversion source is q - 1
    ("alt q-1/0", "alt h/h+1", "h"),
    ("ntt:h", "ntt:h+1", "h+1"),
    ("ntt:alt h/h+1", "ntt:alt q-1/0", "alt q-1/0"),
    ("0", "1", "q-1"),
    ("1", "0", "0"),
]
IDS = ["%s|%s|%s" % s for s in SCENARIOS]
# the scenarios that also run the hoisted and summed ops on the N = 2^16 shapes (the oracle definitions are numpy and slow there)
HEAVY = {0, 3}
SUM_CASES = [(shape, SCENARIOS[k]) for shape in SHAPES for k in range(len(SCENARIOS)) if SHAPES[shape][1] < 65536 or k in HEAVY]

_cache = {}


@pytest.fixture(scope="module", autouse=True)
def contexts():
    Oracle.set_threads(0)  # all host cores for the checker
    yield _cache
    for ctx, _ in _cache.values():
        ctx.close()
    _cache.clear()
    Oracle.set_threads(1)


def _get(name):
    if name not in _cache:
        w, N, ML, A, _ = SHAPES[name]
        _cache[name] = (hml.Context(N=N, max_level=ML, alpha=A, element_bit_width=w), Oracle(N, w, ML, A))
    return _cache[name]


def family(o, idx, name):
    """[len(idx)][N] with the named pattern in the limbs of moduli idx (ntt:... = the forward NTT of that pattern)"""
    q = np.array([o.moduli[i] for i in idx], dtype=np.uint64)[:, None]
    h = (q - np.uint64(1)) // np.uint64(2)
    even = (np.arange(o.N) % 2 == 0)[None, :]
    base = name[4:] if name.startswith("ntt:") else name
    zero = np.zeros((len(idx), o.N), dtype=np.uint64)
    v = {"0": zero, "1": zero + np.uint64(1), "q-1": zero + q - np.uint64(1), "h": zero + h, "h+1": zero + h + np.uint64(1),
         "alt q-1/0": np.where(even, q - np.uint64(1), np.uint64(0)), "alt h/h+1": np.where(even, h, h + np.uint64(1))}[base]
    v = np.ascontiguousarray(v.astype(np.uint64))
    if name.startswith("ntt:"):
        v = np.stack([o.ntt(i, v[r]) for r, i in enumerate(idx)])
    return v


def operands(o, L, evk_q, fa, fb, fk):
    """ciphertexts a, b [2][L][N], a key [beta][2][evk_q + alpha][N] and a plaintext [L + alpha][N]"""
    ML, A = o.max_level, o.alpha
    beta = -(-L // A)
    q_idx = list(range(L))
    a = np.ascontiguousarray(np.stack([family(o, q_idx, fa)] * 2))
    b = np.ascontiguousarray(np.stack([family(o, q_idx, fb)] * 2))
    key = np.ascontiguousarray(np.stack([np.stack([family(o, list(range(evk_q)) + list(range(ML, ML + A)), fk)] * 2)] * beta))
    pt = family(o, o.ext_mod_idx(L), fb)
    return a, b, key, pt


@pytest.mark.parametrize("scenario", SCENARIOS, ids=IDS)
@pytest.mark.parametrize("shape", list(SHAPES))
def test_extreme_keyswitch_rescale_hmult_hrotate(shape, scenario):
    """keyswitch, rescale, hmult, hrotate (word and packed keys, key laid out for L and for maxLevel on the small rings), and the
    batched hmult / hrotate"""
    ctx, o = _get(shape)
    L, ML = SHAPES[shape][4], o.max_level
    for evk_q in ((L, ML) if o.N <= 8192 and ML != L else (L,)):
        a, b, key, _ = operands(o, L, evk_q, *scenario)
        want_m, want_r = check_core(ctx, o, L, a, b, key, evk_q, g=5)
        if evk_q == L:
            check_batched(ctx, o, L, a, b, key, evk_q, want_m, want_r, g=5)


@pytest.mark.parametrize("shape,scenario", SUM_CASES, ids=["%s-%s|%s|%s" % ((c[0],) + c[1]) for c in SUM_CASES])
def test_extreme_hoisted_and_summed_ops(shape, scenario):
    """hrotate_hoisted, hrotate_sum_hoisted with 16 rotations (one full group) and 17 (a second, accumulating launch),
    hrotate_bsgs_hoisted with identity baby and giant steps, and hmult_sum of 1, 16, 17 and 33 identical terms (first and
    accumulating k_tensor_sum launches) and of 17 identical squares"""
    ctx, o = _get(shape)
    big = o.N == 65536
    L, N = SHAPES[shape][4], o.N
    a, b, key, pt = operands(o, L, L, *scenario)
    gs = [pow(5, r, 2 * N) for r in range(1, 18)]
    check_hoisted(ctx, o, L, a, [key] * 3, L, [5, 25, 2 * N - 1])
    for n in ((17,) if big else (16, 17)):
        check_rotsum(ctx, o, L, a, [key] * n, L, gs[:n], [pt] * n, L)
    babies, giants = [1, 5, 25], [1, 125, 2 * N - 1]
    keys = {1: None, 5: key, 25: key, 125: key, 2 * N - 1: key}
    check_bsgs(ctx, o, L, a, babies, giants, keys, L, [[pt] * 3] * 3, L)
    for n in ((1, 17) if big else (1, 16, 17, 33)):
        check_hmult_sum(ctx, o, L, [a] * n, [b] * n, key, L)
    check_hmult_sum(ctx, o, L, [a] * 17, [a] * 17, key, L)

