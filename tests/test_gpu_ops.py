"""GPU parity, composite ops: keyswitch / rescale / hmult / hrotate / hadd / pmult / padd against the oracle,
bit-exact, at small sizes (both oracle tiers) and at BASELINE.json's full sizes."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import homulator_b200 as hml  # noqa: E402
from gpu_common import to_dev, to_host  # noqa: E402
from orc import Oracle, uniform_limbs  # noqa: E402


def make_case(o, L, evk_q, seed, n_ct=2):
    N, ML = o.N, o.max_level
    beta = -(-L // o.alpha)
    cts = [uniform_limbs(o.moduli[:L], N, seed + k, lead=(2,)) for k in range(n_ct)]
    evk = uniform_limbs(o.moduli[:evk_q] + o.moduli[ML:], N, seed + 9, lead=(beta, 2))
    return cts, evk


# (N, maxLevel, L, alpha): beta = 1, L % alpha != 0, L < alpha, L = 1 (hrotate only), several digits
SMALL = [(16, 6, 6, 2), (16, 6, 5, 2), (16, 5, 2, 3), (64, 4, 4, 4), (256, 7, 7, 3), (1024, 3, 1, 2), (4096, 9, 8, 3)]


@pytest.mark.parametrize("N,ML,L,A", SMALL)
def test_keyswitch_and_hrotate_small(N, ML, L, A):
    ctx, o = hml.Context(N=N, max_level=ML, alpha=A), Oracle(N, 36, ML, A)
    for evk_q in sorted({L, ML}):
        (ct, _), evk = make_case(o, L, evk_q, 500)
        for direct in ((0, 1) if N <= 256 else (0,)):
            o.set_direct(direct)
            w0, w1 = o.keyswitch(L, ct[0], evk, evk_q)
            g0, g1 = ctx.keyswitch(L, to_dev(ct[0]), to_dev(evk), evk_q)
            assert np.array_equal(to_host(g0), w0) and np.array_equal(to_host(g1), w1)
            for g in (5, 2 * N - 1):
                want = o.hrotate(L, ct, evk, evk_q, g)
                got = to_host(ctx.hrotate(L, to_dev(ct), to_dev(evk), g, evk_q))
                assert np.array_equal(got, want)
        o.set_direct(0)


@pytest.mark.parametrize("N,ML,L,A", [c for c in SMALL if c[2] >= 2])
def test_rescale_and_hmult_small(N, ML, L, A):
    ctx, o = hml.Context(N=N, max_level=ML, alpha=A), Oracle(N, 36, ML, A)
    (a, b), evk = make_case(o, L, L, 600)
    assert np.array_equal(to_host(ctx.rescale(L, to_dev(a[0]))), o.rescale(L, a[0]))
    for direct in ((0, 1) if N <= 256 else (0,)):
        o.set_direct(direct)
        want = o.hmult(L, a, b, evk, L)
        got = to_host(ctx.hmult(L, to_dev(a), to_dev(b), to_dev(evk)))
        assert np.array_equal(got, want)
    o.set_direct(0)


def test_hadd_pmult_padd():
    N, ML, A, L = 4096, 5, 2, 4
    ctx, o = hml.Context(N=N, max_level=ML, alpha=A), Oracle(N, 36, ML, A)
    (a, b), _ = make_case(o, L, L, 700)
    pt = b[0]
    assert np.array_equal(to_host(ctx.hadd(L, to_dev(a), to_dev(b))), o.hadd(L, a, b))
    assert np.array_equal(to_host(ctx.pmult(L, to_dev(a), to_dev(pt))), o.pmult(L, a, pt))
    assert np.array_equal(to_host(ctx.padd(L, to_dev(a), to_dev(pt))), o.padd(L, a, pt))
    # PMULT followed by HADD in one pass (hml_pmult_add), also in place on the addend
    want = o.hadd(L, o.pmult(L, a, pt), b)
    assert np.array_equal(to_host(ctx.pmult_add(L, to_dev(a), to_dev(pt), to_dev(b))), want)
    acc = to_dev(b)
    ctx.pmult_add(L, to_dev(a), to_dev(pt), acc, out=acc)
    assert np.array_equal(to_host(acc), want)


def test_evk_all_zero_gives_zero_keyswitch():
    N, ML, A, L = 8192, 6, 2, 5
    ctx = hml.Context(N=N, max_level=ML, alpha=A)
    d = ctx.uniform(list(range(L)), 1)
    evk = torch.zeros(3, 2, L + A, N, dtype=torch.int64, device="cuda")
    o0, o1 = ctx.keyswitch(L, d, evk)
    assert int(o0.abs().max()) == 0 and int(o1.abs().max()) == 0


@pytest.fixture(scope="module")
def north_star():
    Oracle.set_threads(0)  # all host cores for the checker; results do not depend on it (tests/test_oracle.py)
    ctx, o = hml.Context(N=65536, max_level=45, alpha=15), Oracle(65536, 36, 45, 15)
    (a, b), evk = make_case(o, 35, 35, 800)
    yield ctx, o, a, b, evk
    Oracle.set_threads(1)


def test_hmult_north_star_bit_exact(north_star):
    """BASELINE.json configs[0]: hmult, config_4.cfg, maxLevel 45, L 35, alpha 15."""
    ctx, o, a, b, evk = north_star
    want = o.hmult(35, a, b, evk, 35)
    got = to_host(ctx.hmult(35, to_dev(a), to_dev(b), to_dev(evk)))
    assert got.shape == (2, 34, 65536)
    assert np.array_equal(got, want)
    # executed-vs-trace bookkeeping (SURVEY.md 3.5): D3 elides 35 NTTs; ModDown is merged with Rescale by linearity of the
    # NTT (DESIGN.md 3.2): the 70 ModDown NTTs and the 68 Rescale NTTs become 68 transforms; the base conversion gains the
    # rescale remainder as a 16th source: 1275 (ModUp) + 2 * 16 * 34
    ctx.exec_counts(reset=True)
    ctx.hmult(35, to_dev(a), to_dev(b), to_dev(evk))
    ex = ctx.exec_counts()
    assert ex["ntt_limbs"] == 115 + 68 and ex["intt_limbs"] == 35 + 30 + 2
    assert ex["bconv_limb_macs"] == 1275 + 2 * 16 * 34
    tr = ctx.counts("hmult", 35)
    assert (tr["NTT"] + tr["INTT"]) // 256 == 289


def test_hrotate_north_star_bit_exact(north_star):
    """BASELINE.json configs[1]: hrotate, config_4.cfg, maxLevel 45, L 35, alpha 15, r=1 (g=5)."""
    ctx, o, a, b, evk = north_star
    want = o.hrotate(35, a, evk, 35, 5)
    got = to_host(ctx.hrotate(35, to_dev(a), to_dev(evk), 5))
    assert np.array_equal(got, want)


def test_hmult_full_level_key_layout(north_star):
    """key laid out for maxLevel (evk_q_limbs = 45) used at L = 20: beta = 2, last digit short."""
    ctx, o, a, b, _ = north_star
    L = 20
    evk = uniform_limbs(o.moduli, 65536, 900, lead=(2, 2))
    a20, b20 = np.ascontiguousarray(a[:, :L]), np.ascontiguousarray(b[:, :L])
    want = o.hmult(L, a20, b20, evk, 45)
    got = to_host(ctx.hmult(L, to_dev(a20), to_dev(b20), to_dev(evk), evk_q_limbs=45))
    assert np.array_equal(got, want)


def test_parameter_set_A_N15_beta1():
    """BASELINE.json configs[2]: config_4_N15.cfg (N=32768), maxLevel 28, alpha 28, levels 28 / 14 / 2."""
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    Oracle.set_threads(0)
    ctx, o = hml.Context(os.path.join(root, "config", "config_4_N15.cfg"), 28, 28), Oracle(32768, 36, 28, 28)
    assert ctx.N == 32768
    for L in (28, 14, 2):
        (a, b), evk = make_case(o, L, L, 1000 + L)
        want = o.hmult(L, a, b, evk, L)
        got = to_host(ctx.hmult(L, to_dev(a), to_dev(b), to_dev(evk)))
        assert np.array_equal(got, want), L
    Oracle.set_threads(1)


def test_batch_and_host_paths_equal_single_calls(north_star):
    ctx, o, a, b, evk = north_star
    L, n = 35, 3
    A = torch.stack([to_dev(a), to_dev(b), to_dev(a)])
    B = torch.stack([to_dev(b), to_dev(b), to_dev(a)])
    K = to_dev(evk)
    singles = torch.stack([ctx.hmult(L, A[i], B[i], K) for i in range(n)])
    assert torch.equal(ctx.hmult_batch(L, A, B, K), singles)
    ah, bh = A.cpu().pin_memory(), B.cpu().pin_memory()
    oh = torch.empty(n, 2, L - 1, 65536, dtype=torch.int64).pin_memory()
    ctx.hmult_host(L, ah, bh, K, oh)
    assert torch.equal(oh, singles.cpu())
    rs = torch.stack([ctx.hrotate(L, A[i], K, 5) for i in range(n)])
    assert torch.equal(ctx.hrotate_batch(L, A, K, 5), rs)
    rh = torch.empty(n, 2, L, 65536, dtype=torch.int64).pin_memory()
    ctx.hrotate_host(L, ah, K, rh, 5)
    assert torch.equal(rh, rs.cpu())


def test_op_objects_mirror_reference_constructor(north_star):
    ctx, *_ = north_star
    op = hml.HMULT("test_hmult", 45, 35, 15, ctx)
    assert op.counts["total"] == 834560 and op.counts["driverTotal"] == 7381760
    r = op.simulate(iters=2, warmup=1)
    assert r["us_median"] > 0
    rot = hml.HROTATE("test_hrotate", 45, 35, 15, ctx)
    assert rot.counts["AUTO"] == 17920 and rot.counts["total"] == 780800


def _oracle_replay(o, L, trace, x, pts, keys, evk, hoist=False):
    """the same trace on the oracle (keys laid out for level L; a slot's level is its limb count); hoist=True groups
    consecutive rotations of one source exactly as hml_replay does"""
    N = o.N
    h = {"x": x}
    lv = lambda name: h[name].shape[1]  # noqa: E731
    i = 0
    while i < len(trace):
        op = trace[i]
        if op[0] == "hrotate":
            j = i
            if hoist:
                while j < len(trace) and trace[j][0] == "hrotate" and trace[j][2] == op[2] and trace[j][1] != op[2] \
                        and trace[j][1] not in [t[1] for t in trace[i:j]]:
                    j += 1
            if j - i >= 2:
                outs = o.hrotate_hoisted(lv(op[2]), h[op[2]], [keys[t[3]] for t in trace[i:j]], L, [pow(5, t[3], 2 * N) for t in trace[i:j]])
                for t, out in zip(trace[i:j], outs):
                    h[t[1]] = out
                i = j
                continue
            h[op[1]] = o.hrotate(lv(op[2]), h[op[2]], keys[op[3]], L, pow(5, op[3], 2 * N))
        elif op[0] == "pmult":
            h[op[1]] = o.pmult(lv(op[2]), h[op[2]], np.ascontiguousarray(pts[op[3]][:lv(op[2])]))
        elif op[0] == "padd":
            h[op[1]] = o.padd(lv(op[2]), h[op[2]], np.ascontiguousarray(pts[op[3]][:lv(op[2])]))
        elif op[0] == "hadd":
            h[op[1]] = o.hadd(lv(op[2]), h[op[2]], h[op[3]])
        elif op[0] == "hmult":
            h[op[1]] = o.hmult(lv(op[2]), h[op[2]], h[op[3]], evk, L)
        i += 1
    return h


def test_replay_across_levels():
    """a trace that goes on from hmult results: two chained multiplications with rotations, plaintext ops and additions at
    the lower levels (keys laid out for the top level serve every level; a plaintext's first limbs serve the lower ones)"""
    N, ML, A, L = 8192, 7, 3, 7
    ctx, o = hml.Context(N=N, max_level=ML, alpha=A), Oracle(N, 36, ML, A)
    Oracle.set_threads(0)
    beta = -(-L // A)
    trace = [("hrotate", "a", "x", 1), ("hmult", "b", "a", "x"),          # b at L-1
             ("hrotate", "c", "b", 2), ("pmult", "d", "c", 0), ("hadd", "e", "d", "b"), ("padd", "e", "e", 1),
             ("hmult", "f", "e", "b"),                                    # f at L-2
             ("hrotate", "g", "f", 1), ("hrotate", "h", "f", 2), ("hadd", "g", "g", "h")]
    x = uniform_limbs(o.moduli[:L], N, 1, lead=(2,))
    pts = {i: uniform_limbs(o.moduli[:L], N, 100 + i) for i in range(2)}
    keys = {r: uniform_limbs(o.moduli[:L] + o.moduli[ML:], N, 200 + r, lead=(beta, 2)) for r in (1, 2)}
    evk = uniform_limbs(o.moduli[:L] + o.moduli[ML:], N, 300, lead=(beta, 2))
    dx, dp, dk, de = to_dev(x), {k: to_dev(v) for k, v in pts.items()}, {k: to_dev(v) for k, v in keys.items()}, to_dev(evk)
    for graph, hoist in ((False, False), (True, False), (True, True)):
        want = _oracle_replay(o, L, trace, x, pts, keys, evk, hoist=hoist)
        rp = hml.Replay(ctx, L, trace, graph=graph, hoist=hoist).bind(dx, dp, dk, de)
        for _ in range(2):
            rp.run()
        for name in ("b", "e", "f", "g"):
            got = to_host(rp.result(name))
            assert got.shape == want[name].shape and np.array_equal(got, want[name]), (name, graph, hoist)
        rp.close()
    Oracle.set_threads(1)


@pytest.mark.parametrize("N,ML,A,L,shape", [(2048, 6, 2, 5, "bsgs"), (8192, 6, 2, 5, "bsgs"), (8192, 7, 3, 7, "rotsum")])
def test_op_sequence_replay_matches_oracle(N, ML, A, L, shape):
    """BASELINE.json configs[4]: synthetic rotation-heavy sequences replayed through hml_replay_* — plain launches, one CUDA
    graph (run twice: the graph must replay), and with hoisted rotations against the oracle's own hoisted definition."""
    from homulator_b200.replay import bsgs_trace, rotsum_trace, trace_counts
    ctx, o = hml.Context(N=N, max_level=ML, alpha=A), Oracle(N, 36, ML, A)
    Oracle.set_threads(0)
    beta = -(-L // A)
    trace = bsgs_trace(3, 2) if shape == "bsgs" else rotsum_trace(5)
    cnt = trace_counts(trace)
    assert cnt["hmult"] == 1 and cnt["hrotate"] == (3 if shape == "bsgs" else 5)
    rots = sorted({op[3] for op in trace if op[0] == "hrotate"})
    x = uniform_limbs(o.moduli[:L], N, 1, lead=(2,))
    pts = {i: uniform_limbs(o.moduli[:L], N, 100 + i) for i in range(6)}
    keys = {r: uniform_limbs(o.moduli[:L] + o.moduli[ML:], N, 200 + r, lead=(beta, 2)) for r in rots}
    evk = uniform_limbs(o.moduli[:L] + o.moduli[ML:], N, 300, lead=(beta, 2))
    dx, dp, dk, de = to_dev(x), {k: to_dev(v) for k, v in pts.items()}, {k: to_dev(v) for k, v in keys.items()}, to_dev(evk)
    want = _oracle_replay(o, L, trace, x, pts, keys, evk)
    want_h = _oracle_replay(o, L, trace, x, pts, keys, evk, hoist=True)
    assert not np.array_equal(want["z"], want_h["z"])   # hoisting is a different (equally valid) function bit for bit
    for graph in (False, True):
        for hoist in (False, True):
            rp = hml.Replay(ctx, L, trace, graph=graph, hoist=hoist).bind(dx, dp, dk, de)
            for _ in range(3 if graph else 1):
                rp.run()
            w = want_h if hoist else want
            assert np.array_equal(to_host(rp.result("y")), w["y"]), (graph, hoist)
            assert np.array_equal(to_host(rp.result("z")), w["z"]), (graph, hoist)
            rp.close()
    Oracle.set_threads(1)


def test_replay_rejects_malformed_traces():
    ctx = hml.Context(N=1024, max_level=4, alpha=2)
    for bad in ([("hadd", "y", "nope", "x")], [("hmult", "z", "x", "x"), ("hadd", "w", "z", "x")], [("hmult", "x2", "x", "x"), ("hmult", "x2", "x2", "x2")]):
        with pytest.raises((hml.HmlError, ValueError)):
            hml.Replay(ctx, 3, bad)
    rp = hml.Replay(ctx, 3, [("hrotate", "a", "x", 1)])
    x = ctx.uniform([0, 1, 2], 1, lead=(2,))
    with pytest.raises(hml.HmlError):
        rp.bind(x, {}, {}, None)       # rotation 1 has no key
    with pytest.raises(hml.HmlError):
        rp.run()                       # not bound
    rp.close()


def test_hoisted_rotations_north_star(north_star):
    """hml_hrotate_hoisted at BASELINE.json's config: 4 rotations of one ciphertext sharing one ModUp, bit-exact against the
    oracle's hoisted definition (and different from the textbook rotation, which stays pinned by its own test)."""
    ctx, o, a, b, evk = north_star
    L, N = 35, 65536
    gs = [pow(5, r, 2 * N) for r in (1, 2, 7)] + [2 * N - 1]
    rks = [evk, uniform_limbs(o.moduli[:L] + o.moduli[45:], N, 811, lead=(3, 2)), evk, evk]
    want = o.hrotate_hoisted(L, a, rks, L, gs)
    dk = [to_dev(k) for k in rks]
    got = ctx.hrotate_hoisted(L, to_dev(a), dk, gs)
    for w, g in zip(want, got):
        assert np.array_equal(to_host(g), w)
    assert not np.array_equal(want[0], o.hrotate(L, a, evk, L, gs[0]))


@pytest.mark.parametrize("N,ML,A,L", [(65536, 24, 6, 24), (65536, 26, 9, 26), (65536, 26, 9, 11), (16384, 12, 4, 9)])
def test_parameter_sets_B_C_two_pass_rings(N, ML, A, L):
    """SURVEY.md 8f rank 2: the reference's other parameter sets (alpha 6 / beta 4, alpha 9 / beta 3) plus shapes with
    L % alpha != 0 and alpha % 4 == 0, on two-pass rings: hmult takes the merged ModDown + Rescale path with 7, 10 and 5
    conversion sources (padding to 8, 12, 8), hrotate the textbook one."""
    Oracle.set_threads(0)
    ctx, o = hml.Context(N=N, max_level=ML, alpha=A), Oracle(N, 36, ML, A)
    (a, b), evk = make_case(o, L, L, 1300 + L)
    got = to_host(ctx.hmult(L, to_dev(a), to_dev(b), to_dev(evk)))
    assert np.array_equal(got, o.hmult(L, a, b, evk, L))
    got = to_host(ctx.hrotate(L, to_dev(a), to_dev(evk), 5))
    assert np.array_equal(got, o.hrotate(L, a, evk, L, 5))
    Oracle.set_threads(1)


def test_small_chunks_in_a_subprocess():
    """HML_BATCH_CHUNK is read once per process: run a 7-ciphertext batch with chunks of 2 in a child process and compare
    with single calls."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = (
        "import sys; sys.path.insert(0, %r)\n"
        "import torch, homulator_b200 as hml\n"
        "ctx = hml.Context(N=8192, max_level=6, alpha=2)\n"
        "L, n = 5, 7\n"
        "q = list(range(L))\n"
        "evk = ctx.uniform(ctx.ext_mod_idx(L), 3, lead=(3, 2))\n"
        "a = ctx.uniform(q, 1, lead=(n, 2)); b = ctx.uniform(q, 2, lead=(n, 2))\n"
        "for rep in range(3):\n"
        "    got = ctx.hmult_batch(L, a, b, evk)\n"
        "    rot = ctx.hrotate_batch(L, a, evk, 5)\n"
        "torch.cuda.synchronize()\n"
        "assert torch.equal(got, torch.stack([ctx.hmult(L, a[i], b[i], evk) for i in range(n)]))\n"
        "assert torch.equal(rot, torch.stack([ctx.hrotate(L, a[i], evk, 5) for i in range(n)]))\n"
        "print('chunks ok')\n" % root)
    env = dict(os.environ, HML_BATCH_CHUNK="2")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "chunks ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.parametrize("n", [1, 8, 35, 70])
def test_batch_chunking_small(n):
    """hml_*_batch runs up to 64 ciphertexts per launch: cover partial chunks and a full + partial chunk."""
    N, ML, A, L = 2048, 7, 3, 7
    ctx, o = hml.Context(N=N, max_level=ML, alpha=A), Oracle(N, 36, ML, A)
    (a, b), evk = make_case(o, L, L, 1200)
    q = list(range(L))
    As = torch.stack([to_dev(a) if i % 2 == 0 else to_dev(b) for i in range(n)])
    Bs = ctx.uniform(q, 77, lead=(n, 2))
    K = to_dev(evk)
    got = ctx.hmult_batch(L, As, Bs, K)
    for i in (0, n // 2, n - 1):
        want = o.hmult(L, to_host(As[i]), to_host(Bs[i]), evk, L)
        assert np.array_equal(to_host(got[i]), want), i
    rot = ctx.hrotate_batch(L, Bs, K, 25)
    for i in (0, n - 1):
        assert np.array_equal(to_host(rot[i]), o.hrotate(L, to_host(Bs[i]), evk, L, 25)), i


def test_invalid_key_layout_is_rejected():
    ctx = hml.Context(N=1024, max_level=6, alpha=2)
    x = ctx.uniform(list(range(4)), 1, lead=(2,))
    evk = ctx.uniform(ctx.ext_mod_idx(4), 2, lead=(2, 2))
    with pytest.raises(hml.HmlError):
        ctx.hmult(4, x, x, evk, evk_q_limbs=3)   # fewer Q-limbs in the key than the level needs
    with pytest.raises(hml.HmlError):
        ctx.hmult(4, x, x, evk, evk_q_limbs=7)   # more than maxLevel


def test_buffer_plan_follows_reference_names(north_star):
    """reference AddrManage::MallocMem (include/Addr.h:29-48) prints one `Malloc <name> from A to B` line per intermediate,
    addresses in units of batchSize per limb; hml_buffer_plan does the same for the device workspace"""
    ctx, *_ = north_star
    plan = ctx.buffer_plan("hmult", 35).splitlines()
    assert plan[0] == "Malloc TensorD0Out from 0 to %d" % (34 * 256)
    assert plan[1] == "Malloc TensorD1Out from %d to %d" % (35 * 256, 69 * 256)
    assert any(l.startswith("Malloc ModUpINTTOut from") for l in plan)
    assert sum(l.startswith("Malloc BConvOut_(") for l in plan) == 3          # beta = 3 digits of 50 limbs
    assert sum(l.startswith("Malloc InnerProduceOut_Key") for l in plan) == 2
    last = int(plan[-1].split()[-1]) // 256 + 1                                # limbs used by the plan
    assert last == 3 * 35 + 35 + 3 * 50 + 2 * 51 + 2 * 34
    rot = ctx.buffer_plan("hrotate", 35)
    assert rot.startswith("Malloc AUTOOutput(0) from 0 to") and "NTTOut_ModDown_Key1" in rot
    with pytest.raises(hml.HmlError):
        ctx.buffer_plan("nonsense", 35)


def test_parameter_set_sweep_module(tmp_path):
    """python -m homulator_b200.sweep walks the reference's benchmark matrix (script/para*/micro24_*.sh): a thinned set-A
    sweep must log one file per (op, level) under the reference's outLogs layout and summarise them"""
    from homulator_b200 import sweep
    rows = sweep.run(["A"], ["hmult", "padd"], 13, 1, str(tmp_path / "outLogs"), str(tmp_path / "sweep.md"))
    assert [(r["op"], r["L"]) for r in rows] == [("hmult", 28), ("hmult", 15), ("hmult", 2), ("padd", 28), ("padd", 15), ("padd", 2)]
    assert all(r["us_median"] > 0 and r["N"] == 32768 for r in rows)
    assert rows[0]["trace_total"] == 390656  # SURVEY.md 8a golden: config_4_N15 hmult 28 28 28
    assert (tmp_path / "outLogs" / "paraA" / "gpu" / "hmult" / "28_28" / "hmult_28_28_15.log").exists()
    assert "## Set A" in (tmp_path / "sweep.md").read_text()


def test_repeatability_stress(north_star):
    """The kernels synchronise with warp-level barriers, cp.async groups, mbarriers and programmatic dependent launch;
    a missing ordering would show up as run-to-run differences.  Repeat single and batched ops back to back (no host
    synchronisation in between) and demand bit-identical results."""
    ctx, o, a, b, evk = north_star
    L, n = 35, 5
    A = torch.stack([to_dev(a if i % 2 == 0 else b) for i in range(n)])
    B = torch.stack([to_dev(b if i % 3 == 0 else a) for i in range(n)])
    K = to_dev(evk)
    ref_m, ref_r = ctx.hmult_batch(L, A, B, K), ctx.hrotate_batch(L, A, K, 5)
    ref_1 = ctx.hmult(L, A[1], B[1], K)
    assert torch.equal(ref_m[1], ref_1)
    outs = []
    for _ in range(8):
        outs.append((ctx.hmult_batch(L, A, B, K), ctx.hrotate_batch(L, A, K, 5), ctx.hmult(L, A[1], B[1], K)))
    torch.cuda.synchronize()
    for m, r, s1 in outs:
        assert torch.equal(m, ref_m) and torch.equal(r, ref_r) and torch.equal(s1, ref_1)


def test_hmult_is_commutative_bitwise(north_star):
    """d0 = a0 b0, d1 = a0 b1 + a1 b0, d2 = a1 b1 are symmetric in (a, b) and everything after the tensor product is a
    function of (d0, d1, d2): hmult(a, b) and hmult(b, a) must agree bit for bit, single and batched."""
    ctx, o, a, b, evk = north_star
    A, B, K = to_dev(a), to_dev(b), to_dev(evk)
    assert torch.equal(ctx.hmult(35, A, B, K), ctx.hmult(35, B, A, K))
    AB, BA = torch.stack([A, B, A]), torch.stack([B, A, A])
    assert torch.equal(ctx.hmult_batch(35, AB, BA, K), ctx.hmult_batch(35, BA, AB, K))


@pytest.mark.parametrize("N,ML,A,L", [(8192, 6, 2, 5), (8192, 6, 2, 2), (32768, 8, 3, 8), (65536, 45, 15, 35), (65536, 45, 15, 2)])
def test_rescale_and_keyswitch_standalone_two_pass_rings(N, ML, A, L):
    """hml_rescale / hml_keyswitch on two-pass rings (N >= 8192) take their own code paths (ntt_rows<0,1> with no z / cst2
    for the rescale, the textbook K8-K10 for the key switch): compare them with the oracle directly, not only through
    hmult / hrotate (reference Rescale src/Operation.cpp:741-911, KeySwitch :9-54)."""
    Oracle.set_threads(0)
    ctx, o = hml.Context(N=N, max_level=ML, alpha=A), Oracle(N, 36, ML, A)
    (a, b), evk = make_case(o, L, L, 1500 + L)
    for poly in (a[0], a[1], b[1]):
        assert np.array_equal(to_host(ctx.rescale(L, to_dev(poly))), o.rescale(L, poly))
    w0, w1 = o.keyswitch(L, b[0], evk, L)
    g0, g1 = ctx.keyswitch(L, to_dev(b[0]), to_dev(evk), L)
    assert np.array_equal(to_host(g0), w0) and np.array_equal(to_host(g1), w1)
    Oracle.set_threads(1)


def test_hmult_many_special_primes_dmma_fold():
    """alpha = 50 > 48 sources: the merged ModDown + Rescale of hmult falls off the tcgen05 kernel onto the FP64 tensor-core
    kernel, whose fold pre-pass sums alpha products of < 2^48 — more than the 16 an exact double sum can hold unreduced
    (ADVICE r1: the fold must reduce every 16 terms like the main loop)."""
    N, ML, A, L = 8192, 4, 50, 3
    Oracle.set_threads(0)
    ctx, o = hml.Context(N=N, max_level=ML, alpha=A), Oracle(N, 36, ML, A)
    (a, b), evk = make_case(o, L, L, 1700)
    assert np.array_equal(to_host(ctx.hmult(L, to_dev(a), to_dev(b), to_dev(evk))), o.hmult(L, a, b, evk, L))
    assert np.array_equal(to_host(ctx.hrotate(L, to_dev(a), to_dev(evk), 5)), o.hrotate(L, a, evk, L, 5))
    Oracle.set_threads(1)


def test_packed_keys(north_star):
    """hml_key_pack + HML_KEY_PACKED: the same results from a key whose limb slots hold packed limbs (5 of every 8 bytes read) —
    the fused inner product of one ciphertext, the stand-alone inner product of batches and of hoisted rotations, key switch."""
    ctx, o, a, b, evk = north_star
    L = 35
    K = to_dev(evk)
    P = ctx.key_pack(K)
    assert not torch.equal(P, K)
    kp = L | hml.KEY_PACKED
    assert np.array_equal(to_host(ctx.hmult(L, to_dev(a), to_dev(b), P, evk_q_limbs=kp)), o.hmult(L, a, b, evk, L))
    assert np.array_equal(to_host(ctx.hrotate(L, to_dev(a), P, 25, evk_q_limbs=kp)), o.hrotate(L, a, evk, L, 25))
    w0, w1 = o.keyswitch(L, b[1], evk, L)
    g0, g1 = ctx.keyswitch(L, to_dev(b[1]), P, kp)
    assert np.array_equal(to_host(g0), w0) and np.array_equal(to_host(g1), w1)
    A3, B3 = torch.stack([to_dev(a), to_dev(b), to_dev(a)]), torch.stack([to_dev(b), to_dev(b), to_dev(a)])
    assert torch.equal(ctx.hmult_batch(L, A3, B3, P, evk_q_limbs=kp), ctx.hmult_batch(L, A3, B3, K))
    assert torch.equal(ctx.hrotate_batch(L, A3, P, 5, evk_q_limbs=kp), ctx.hrotate_batch(L, A3, K, 5))
    gs = [5, 25, 125]
    for x, y in zip(ctx.hrotate_hoisted(L, to_dev(a), [P] * 3, gs, evk_q_limbs=kp), ctx.hrotate_hoisted(L, to_dev(a), [K] * 3, gs)):
        assert torch.equal(x, y)
    with pytest.raises(hml.HmlError):
        ctx._chk(ctx.lib.hml_key_pack(ctx.h, K.data_ptr(), K.numel() // ctx.N, K.data_ptr(), None))  # in place is refused


def test_hrotate_in_place_and_identity(north_star):
    """hml_hrotate with ct_out == ct (the epilogue must not gather sigma(c0) from rows it has already overwritten: the library
    falls back to the automorphism kernel there), several galois elements through the fused loads, and g = 1."""
    ctx, o, a, b, evk = north_star
    L = 35
    K = to_dev(evk)
    for g in (5, 25, 2 * 65536 - 1, 3 ** 7):
        want = o.hrotate(L, a, evk, L, g)
        assert np.array_equal(to_host(ctx.hrotate(L, to_dev(a), K, g)), want), g
    buf = to_dev(a).clone()
    ctx.hrotate(L, buf, K, 25, out=buf)
    assert np.array_equal(to_host(buf), o.hrotate(L, a, evk, L, 25))
    assert np.array_equal(to_host(ctx.hrotate(L, to_dev(a), K, 1)), o.hrotate(L, a, evk, L, 1))


@pytest.mark.parametrize("env", [{"HML_BCONV_UMMA": "0"}, {"HML_PDL": "0"}, {"HML_BATCH_CHUNK": "2"}],
                         ids=lambda e: ",".join("%s=%s" % kv for kv in e.items()))
def test_alternative_kernel_paths(env):
    """Every setting of a process-wide switch — the FP64 tensor-core conversion everywhere, programmatic dependent launch
    off, batches in chunks of two — is bit-exact against the oracle too (tests/sp_env_paths.py, one child process per
    setting)."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tests", "sp_env_paths.py")], env=dict(os.environ, **env), capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0 and "ENV_PATHS_OK" in r.stdout, r.stdout[-1500:] + r.stderr[-1500:]


def test_host_buffer_paths_words_and_packed(north_star):
    """hml_hmult_host / hml_hrotate_host (uint64 words, the reference's layout) and the *_packed variants (5 bytes per
    coefficient over PCIe) run chunks of 8 ciphertexts through the batched schedule: 11 ciphertexts = one full + one partial
    chunk, results equal to single calls; pack / unpack round trip on the CPU."""
    ctx, o, a, b, evk = north_star
    L, n, N = 35, 11, 65536
    A = torch.stack([to_dev(a if i % 2 == 0 else b) for i in range(n)])
    B = torch.stack([to_dev(b if i % 3 == 0 else a) for i in range(n)])
    K = to_dev(evk)
    want_m = torch.stack([ctx.hmult(L, A[i], B[i], K) for i in (0, 7, 8, 10)]).cpu()
    want_r = torch.stack([ctx.hrotate(L, A[i], K, 5) for i in (0, 7, 8, 10)]).cpu()
    ah, bh = A.cpu().pin_memory(), B.cpu().pin_memory()
    oh = torch.empty(n, 2, L - 1, N, dtype=torch.int64).pin_memory()
    ctx.hmult_host(L, ah, bh, K, oh)
    assert torch.equal(oh[[0, 7, 8, 10]], want_m)
    ap, bp = ctx.pack_host(ah), ctx.pack_host(bh)
    assert ap.numel() == n * 2 * L * 5 * N
    assert torch.equal(ctx.unpack_host(ap, ah.shape), ah)
    op = torch.empty(n * 2 * (L - 1) * 5 * N, dtype=torch.uint8).pin_memory()
    ctx.hmult_host_packed(L, n, ap, bp, K, op)
    assert torch.equal(ctx.unpack_host(op, oh.shape), oh)
    rp = torch.empty(n * 2 * L * 5 * N, dtype=torch.uint8).pin_memory()
    ctx.hrotate_host_packed(L, n, ap, K, rp, 5)
    assert torch.equal(ctx.unpack_host(rp, ah.shape)[[0, 7, 8, 10]], want_r)


@pytest.mark.parametrize("L", [45, 31, 16, 2])
def test_north_star_ring_other_levels(north_star, L):
    """config_4.cfg's ring at the maximum level (45 = three full digits), at ragged digit shapes (31 = 15 + 15 + 1,
    16 = 15 + 1) and below one digit (2): hmult (merged ModDown + Rescale, fused inner product), hrotate, and the batched
    schedule (stand-alone inner product) against the oracle."""
    ctx, o, a, b, _ = north_star
    N = 65536
    beta = -(-L // 15)
    full = [uniform_limbs(o.moduli[:L], N, 1800 + k, lead=(2,)) for k in range(2)] if L > 35 else None
    aL = full[0] if full else np.ascontiguousarray(a[:, :L])
    bL = full[1] if full else np.ascontiguousarray(b[:, :L])
    evk = uniform_limbs(o.moduli[:L] + o.moduli[45:], N, 1810 + L, lead=(beta, 2))
    K = to_dev(evk)
    want_m, want_r = o.hmult(L, aL, bL, evk, L), o.hrotate(L, aL, evk, L, 5)
    assert np.array_equal(to_host(ctx.hmult(L, to_dev(aL), to_dev(bL), K)), want_m)
    assert np.array_equal(to_host(ctx.hrotate(L, to_dev(aL), K, 5)), want_r)
    A2, B2 = torch.stack([to_dev(aL), to_dev(bL)]), torch.stack([to_dev(bL), to_dev(bL)])
    got = ctx.hmult_batch(L, A2, B2, K)
    assert np.array_equal(to_host(got[0]), want_m)
    rot = ctx.hrotate_batch(L, A2, K, 5)
    assert np.array_equal(to_host(rot[0]), want_r)


def test_empty_batches_and_zero_rotations_are_no_ops(north_star):
    ctx, o, a, b, evk = north_star
    K = to_dev(evk)
    empty = ctx.empty(0, 2, 35, 65536)
    assert ctx.hmult_batch(35, empty, empty, K).shape[0] == 0
    assert ctx.hrotate_batch(35, empty, K, 5).shape[0] == 0
    assert ctx.hrotate_hoisted(35, to_dev(a), [], []) == []
