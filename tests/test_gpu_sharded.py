"""GPU parity of the limb-sharded key switch (SURVEY.md 8e mode 2).

On one GPU the ranks are emulated one after another (a context per rank, the all-gathers done as device copies), so the
sharded arithmetic is checked bit-exactly against the oracle on every box; with >= 2 GPUs the real NCCL path
(tests/mp_sharded_keyswitch.py under torch.distributed.run) is exercised as well."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import homulator_b200 as hml  # noqa: E402
from gpu_common import to_dev, to_host  # noqa: E402
from orc import Oracle, uniform_limbs  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def sharded_keyswitch_emulated(ctxs, L, d, evk, world):
    """d [L][N], evk [beta][2][L+alpha][N] numpy; returns (out0, out1) [L][N] assembled from all ranks."""
    A, N = ctxs[0].alpha, ctxs[0].N
    lays = [hml.shard_layout(L, A, r, world) for r in range(world)]
    d_own, evk_own, g1, g2 = [], [], [], []
    for r, lay in enumerate(lays):
        own_e = lay["own_q"] + [L + j for j in lay["own_p"]]
        d_own.append(to_dev(d[lay["own_q"]] if lay["own_q"] else np.zeros((1, N), dtype=np.uint64)))
        evk_own.append(to_dev(evk[:, :, own_e]) if own_e else None)
        g1.append(torch.zeros(world, lay["gather1_slots"], N, dtype=torch.int64, device="cuda"))
        g2.append(torch.zeros(world, 2, lay["gather2_slots"], N, dtype=torch.int64, device="cuda"))
    st = torch.cuda.current_stream().cuda_stream
    for r, c in enumerate(ctxs):
        c._chk(c.lib.hml_keyswitch_shard_begin(c.h, L, r, world, d_own[r].data_ptr(), g1[r].data_ptr(), st))
    for r in range(world):  # all-gather 1
        for s in range(world):
            g1[r][s].copy_(g1[s][s])
    for r, c in enumerate(ctxs):
        if evk_own[r] is None:
            continue
        c._chk(c.lib.hml_keyswitch_shard_mid(c.h, L, r, world, d_own[r].data_ptr(), g1[r].data_ptr(), evk_own[r].data_ptr(),
                                             g2[r].data_ptr(), st))
    for r in range(world):  # all-gather 2
        for s in range(world):
            g2[r][s].copy_(g2[s][s])
    out0, out1 = np.zeros((L, N), dtype=np.uint64), np.zeros((L, N), dtype=np.uint64)
    for r, c in enumerate(ctxs):
        nq = len(lays[r]["own_q"])
        o0 = torch.zeros(max(nq, 1), N, dtype=torch.int64, device="cuda")
        o1 = torch.zeros_like(o0)
        c._chk(c.lib.hml_keyswitch_shard_end(c.h, L, r, world, g2[r].data_ptr(), o0.data_ptr(), o1.data_ptr(), st))
        if nq:
            out0[lays[r]["own_q"]] = to_host(o0)[:nq]
            out1[lays[r]["own_q"]] = to_host(o1)[:nq]
    return out0, out1


@pytest.mark.parametrize("N,ML,L,A,world", [(256, 7, 7, 3, 2), (256, 7, 7, 3, 3), (1024, 6, 5, 2, 4), (64, 5, 2, 3, 2),
                                             (4096, 4, 4, 4, 8), (8192, 9, 8, 3, 2), (65536, 45, 35, 15, 4)])
def test_sharded_keyswitch_emulated_ranks(N, ML, L, A, world):
    o = Oracle(N, 36, ML, A)
    Oracle.set_threads(0)
    beta = -(-L // A)
    d = uniform_limbs(o.moduli[:L], N, 2000 + L)
    evk = uniform_limbs(o.moduli[:L] + o.moduli[ML:], N, 2001, lead=(beta, 2))
    want0, want1 = o.keyswitch(L, d, evk, L)
    Oracle.set_threads(1)
    ctxs = [hml.Context(N=N, max_level=ML, alpha=A) for _ in range(world)]
    got0, got1 = sharded_keyswitch_emulated(ctxs, L, d, evk, world)
    assert np.array_equal(got0, want0) and np.array_equal(got1, want1)
    # world = 1 degenerates to the unsharded schedule
    one0, one1 = sharded_keyswitch_emulated(ctxs[:1], L, d, evk, 1)
    assert np.array_equal(one0, want0) and np.array_equal(one1, want1)


def _split(o, L, world, a, evk):
    """owned-limb slices of a ciphertext-like array [.., L, N] and of a key [beta][2][E][N] for every rank"""
    A = o.alpha
    own = [list(range(r, L, world)) for r in range(world)]
    own_e = [[e for e in range(L + A) if e % world == r] for r in range(world)]
    a_own = [to_dev(a[..., own[r], :]) if own[r] else None for r in range(world)]
    evk_own = [to_dev(evk[:, :, own_e[r]]) if own_e[r] else None for r in range(world)]
    return own, a_own, evk_own


@pytest.mark.parametrize("N,ML,L,A,world", [(256, 7, 7, 3, 2), (256, 7, 7, 3, 3), (1024, 6, 5, 2, 4), (8192, 9, 8, 3, 2), (8192, 9, 9, 3, 8),
                                             (65536, 45, 35, 15, 4)])
def test_sharded_ops_through_the_c_abi_emulated_ranks(N, ML, L, A, world):
    """hml_group_op: keyswitch, hrotate, hmult and rescale on limb-sharded operands, every op ONE C-ABI call that composes the
    limb-local phases and the exchanges inside the library (homulator_b200/csrc/shard.cu).  The ranks share this GPU and one
    stream (signals are enqueued before the waits that need them, so nothing ever spins); the base conversions read the other
    ranks' gather buffers through per-source offsets exactly as they do over NVLink.  Against the oracle's unsharded ops;
    every op runs twice (buffer reuse across epochs)."""
    o = Oracle(N, 36, ML, A)
    Oracle.set_threads(0)
    beta = -(-L // A)
    a = uniform_limbs(o.moduli[:L], N, 2200 + L, lead=(2,))
    b = uniform_limbs(o.moduli[:L], N, 2201 + L, lead=(2,))
    evk = uniform_limbs(o.moduli[:L] + o.moduli[ML:], N, 2202, lead=(beta, 2))
    g = 25
    want_ks = o.keyswitch(L, a[1], evk, L)
    want_rot = o.hrotate(L, a, evk, L, g)
    want_mul = o.hmult(L, a, b, evk, L)
    want_rs = np.stack([o.rescale(L, b[0]), o.rescale(L, b[1])])
    Oracle.set_threads(1)
    ctxs = [hml.Context(N=N, max_level=ML, alpha=A) for _ in range(world)]
    group = hml.Shard.local_group(ctxs, L)
    for sh in group:
        sh.prepare(L)
    R = range(world)
    own, a_own, evk_own = _split(o, L, world, a, evk)
    _, b_own, _ = _split(o, L, world, b, evk)
    nq = [len(own[r]) for r in R]
    keep = [[i for i in own[r] if i < L - 1] for r in R]

    def empty(r, *shape):
        return ctxs[r].empty(*shape)

    def assemble(outs, idx, shape):
        got = np.zeros(shape, dtype=np.uint64)
        for r in R:
            if idx[r]:
                got[..., idx[r], :] = to_host(outs[r])[..., :len(idx[r]), :]
        return got

    for _ in range(2):
        o0 = [empty(r, max(nq[r], 1), N) for r in R]
        o1 = [empty(r, max(nq[r], 1), N) for r in R]
        d_own = [x[1].contiguous() if x is not None else None for x in a_own]
        hml.group_op(group, "keyswitch", L, d_own, key=evk_own, out0=o0, out1=o1)
        assert np.array_equal(assemble(o0, own, (L, N)), want_ks[0]) and np.array_equal(assemble(o1, own, (L, N)), want_ks[1])
        rot = [empty(r, 2, max(nq[r], 1), N) for r in R]
        hml.group_op(group, "hrotate", L, a_own, key=evk_own, out0=rot, galois_elt=g)
        assert np.array_equal(assemble(rot, own, (2, L, N)), want_rot)
        mul = [empty(r, 2, max(len(keep[r]), 1), N) for r in R]
        hml.group_op(group, "hmult", L, a_own, b=b_own, key=evk_own, out0=mul)
        assert np.array_equal(assemble(mul, keep, (2, L - 1, N)), want_mul)
        for _ in range(2):  # rescale straight after a rescale: the rescale buffer is reused (write-after-read ordering)
            rs = [empty(r, 2, max(len(keep[r]), 1), N) for r in R]
            hml.group_op(group, "rescale", L, b_own, out0=rs)
            assert np.array_equal(assemble(rs, keep, (2, L - 1, N)), want_rs)
    for sh in group:
        sh.check()
        sh.close()


def test_peer_direct_needs_the_tcgen05_conversion():
    ctxs = [hml.Context(N=64, max_level=5, alpha=3) for _ in range(2)]  # N < 128: the FP64 tensor-core kernel has no per-source offsets
    group = hml.Shard.local_group(ctxs, 2)
    with pytest.raises(hml.HmlError):
        group[0].prepare(2)
    for sh in group:
        sh.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_local_group_across_devices():
    """one process driving one rank per DEVICE (hml_shard_connect_local: peer access, fused one-launch exchanges) — the mode the
    CLI's [cluster] argument uses"""
    n = min(torch.cuda.device_count(), 4)
    r = subprocess.run([os.path.join(ROOT, "homulator_b200", "Homulator.run"), os.path.join(ROOT, "config", "config_4.cfg"), "hmult", "45", "35", "15",
                        str(n), "--iters", "3", "--warmup", "1", "--verify"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    import json
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["cluster"] == n and line["gpus_used"] == n and line["sharded_matches_one_gpu"] is True


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_sharded_keyswitch_nccl():
    n = min(torch.cuda.device_count(), 4)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
           "--master-port", "29531", os.path.join(ROOT, "tests", "mp_sharded_keyswitch.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "SHARDED_KS_OK" in r.stdout


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_sharded_keyswitch_peer_direct_over_nvlink():
    n = min(torch.cuda.device_count(), 4)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(ROOT, "tests", "mp_sharded_keyswitch_p2p.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "SHARDED_P2P_OK" in r.stdout


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_sharded_op_sequence_over_nvlink():
    n = min(torch.cuda.device_count(), 4)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
           "--master-port", "29539", os.path.join(ROOT, "tests", "mp_sharded_replay.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "SHARDED_REPLAY_OK" in r.stdout
