#!/usr/bin/env python3
"""bench.py — hmult latency/throughput at N=2^16, l=35, alpha=15 (BASELINE.json north-star config) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B]           # this repo's CUDA path
    python bench.py --impl reference [--steps K] [--warmup W]                  # CPU reference arm
    python bench.py ... --dump-outputs DIR     # also write a seeded sample of the last timed step's result to DIR/*.npy

A "step" is one pass of the hot path over one batch of synthetic input: B independent hmult
(config_4.cfg, maxLevel 45, currentLevel 35, alpha 15) per GPU, all B ciphertext pairs distinct and resident
in HBM (2*B*36.7 MB of input per GPU, far larger than L2, so no L2 flush is needed between steps).
`value` = microseconds per hmult over the whole job (all ranks), lower is better.  One process per GPU,
independent ciphertexts sharded across ranks, no data-path collective ("scaling": "weak").

The JSON line also carries: `e2e` (same metric through the host-buffer C-ABI call, H2D/D2H inside the timed
region), `roofline` (the forward-NTT kernel pair timed alone with CUDA events on the batched ModUp launch shape), `cpu_baseline` (the scalar
oracle port timed on one host core on a bounded sample), `extra` (single-op latencies with L2 flushed,
hrotate, NTT limbs/s, the reference's published-by-survey simulator figures).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

CFG = os.path.join(ROOT, "config", "config_4.cfg")
N_RING, MAX_LEVEL, LEVEL, ALPHA = 65536, 45, 35, 15
METRIC = "hmult_us_N65536_l35_alpha15"
HMULT_SIM_CYCLES = 221716  # the reference's own `Homulator.run config_4.cfg hmult 45 35 15` (353 host minutes on one core, BASELINE.md)
WORKLOAD = "hmult config_4.cfg maxLevel=45 currentLevel=35 alpha=15 (BASELINE.json configs[0]/[3])"


def bench_config(world):
    """The workload both arms name: BASELINE.json configs[3], 256 ciphertexts per step over the job."""
    return {"workload": WORKLOAD, "batch_per_gpu_per_step": max(1, 256 // world), "ciphertexts_per_step": max(1, 256 // world) * world,
            "l2": "inputs larger than L2 (no flush)"}


def measured_peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons through NVML every few ms while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.sm, self.max_mhz, self.reasons, self.stop_flag = index, [], None, set(), False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.003)

    def summary(self):
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(sm)}


DUMP_BYTES = 32 << 20  # one step's result is 9.1 GB (256 x 2 x 34 x 65536 words); --dump-outputs writes a sample of this size
DUMP_SEED = 0x64756D70


def dump_outputs(dirname, name, out, budget, torch):
    """Write a seeded sample of `out` (int64 [..., N] residues below 2^36, exact in float64) as dirname/name.npy: per row
    (every ciphertext, component and limb) the same pseudo-random coefficient positions on every run, so that two builds of
    the project can be compared output for output.  Shape [..., k] with k = budget / (8 bytes x rows)."""
    import numpy as np
    rows, n = out.numel() // out.shape[-1], out.shape[-1]
    k = max(1, min(n, budget // (8 * rows)))
    g = torch.Generator().manual_seed(DUMP_SEED)
    idx = torch.randint(0, n, (*out.shape[:-1], k), generator=g).to(out.device)
    sample = torch.gather(out, -1, idx).cpu().numpy().astype(np.float64)
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, name + ".npy"), sample)


def cpu_port_sample(n_ops, threads):
    """Time the scalar oracle port (oracle/oracle.c) on the same workload: n_ops hmult, `threads` host threads."""
    from orc import Oracle, uniform_limbs
    o = Oracle(N_RING, 36, MAX_LEVEL, ALPHA)
    L = LEVEL
    a = uniform_limbs(o.moduli[:L], N_RING, 1, lead=(2,))
    b = uniform_limbs(o.moduli[:L], N_RING, 2, lead=(2,))
    evk = uniform_limbs(o.moduli[:L] + o.moduli[MAX_LEVEL:], N_RING, 3, lead=(3, 2))
    used = Oracle.set_threads(threads)
    t0 = time.perf_counter()
    for _ in range(n_ops):
        o.hmult(L, a, b, evk, L)
    dt = time.perf_counter() - t0
    Oracle.set_threads(1)
    return dt / n_ops * 1e6, used


def run_reference(args, real_stdout):
    """Reference arm.  The reference itself (a cycle simulator) computes no ciphertext values and its own run of this
    config takes hours (BASELINE.md section 2), so the CPU implementation of the path timed here is the scalar oracle
    port with all host threads; each step is ONE hmult (bounded sample of the workload)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    for _ in range(max(0, min(args.warmup, 1))):
        cpu_port_sample(1, threads)
    steps = args.steps
    us, used = cpu_port_sample(steps, threads)
    sim = {}
    run = os.path.join(ROOT, "oracle", "_ref", "count.run")
    if os.path.exists(run) and not args.no_extra:  # the reference's own instruction generation for this op (the part our planner replaces)
        try:
            line = subprocess.run([run, CFG, "hmult", str(MAX_LEVEL), str(LEVEL), str(ALPHA)], capture_output=True, text=True,
                                  timeout=120).stdout.strip().splitlines()[-1]
            sim["homulator_insgen_seconds"] = json.loads(line)["insgen_seconds"]
        except Exception:
            pass
    # Homulator's own host wall-clock: the unmodified reference CLI (oracle/_ref/Homulator.run) simulating THIS op and config
    # on one host core for a bounded time; the full run takes hours (BASELINE.md section 2), so the sample reports how far
    # the cycle simulator got and the cycles it simulates per second of host time.
    cli = os.path.join(ROOT, "oracle", "_ref", "Homulator.run")
    if os.path.exists(cli) and not args.no_extra:
        try:
            budget = 20
            t0 = time.perf_counter()
            r = subprocess.run(["timeout", str(budget), "stdbuf", "-oL", cli, CFG, "hmult", str(MAX_LEVEL), str(LEVEL), str(ALPHA)],
                               capture_output=True, text=True, timeout=budget + 30)
            dt = time.perf_counter() - t0
            cyc = [int(l.split()[2]) for l in r.stdout.splitlines() if l.startswith("FHE-Sim running")]
            done = [int(l.split()[3]) for l in r.stdout.splitlines() if l.startswith("We have executed") and "instructions!" in l]
            sim["homulator_cli_sample"] = {
                "command": "Homulator.run config_4.cfg hmult 45 35 15", "host_seconds": dt, "cores": 1,
                "simulated_cycles_reached": cyc[-1] if cyc else 0, "instructions_completed": done[-1] if done else 0,
                "instructions_total": 7381760, "status": "DNF(budget)" if r.returncode == 124 else "exit %d" % r.returncode}
        except Exception as e:  # reported baseline only
            sim["homulator_cli_sample"] = {"error": str(e)[:120]}
    line = {
        "impl": "reference", "metric": METRIC, "value": us, "unit": "us", "n_gpus": args.gpus, "steps": steps,
        "warmup": args.warmup, "ms_per_step": us / 1e3, "higher_is_better": False, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64 residues (36-bit), arithmetic on the FP64 pipe", "data": "synthetic",
        # the same `config` as the GPU arm; each step here is a bounded SAMPLE of that step (one hmult), see cpu_baseline.sample
        "config": bench_config(max(1, args.gpus)),
        "cpu_baseline": {"value": us, "unit": "us", "cores": used, "kind": "port",
                         "sample": "%d hmult at the full config, oracle/oracle.c with OpenMP over limbs" % steps},
        "e2e": {"value": us, "unit": "us", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "extra": sim,
    }
    _emit(real_stdout, line)
    return 0


def _claim_stdout():
    """Everything libraries print to stdout while the bench runs (e.g. NCCL's version banner) goes to stderr; the JSON line is
    written to the real stdout, which therefore holds exactly one line."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return real


def _emit(real_stdout, line):
    sys.stdout.flush()
    os.write(real_stdout, (json.dumps(line) + "\n").encode())


def limb_sharded(ctx, rank, world, L, evk, dist, torch):
    """SURVEY.md 8e mode 2 / BASELINE.json configs[4] on all ranks: one ciphertext's key switch and the rotation-heavy op
    sequence with the limbs sharded over the GPUs (limb i on rank i % world), every sharded op ONE C-ABI call
    (hml_keyswitch_sharded, hml_replay_* over an hml_shard).  Device events, max over ranks."""
    import homulator_b200 as hml
    from homulator_b200.replay import bsgs_trace, shard_operands, trace_counts
    q = list(range(L))
    d = ctx.uniform(q, 900)
    x = ctx.uniform(q, 901, lead=(2,))

    def exchange(obj):
        out = [None] * world
        dist.all_gather_object(out, obj)
        return out

    def timeit(fn, reps):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) * 1e3 / reps], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    sh = hml.Shard.ipc(ctx, L, rank, world, exchange)
    sh.prepare(L)
    oi = torch.tensor(sh.own_q(L), device="cuda", dtype=torch.long)
    oe = torch.tensor(sh.own_ext(L), device="cuda", dtype=torch.long)
    d_own, evk_own = d[oi].contiguous(), evk[:, :, oe].contiguous()
    dist.barrier()
    ref0, ref1 = ctx.keyswitch(L, d, evk)
    o0, o1 = ctx.empty(max(len(oi), 1), N_RING), ctx.empty(max(len(oi), 1), N_RING)
    sh.keyswitch(L, d_own, evk_own, o0, o1)
    ok = bool(torch.equal(o0[:len(oi)], ref0[oi]) and torch.equal(o1[:len(oi)], ref1[oi]))
    t0 = time.perf_counter()
    for _ in range(20):
        sh.keyswitch(L, d_own, evk_own, o0, o1)
    host_us = (time.perf_counter() - t0) / 20 * 1e6
    torch.cuda.synchronize()
    res = {"keyswitch_peer_direct_us": timeit(lambda: sh.keyswitch(L, d_own, evk_own, o0, o1), 20),
           "keyswitch_host_enqueue_us": host_us,
           "keyswitch_nccl_allgather_us": timeit(lambda: ctx.keyswitch_sharded(
               L, d_own, evk_own, rank, world, lambda buf: dist.all_gather_into_tensor(buf, buf[rank].clone())), 20),
           "keyswitch_one_gpu_us": timeit(lambda: ctx.keyswitch(L, d, evk), 20)}
    tr = bsgs_trace(4, 4)
    pts = {i: ctx.uniform(q, 920 + i) for i in range(16)}
    keys = {r: evk for r in sorted({op[3] for op in tr if op[0] == "hrotate"})}
    x_own, pts_own, keys_own, _ = shard_operands(sh, L, x, pts, keys, evk)
    one = hml.Replay(ctx, L, tr).bind(x, pts, keys, evk)
    ref = one.run().result("z").clone()
    keep = torch.tensor([i for i in sh.own_q(L) if i < L - 1], device="cuda", dtype=torch.long)
    res["sequence_ops"] = trace_counts(tr)
    for name, graph in (("sequence_peer_direct_us", False), ("sequence_peer_direct_graph_us", True)):
        rp = hml.Replay(ctx, L, tr, shard=sh, graph=graph).bind(x_own, pts_own, keys_own, evk_own)
        got = rp.run().result("z")
        torch.cuda.synchronize()
        ok = ok and bool(torch.equal(got.contiguous(), ref[:, keep]))
        res[name] = timeit(rp.run, 5)
        dist.barrier()
        rp.close()
    res["sequence_one_gpu_us"] = timeit(one.run, 5)
    try:
        sh.check()
    except hml.HmlError:
        ok = False
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    res["bit_identical_to_one_gpu"] = bool(int(flag) == 1)
    dist.barrier()
    torch.cuda.synchronize()
    one.close()
    sh.close()
    dist.barrier()
    return res


def main():
    real_stdout = _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=0,
                    help="hmult per GPU per step; default 256 / n_gpus (BASELINE.json configs[3]: 256 ciphertexts per step over the job)")
    ap.add_argument("--e2e-batch", type=int, default=32, help="hmult per GPU per step on the host-buffer path")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-sharded", action="store_true",
                    help="with --gpus N > 1 the bench also times ONE ciphertext's key switch and the op sequence limb-sharded over the "
                         "N GPUs (peer-direct NVLink exchanges vs NCCL all-gathers vs one GPU) -> extra.limb_sharded; this skips it")
    ap.add_argument("--sharded", action="store_true", help="(default for N > 1; kept for compatibility)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a seeded %d MB sample of the last step's hmult results (float64) to "
                         "DIR/hmult_out.npy (DIR/hmult_out_rank<r>.npy per rank with several GPUs)" % (DUMP_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args, real_stdout)

    import torch
    import torch.distributed as dist
    import homulator_b200 as hml

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; homulator_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    # run this rank's host threads on the CPUs next to its GPU before any pinned buffer is allocated (first touch): with several
    # ranks per box the host-buffer path is bound by the host's memory and PCIe paths, and remote-socket staging halves it
    numa = "unset"
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
        numa = "nvml ideal cpus (%d)" % len(os.sched_getaffinity(0))
    except Exception as e:  # not fatal: the run proceeds with the inherited affinity
        numa = "unchanged (%s)" % type(e).__name__
    W = max(3, args.warmup)
    K, L = args.steps, LEVEL
    B = args.batch if args.batch > 0 else max(1, 256 // world)

    ctx = hml.Context(CFG, MAX_LEVEL, ALPHA, device=local)
    q = list(range(L))
    evk = ctx.uniform(ctx.ext_mod_idx(L), 3, lead=(ctx.beta(L), 2))
    ct_a = ctx.uniform(q, 10 + rank, lead=(B, 2))
    ct_b = ctx.uniform(q, 1000 + rank, lead=(B, 2))
    out = ctx.empty(B, 2, L - 1, N_RING)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- roofline of the dominant kernel pair: forward NTT (column pass + row pass), timed ALONE on the launch
    # shape the batched step uses — the ModUp NTT of one chunk: 32 ciphertexts x 115 limbs in ONE launch pair — and BEFORE the
    # sustained region: MEASURED_PEAKS.json's HBM figure is a burst measurement (best of 10 copies), and so is this; the boxes
    # of this pool drop to 1700-1900 MHz under their 1000 W cap once the step loop has run for a second.  The same pair under
    # sustained load is reported as extra.ntt_us_per_limb_sustained (re-timed at the end of the run).
    peak, peak_src = measured_peaks()
    W_bytes = 8 * N_RING
    n_limbs, n_b = 115, 32
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def ntt_pair_ms(reps=10, settle=False):
        idx = [ctx.ext_mod_idx(L)[i % (L + ALPHA)] for i in range(n_limbs)]
        bufs = [ctx.uniform(idx, 50 + i, lead=(n_b,)) for i in range(2)]  # 2 x 1.9 GB >> L2: every launch reads from HBM
        dst = ctx.empty(n_b, n_limbs, N_RING)
        if settle:  # generating the inputs is a burst of its own
            torch.cuda.synchronize()
            time.sleep(1.0)
        for i in range(3):
            ctx.ntt_batch(bufs[i % 2], idx, out=dst)
        torch.cuda.synchronize()
        e0.record()
        for i in range(reps):
            ctx.ntt_batch(bufs[i % 2], idx, out=dst)
        e1.record()
        torch.cuda.synchronize()
        pair = e0.elapsed_time(e1) / reps
        # single-ciphertext launch (115 limbs), for the latency-mode figure
        for i in range(3):
            ctx.ntt(bufs[i % 2][0], idx, out=dst[0])
        torch.cuda.synchronize()
        e0.record()
        for i in range(20):
            ctx.ntt(bufs[i % 2][i % n_b], idx, out=dst[0])
        e1.record()
        torch.cuda.synchronize()
        return pair, e0.elapsed_time(e1) / 20 * 1e3 / n_limbs

    flush = torch.empty(64 << 20, dtype=torch.int64, device="cuda") if rank == 0 and not args.no_extra else None  # 512 MiB

    def lat(fn, iters=10):
        ts = []
        for _ in range(iters):
            flush.fill_(1)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            fn()
            a1.record()
            a1.synchronize()
            ts.append(a0.elapsed_time(a1) * 1e3)
        ts.sort()
        return ts[len(ts) // 2]

    ntt_ms = ntt1_us_per_limb = ntt_clock = hm = hr = hm_pk = hr_pk = None
    burst = {}

    def cool():
        """The board's power controller averages over about a second: the burst measurements below are separated by short idle
        gaps so that none of them starts inside the previous one's power-cap tail."""
        torch.cuda.synchronize()
        time.sleep(1.0)

    if rank == 0:
        ntt_ms, ntt1_us_per_limb = ntt_pair_ms(settle=True)
        try:
            import pynvml
            ntt_clock = pynvml.nvmlDeviceGetClockInfo(pynvml.nvmlDeviceGetHandleByIndex(local), pynvml.NVML_CLOCK_SM)
        except Exception:
            pass
        cool()
        if flush is not None:  # one-ciphertext latencies (L2 flushed), also before the sustained region: a latency figure
            o1, o2 = ctx.empty(2, L - 1, N_RING), ctx.empty(2, L, N_RING)
            for _ in range(3):
                ctx.hmult(L, ct_a[0], ct_b[0], evk, out=o1)
                ctx.hrotate(L, ct_a[0], evk, 5, out=o2)
            hm = lat(lambda: ctx.hmult(L, ct_a[0], ct_b[0], evk, out=o1), 20)
            hr = lat(lambda: ctx.hrotate(L, ct_a[0], evk, 5, out=o2), 20)
            # the same with the key handed over packed (hml_key_pack + HML_KEY_PACKED: 94 instead of 150 MB read per key switch)
            evk_p = ctx.key_pack(evk)
            kp = L | hml.KEY_PACKED
            for _ in range(3):
                ctx.hmult(L, ct_a[0], ct_b[0], evk_p, evk_q_limbs=kp, out=o1)
                ctx.hrotate(L, ct_a[0], evk_p, 5, evk_q_limbs=kp, out=o2)
            hm_pk = lat(lambda: ctx.hmult(L, ct_a[0], ct_b[0], evk_p, evk_q_limbs=kp, out=o1), 20)
            hr_pk = lat(lambda: ctx.hrotate(L, ct_a[0], evk_p, 5, evk_q_limbs=kp, out=o2), 20)
            del o1, o2, evk_p
        cool()
        # one 32-ciphertext chunk of the batched ops timed alone (a 25 ms burst at full clocks): what the kernels do before the
        # board reaches its power cap; `value` below is the sustained figure of the 256-ciphertext steps
        nb32 = min(32, B)
        ob = ctx.empty(nb32, 2, L, N_RING)
        for name, fn in (("hmult", lambda: ctx.hmult_batch(L, ct_a[:nb32], ct_b[:nb32], evk, out=out[:nb32])),
                         ("hrotate", lambda: ctx.hrotate_batch(L, ct_a[:nb32], evk, 5, out=ob))):
            for _ in range(2):
                fn()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(3):
                fn()
            e1.record()
            torch.cuda.synchronize()
            burst[name] = e0.elapsed_time(e1) * 1e3 / (3 * nb32)
        del ob
        cool()

    # the process group is created only now: while rank 0 timed its kernels alone, the other ranks waited in the rendezvous on
    # the host (in an NCCL barrier their kernels would spin on peer memory next to the measurement: 0.35 -> 0.40 us per limb)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    # ---------------- device-resident throughput (value)
    for _ in range(W):
        ctx.hmult_batch(L, ct_a, ct_b, evk, out=out)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    ctx.exec_counts(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(K):
        ctx.hmult_batch(L, ct_a, ct_b, evk, out=out)
    e1.record()
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    sampler.stop_flag = True
    launches = ctx.exec_counts()["kernel_launches"]
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    n_ops = K * B * world
    us_per_op = ms_total * 1e3 / n_ops
    sampler.join(timeout=2)
    if args.dump_outputs:  # `out` holds the last timed step's results until the profile below rewrites its first chunk
        dump_outputs(args.dump_outputs, "hmult_out" if world == 1 else "hmult_out_rank%d" % rank, out, DUMP_BYTES // world, torch)

    # ---------------- end to end through the host-buffer C-ABI call (pinned host memory, H2D + D2H inside)
    Be = args.e2e_batch
    ah = ct_a[:Be].cpu().pin_memory()
    bh = ct_b[:Be].cpu().pin_memory()
    oh = torch.empty(Be, 2, L - 1, N_RING, dtype=torch.int64).pin_memory()
    for _ in range(2):
        ctx.hmult_host(L, ah, bh, evk, oh)
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        ctx.hmult_host(L, ah, bh, evk, oh)
    barrier()
    e2e_ms = torch.tensor([(time.perf_counter() - t0) * 1e3], device="cuda")
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_us = float(e2e_ms.item()) * 1e3 / (K * Be * world)
    e2e_ok = bool(torch.equal(oh.cuda(), out[:Be]))
    # the same call with the ciphertexts packed in host memory (5 bytes per coefficient over PCIe instead of the reference's
    # 8-byte words): reported next to `e2e`, which stays the drop-in uint64 layout
    ap, bp = ctx.pack_host(ah), ctx.pack_host(bh)
    op = torch.empty(Be * 2 * (L - 1) * 5 * N_RING, dtype=torch.uint8).pin_memory()
    for _ in range(2):
        ctx.hmult_host_packed(L, Be, ap, bp, evk, op)
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        ctx.hmult_host_packed(L, Be, ap, bp, evk, op)
    barrier()
    e2ep_ms = torch.tensor([(time.perf_counter() - t0) * 1e3], device="cuda")
    if world > 1:
        dist.all_reduce(e2ep_ms, op=dist.ReduceOp.MAX)
    e2e_packed_us = float(e2ep_ms.item()) * 1e3 / (K * Be * world)
    e2e_packed_ok = bool(torch.equal(ctx.unpack_host(op, oh.shape), oh))
    del ap, bp, op

    # ---------------- hrotate, batched (same step shape), all ranks
    out_r = ctx.empty(B, 2, L, N_RING)
    for _ in range(2):
        ctx.hrotate_batch(L, ct_a, evk, 5, out=out_r)
    barrier()
    e0.record()
    for _ in range(max(2, K // 2)):
        ctx.hrotate_batch(L, ct_a, evk, 5, out=out_r)
    e1.record()
    barrier()
    hr_ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(hr_ms, op=dist.ReduceOp.MAX)
    hrot_batched_us = float(hr_ms.item()) * 1e3 / (max(2, K // 2) * B * world)
    del out_r

    sharded = limb_sharded(ctx, rank, world, L, evk, dist, torch) if (world > 1 and not args.no_sharded) else None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    ntt_bytes = 2.0 * W_bytes * n_limbs * n_b
    ntt_ms_early = ntt_ms
    ntt_ms_sustained, _ = ntt_pair_ms(5)  # the same pair after the step loop: power-capped clocks at one GPU; with several ranks
    # the steps are short (no cap) and this placement is the undisturbed one (the other ranks start up beside the first one)
    ntt_ms = min(ntt_ms_early, ntt_ms_sustained)
    ntt_gbs = ntt_bytes / (ntt_ms * 1e-3) / 1e9
    ntt_limbs_per_s = n_limbs * n_b / (ntt_ms * 1e-3)
    reps = 10
    # base conversion on the tensor cores (tcgen05 kind::i8), batched ModDown shape: 64 polynomials x (15 P-limbs -> 35 Q-limbs)
    # in one launch through hml_bconv_batch (that entry point also applies step 1 and stores canonical words)
    src_p, dst_q, n_bc = list(range(MAX_LEVEL, MAX_LEVEL + ALPHA)), list(range(L)), 64
    xb = [ctx.uniform(src_p, 70 + i, lead=(n_bc,)) for i in range(2)]
    ob = ctx.empty(n_bc, L, N_RING)
    for i in range(3):
        ctx.bconv_batch(xb[i % 2], src_p, dst_q, out=ob)
    torch.cuda.synchronize()
    e0.record()
    for i in range(reps):
        ctx.bconv_batch(xb[i % 2], src_p, dst_q, out=ob)
    e1.record()
    torch.cuda.synchronize()
    bconv_ms = e0.elapsed_time(e1) / reps
    bconv_bytes = float(ALPHA + L) * W_bytes * n_bc
    del xb, ob
    # the same kernel as it runs INSIDE the op (hml_profile_*: an event after every launch group of one 32-ciphertext chunk):
    # no step-1 multiply in the packer (the INTT folds it), doubles out (the forward transform's input format).  Bytes per
    # ciphertext: ModUp L -> beta (L + alpha) - L limbs, ModDown 2 x (alpha (+ the folded source row) -> L - 1)
    nbp = min(32, B)
    prof = ctx.profile(lambda: ctx.hmult_batch(L, ct_a[:nbp], ct_b[:nbp], evk, out=out[:nbp]))
    beta = ctx.beta(L)
    conv_limbs = (L + (beta * (L + ALPHA) - L)) + 2 * ((ALPHA + 1) + (L - 1))
    inop_bytes = float(conv_limbs) * W_bytes * nbp
    inop_us = prof["us"]["BCONV"]
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "ntt_traffic.json")))["dram_bytes_per_launch"]
    except Exception:
        pass

    # the FP64 butterfly's issue floor (8 DP instructions per butterfly, each holding the issue port for two cycles, DESIGN.md 3.0):
    # 524288 butterflies x 16 cycles / (592 sub-partitions x 32 lanes) per limb at the clock sampled during the run
    clk = ntt_clock or sampler.summary().get("sm_mhz") or 1965
    fp64_floor_us = 524288 * 16 / (4 * 148 * 32) / clk
    extra = {"hrotate_batched_us": hrot_batched_us, "hmult_batched_us": us_per_op, "throughput_hmult_per_s": n_ops / (ms_total * 1e-3),
             "ntt_fp64_issue_floor_us_per_limb": fp64_floor_us, "ntt_frac_of_fp64_issue_floor": fp64_floor_us / (ntt_ms * 1e3 / (n_limbs * n_b)), "ntt_limbs_per_s": ntt_limbs_per_s, "ntt_us_per_limb": ntt_ms * 1e3 / (n_limbs * n_b),
             "ntt_us_per_limb_before_step_loop": ntt_ms_early * 1e3 / (n_limbs * n_b),
             "ntt_us_per_limb_sustained": ntt_ms_sustained * 1e3 / (n_limbs * n_b), "ntt_sm_mhz_when_timed_alone": ntt_clock,
             "hmult_batched_us_one_chunk_burst": burst["hmult"], "hrotate_batched_us_one_chunk_burst": burst["hrotate"],
             "ntt_us_per_limb_single_ciphertext_launch": ntt1_us_per_limb, "e2e_matches_device_path": e2e_ok,
             "e2e_packed_host_format": {"value": e2e_packed_us, "unit": "us", "h2d_bytes_per_step": 2 * 2 * L * 5 * N_RING * Be,
                                        "d2h_bytes_per_step": 2 * (L - 1) * 5 * N_RING * Be, "matches_u64_path": e2e_packed_ok,
                                        "call": "hml_hmult_host_packed (5 bytes per coefficient in pinned host memory)"},
             "bconv_tcgen05": {"kernel": "k_bconv_umma (tcgen05.mma kind::i8, 64 polynomials x 15 -> 35 limbs per launch)",
                               "us_per_launch": bconv_ms * 1e3, "algorithmic_bytes_per_launch": bconv_bytes,
                               "achieved_gbs": bconv_bytes / (bconv_ms * 1e-3) / 1e9, "hbm_frac": bconv_bytes / (bconv_ms * 1e-3) / 1e9 / peak,
                               "limb_macs_per_s": ALPHA * L * n_bc / (bconv_ms * 1e-3),
                               "in_op": {"what": "the two conversion launches of one %d-ciphertext hmult chunk (ModUp 35 -> 115 limbs, "
                                                 "ModDown 2 x (15 + folded row -> 34)), doubles out, event-timed inside the op" % nbp,
                                         "us_per_chunk": inop_us, "algorithmic_bytes_per_chunk": inop_bytes,
                                         "achieved_gbs": inop_bytes / (inop_us * 1e-6) / 1e9,
                                         "hbm_frac": inop_bytes / (inop_us * 1e-6) / 1e9 / peak}},
             "hmult_chunk_class_us": dict(prof["us"], total=prof["total_us"], ciphertexts=nbp)}
    if not args.no_extra:
        o_late = ctx.empty(2, L - 1, N_RING)
        hm_late = lat(lambda: ctx.hmult(L, ct_a[0], ct_b[0], evk, out=o_late))  # the same after the sustained region
        aw_m, aw_r = hml.algorithmic_words("hmult", L, ALPHA), hml.algorithmic_words("hrotate", L, ALPHA)
        extra.update({
            "hmult_single_us_l2_flushed": hm, "hrotate_single_us_l2_flushed": hr, "hmult_single_us_l2_flushed_after_sustained_load": hm_late,
            "hmult_single_us_l2_flushed_packed_key": hm_pk, "hrotate_single_us_l2_flushed_packed_key": hr_pk,
            "hmult_single_unfused_bytes_equivalent_over_hbm_peak": aw_m * W_bytes / (hm * 1e-6) / 1e9 / peak,
            "hrotate_single_unfused_bytes_equivalent_over_hbm_peak": aw_r * W_bytes / (hr * 1e-6) / 1e9 / peak,
            # NOT a roofline fraction: SURVEY 8d's UNFUSED byte count divided by the time of the fused / merged schedule (which
            # moves ~0.9 GB per hmult, not 1.32 GB) — can exceed 1; quoted because 8d asks for it
            "hmult_batched_unfused_bytes_equivalent_over_hbm_peak": aw_m * W_bytes / (us_per_op * 1e-6) / 1e9 / (peak * world),
            "hrotate_batched_unfused_bytes_equivalent_over_hbm_peak": aw_r * W_bytes / (hrot_batched_us * 1e-6) / 1e9 / (peak * world),
            "homulator_simulated_cycles": {"hrotate_45_35_15": 203651, "hrotate_host_minutes_1core": 235.9, "hmult_host_minutes_1core": 353.4,
                                           "hmult_45_35_15": HMULT_SIM_CYCLES, "note": "unmodified reference CLI, g++ -O2, build container; "
                                           "cycles are machine-independent (BASELINE.md section 2); 1 cycle = 1 ns at an assumed 1 GHz"},
        })
        # BASELINE.json configs[4]: synthetic rotation-heavy op sequences through hml_replay_*: the baby-step/giant-step trace
        # (6 rotations) and the 16-rotation sum SURVEY.md 8d suggests; plain launches, one CUDA graph, hoisted rotations
        from homulator_b200.replay import bsgs_trace, rotsum_trace, trace_counts
        pts = {i: ct_b[1][0] for i in range(16)}
        seqs = {}
        for name, tr in (("bsgs_4x4", bsgs_trace(4, 4)), ("rotsum_16", rotsum_trace(16))):
            keys = {r: evk for r in sorted({op[3] for op in tr if op[0] == "hrotate"})}
            row = {"ops": trace_counts(tr)}
            for mode, kw in (("launches_us", {}), ("graph_us", {"graph": True}), ("hoisted_graph_us", {"graph": True, "hoist": True})):
                rp = hml.Replay(ctx, L, tr, **kw).bind(ct_a[0], pts, keys, evk)
                rp.run()
                rp.run()
                row[mode] = lat(rp.run, iters=5)
                rp.close()
            seqs[name] = row
        extra["op_sequences"] = seqs
        extra["bsgs_sequence"] = {"ops": seqs["bsgs_4x4"]["ops"], "us": seqs["bsgs_4x4"]["launches_us"]}

    if sharded is not None:
        extra["limb_sharded"] = sharded
    cpu = None
    if not args.no_cpu_baseline:
        v, used = cpu_port_sample(3, 1)
        cpu = {"value": v, "unit": "us", "cores": used, "kind": "port",
               "sample": "3 hmult at the full config on one host core (oracle/oracle.c, scalar)"}

    in_bytes = 2 * 2 * L * W_bytes * Be
    out_bytes = 2 * (L - 1) * W_bytes * Be
    line = {
        "metric": METRIC, "value": us_per_op, "unit": "us", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_total / K, "higher_is_better": False, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64 residues (36-bit), arithmetic on the FP64 pipe", "data": "synthetic",
        "config": bench_config(world) if args.batch <= 0 else dict(bench_config(world), batch_per_gpu_per_step=B, ciphertexts_per_step=B * world),
        "e2e": {"value": e2e_us, "unit": "us", "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": out_bytes,
                "batch_per_gpu_per_step": Be, "host_cpu_affinity": numa},
        "gpu_launches": int(launches),
        # `value` is the SUSTAINED figure: 256 / n_gpus ciphertexts per step keep one GPU busy for over a second, and the boards of
        # this pool then sit at their 1000 W cap (clocks.sm_mhz vs sm_max_mhz below).  Round 1's line (170 us) was taken with
        # 32-ciphertext steps at 1965 MHz; the like-for-like figure of this tree is the one-chunk burst below.
        "value_one_chunk_at_burst_clocks": burst["hmult"] if rank == 0 and burst else None,
        "clocks": sampler.summary(),
        "roofline": {"bound": "hbm", "kernel": "ntt_fwd_cols + ntt_rows (forward NTT pair, 32 ciphertexts x 115 limbs per launch)",
                     "timed": "alone, before and after the step loop, the faster of the two (burst clocks, like the burst peak): extra.ntt_us_per_limb_before_step_loop / _sustained",
                     "achieved": ntt_gbs,
                     "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": ntt_gbs / peak, "traffic": traffic,
                     "algorithmic_bytes_per_launch": ntt_bytes},
        "cpu_baseline": cpu,
        "extra": extra,
    }
    _emit(real_stdout, line)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
