"""torchrun worker: hoisted rotations on limb-sharded ciphertexts against textbook sharded rotations and one-GPU hoisted ones.

For rotsum_16 (rotsum_trace(16)) and bsgs_4x4 (bsgs_trace(4, 4)) at BASELINE.json's north star (N = 2^16, maxLevel 45, L 35,
alpha 15) it times, with CUDA events, the maximum over ranks of:
  textbook sharded, as launches and as one CUDA graph per rank
  hoisted sharded (max_rot 16: one exchange group per run of rotations), as launches and as one graph
  one-GPU hoisted, as one graph (rank 0's device, the others idle)
and checks that the sharded hoisted results equal the one-GPU hoisted replay bit for bit.  Prints ONE JSON line with the card
name, power limit and SM clock read in the same run.
Run as: python -m torch.distributed.run --nproc-per-node G --master-addr 127.0.0.1 profiles/sharded_hoisted.py [--reps R]"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import homulator_b200 as hml  # noqa: E402
from homulator_b200.replay import bsgs_trace, rotsum_trace, shard_operands  # noqa: E402


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                       capture_output=True, text=True)
    vals = [v.strip() for v in r.stdout.strip().split(",")] if r.returncode == 0 else []
    return dict(zip(("card", "power_limit", "sm_clock", "sm_clock_max"), vals)) if len(vals) == 4 else {"card": torch.cuda.get_device_name()}


def main():
    reps = int(sys.argv[sys.argv.index("--reps") + 1]) if "--reps" in sys.argv else 20
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    N, ML, L, A = 65536, 45, 35, 15
    ctx = hml.Context(N=N, max_level=ML, alpha=A, device=local)
    q = list(range(L))
    x = ctx.uniform(q, 1, lead=(2,))
    evk = ctx.uniform(ctx.ext_mod_idx(L), 3, lead=(3, 2))
    pts = {i: ctx.uniform(q, 200 + i) for i in range(16)}
    traces = {"rotsum_16": rotsum_trace(16), "bsgs_4x4": bsgs_trace(4, 4)}
    rots = sorted({op[3] for tr in traces.values() for op in tr if op[0] == "hrotate"})
    keys = {r: ctx.uniform(ctx.ext_mod_idx(L), 100 + r, lead=(3, 2)) for r in rots}

    def exchange(obj):
        out = [None] * world
        dist.all_gather_object(out, obj)
        return out

    def timeit(fn, on=True):
        """device-event time of one fn() on this rank (0 where `on` is False), maximum over ranks"""
        if on:
            for _ in range(3):
                fn()
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps if on else 0):
            fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) * 1e3 / reps if on else 0.0], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return round(float(t), 1)

    sh = hml.Shard.ipc(ctx, L, rank, world, exchange, max_rot=16)
    sh.prepare(L)
    x_own, pts_own, keys_own, evk_own = shard_operands(sh, L, x, pts, keys, evk)
    keep = torch.tensor([i for i in sh.own_q(L) if i < L - 1], device="cuda", dtype=torch.long)
    res, same = {}, True
    for name, tr in traces.items():
        one = hml.Replay(ctx, L, tr, graph=True, hoist=True).bind(x, pts, keys, evk)
        want = one.run().result("z").clone()
        r = {"one_gpu_hoisted_graph_us": timeit(one.run, rank == 0)}
        one.close()
        for hoist in (False, True):
            for graph in (False, True):
                rp = hml.Replay(ctx, L, tr, shard=sh, graph=graph, hoist=hoist).bind(x_own, pts_own, keys_own, evk_own)
                r["%s_sharded_%s_us" % ("hoisted" if hoist else "textbook", "graph" if graph else "launches")] = timeit(rp.run)
                if hoist:
                    got = rp.result("z")
                    torch.cuda.synchronize()
                    same = same and torch.equal(got.contiguous(), want[:, keep])
                dist.barrier()
                rp.close()
        res[name] = r
    sh.check()
    flag = torch.tensor([1 if same else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        line = {"world": world, **card(), "N": N, "L": L, "alpha": A, "reps": reps, "timing": "CUDA events, max over ranks"}
        line.update(res)
        line["hoisted_sharded_matches_one_gpu_hoisted"] = bool(int(flag))
        print(json.dumps(line))
    dist.barrier()
    torch.cuda.synchronize()
    sh.close()
    dist.barrier()
    dist.destroy_process_group()
    return 0 if int(flag) == 1 else 1


if __name__ == "__main__":
    sys.exit(main())
