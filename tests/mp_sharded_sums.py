"""torchrun worker: the double-hoisted rotation sum and the lazily relinearised product sum on limb-sharded ciphertexts, one rank
per GPU, peer-direct over NVLink.  Shard.hrotate_sum_hoisted (hml_hrotate_sum_hoisted_sharded) and Shard.hmult_sum
(hml_hmult_sum_sharded) against the single-GPU Context.hrotate_sum_hoisted / Context.hmult_sum, at BASELINE.json's north star
(N = 2^16, maxLevel 45, L 35, alpha 15), 17 rotations and 17 products (two kernel groups each, one square).  Rank 0 prints
SHARDED_SUMS_OK, then one line "SHARDED_SUMS_TIME {json}" with the median device time of each op over 5 runs (microseconds,
16 rotations / 16 products), read by profiles/sharded_sums.py.
Run as: python -m torch.distributed.run --nproc-per-node G --master-addr 127.0.0.1 tests/mp_sharded_sums.py"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import homulator_b200 as hml  # noqa: E402
from homulator_b200.replay import shard_plaintexts  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    N, ML, L, A = 65536, 45, 35, 15
    n = 17
    ctx = hml.Context(N=N, max_level=ML, alpha=A, device=local)
    q, ext, beta = list(range(L)), ctx.ext_mod_idx(L), ctx.beta(L)
    ct = ctx.uniform(q, 1, lead=(2,))
    keys = [ctx.uniform(ext, 100 + i, lead=(beta, 2)) for i in range(n)]
    pts = [ctx.uniform(ext, 200 + i) for i in range(n)]
    a = [ctx.uniform(q, 300 + i, lead=(2,)) for i in range(n)]
    b = [ctx.uniform(q, 400 + i, lead=(2,)) for i in range(n)]
    b[5] = a[5]
    evk = ctx.uniform(ext, 3, lead=(beta, 2))
    gs = [1, 2 * N - 1] + [pow(5, r, 2 * N) for r in range(1, n - 1)]
    want_rot = ctx.hrotate_sum_hoisted(L, ct, keys, gs, pts)
    want_mul = ctx.hmult_sum(L, a, b, evk)

    def exchange(obj):
        out = [None] * world
        dist.all_gather_object(out, obj)
        return out

    sh = hml.Shard.ipc(ctx, L, rank, world, exchange, max_rot=4)
    sh.prepare(L)
    oi = torch.tensor(sh.own_q(L), device="cuda", dtype=torch.long)
    oe = torch.tensor(sh.own_ext(L), device="cuda", dtype=torch.long)
    keep = [i for i in sh.own_q(L) if i < L - 1]
    ct_own = ct[:, oi].contiguous()
    keys_own = [k[:, :, oe].contiguous() for k in keys]
    pts_own = shard_plaintexts(sh, L, pts)
    a_own = [t[:, oi].contiguous() for t in a]
    b_own = [t[:, oi].contiguous() for t in b]
    b_own[5] = a_own[5]
    evk_own = evk[:, :, oe].contiguous()
    dist.barrier()
    ok = True
    for _ in range(2):
        rot = sh.hrotate_sum_hoisted(L, ct_own, keys_own, gs, pts_own)
        mul = sh.hmult_sum(L, a_own, b_own, evk_own)
        torch.cuda.synchronize()
        ok = ok and torch.equal(rot, want_rot[:, oi])
        ok = ok and (not keep or torch.equal(mul[:, :len(keep)], want_mul[:, keep]))
    dist.barrier()

    def timed(fn, reps=5):
        ts = []
        for _ in range(reps):
            dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1000.0)
        return sorted(ts)[len(ts) // 2]

    t_rot = timed(lambda: sh.hrotate_sum_hoisted(L, ct_own, keys_own[:16], gs[:16], pts_own[:16]))
    t_mul = timed(lambda: sh.hmult_sum(L, a_own[:16], b_own[:16], evk_own))
    sh.check()
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("SHARDED_SUMS_OK" if int(flag) == 1 else "SHARDED_SUMS_MISMATCH")
        print("SHARDED_SUMS_TIME " + json.dumps({"world": world, "gpu": torch.cuda.get_device_name(local),
                                                 "rotsum16_us": round(t_rot, 1), "hmult_sum16_us": round(t_mul, 1)}))
    dist.barrier()
    torch.cuda.synchronize()
    sh.close()
    dist.barrier()
    dist.destroy_process_group()
    return 0 if int(flag) == 1 else 1


if __name__ == "__main__":
    sys.exit(main())
