"""torchrun worker: hoisted rotations on limb-sharded ciphertexts, one rank per GPU, peer-direct over NVLink.
Shard.hrotate_hoisted (hml_hrotate_hoisted_sharded) against the single-GPU Context.hrotate_hoisted, then the 16-rotation sum
(rotsum_trace(16)) replayed hoisted and sharded, as launches and as one CUDA graph per rank, against the single-GPU hoisted
replay.  Everything at BASELINE.json's north star (N = 2^16, maxLevel 45, L 35, alpha 15).
Run as: python -m torch.distributed.run --nproc-per-node G --master-addr 127.0.0.1 tests/mp_sharded_hoisted.py"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import homulator_b200 as hml  # noqa: E402
from homulator_b200.replay import rotsum_trace, shard_operands  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    N, ML, L, A = 65536, 45, 35, 15
    ctx = hml.Context(N=N, max_level=ML, alpha=A, device=local)
    q = list(range(L))
    x = ctx.uniform(q, 1, lead=(2,))
    evk = ctx.uniform(ctx.ext_mod_idx(L), 3, lead=(3, 2))
    tr = rotsum_trace(16)
    rots = sorted({op[3] for op in tr if op[0] == "hrotate"})
    keys = {r: ctx.uniform(ctx.ext_mod_idx(L), 100 + r, lead=(3, 2)) for r in rots}
    pts = {i: ctx.uniform(q, 200 + i) for i in range(16)}

    def exchange(obj):
        out = [None] * world
        dist.all_gather_object(out, obj)
        return out

    ok = True
    # max_rot 4: the 16 rotations run as four groups (with the extra exchanges between them)
    sh = hml.Shard.ipc(ctx, L, rank, world, exchange, max_rot=4)
    sh.prepare(L)
    x_own, pts_own, keys_own, evk_own = shard_operands(sh, L, x, pts, keys, evk)
    oi = torch.tensor(sh.own_q(L), device="cuda", dtype=torch.long)
    gs = [pow(5, r, 2 * N) for r in rots[:6]] + [2 * N - 1]
    rk = [keys[r] for r in rots[:6]] + [keys[rots[0]]]
    ref = ctx.hrotate_hoisted(L, x, rk, gs)
    dist.barrier()
    for _ in range(2):
        got = sh.hrotate_hoisted(L, x_own, [k[:, :, torch.tensor(sh.own_ext(L), device="cuda")].contiguous() for k in rk], gs)
        torch.cuda.synchronize()
        for g, w in zip(got, ref):
            ok = ok and torch.equal(g, w[:, oi])
    one = hml.Replay(ctx, L, tr, hoist=True).bind(x, pts, keys, evk)
    want = one.run().result("z").clone()
    keep = torch.tensor([i for i in sh.own_q(L) if i < L - 1], device="cuda", dtype=torch.long)
    dist.barrier()
    for graph in (False, True):
        rp = hml.Replay(ctx, L, tr, shard=sh, graph=graph, hoist=True).bind(x_own, pts_own, keys_own, evk_own)
        for _ in range(2):
            got = rp.run().result("z")
            torch.cuda.synchronize()
            ok = ok and torch.equal(got.contiguous(), want[:, keep])
        dist.barrier()
        rp.close()
    sh.check()
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("SHARDED_HOISTED_OK" if int(flag) == 1 else "SHARDED_HOISTED_MISMATCH")
    dist.barrier()
    torch.cuda.synchronize()
    one.close()
    sh.close()
    dist.barrier()
    dist.destroy_process_group()
    return 0 if int(flag) == 1 else 1


if __name__ == "__main__":
    sys.exit(main())
