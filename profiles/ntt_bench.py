"""Transform microbenchmark: microseconds per launch of hml_ntt / hml_intt at several limb counts (one ciphertext-sized
launch each) and per limb on the batched ModUp shape (32 x 115 limbs)."""
import os, sys, torch
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import homulator_b200 as hml
ctx = hml.Context(os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "config", "config_4.cfg"), 45, 15)
L = 35
idx = [ctx.ext_mod_idx(L)[i % 50] for i in range(115)]
def t(fn, reps=10):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3
bufs = [ctx.uniform(idx, 50 + i, lead=(32,)) for i in range(2)]
dst = ctx.empty(32, 115, 65536)
k = [0]
def batched(inv):
    def f():
        k[0] += 1; ctx.ntt_batch(bufs[k[0] % 2], idx, out=dst, inverse=inv)
    return f
def single(n, inv):
    def f():
        k[0] += 1; ctx.ntt(bufs[k[0] % 2][k[0] % 32][:n], idx[:n], out=dst[0][:n], inverse=inv)
    return f
row = {"fwd_batched_us_per_limb": t(batched(False)) / (115 * 32), "inv_batched_us_per_limb": t(batched(True)) / (115 * 32)}
for n in (2, 7, 16, 35, 70, 115):
    row["fwd_%d" % n] = t(single(n, False), 20)
    row["inv_%d" % n] = t(single(n, True), 20)
print(" ".join("%s=%.3f" % kv for kv in row.items()))
