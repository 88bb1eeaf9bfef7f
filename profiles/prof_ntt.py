"""Profiling driver for the forward transform on the launch shape bench.py's roofline times (32 ciphertexts x 115 limbs):
    python profiles/prof_ntt.py [n_warm] [n_prof]"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import homulator_b200 as hml  # noqa: E402
n_warm = int(sys.argv[1]) if len(sys.argv) > 1 else 2
n_prof = int(sys.argv[2]) if len(sys.argv) > 2 else 1
ctx = hml.Context(os.path.join(ROOT, "config", "config_4.cfg"), 45, 15)
idx = [ctx.ext_mod_idx(35)[i % 50] for i in range(115)]
bufs = [ctx.uniform(idx, 50 + i, lead=(32,)) for i in range(2)]
dst = ctx.empty(32, 115, 65536)
torch.cuda.synchronize()
for i in range(n_warm + n_prof):
    ctx.ntt_batch(bufs[i % 2], idx, out=dst)
torch.cuda.synchronize()
print("done")
