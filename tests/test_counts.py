"""CPU tests: the library's trace counts equal the reference's InsGen trace (tests/golden/ref_counts.json, produced
from the UNMODIFIED reference by oracle/ref_count_harness.cpp via tests/golden/gen_ref_counts.py), the C-ABI library
loads and exports every symbol include/homulator_b200.h declares, and the .cfg reader accepts the reference format."""
import ctypes
import json
import os
import re

import pytest

import homulator_b200 as hml
from homulator_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "ref_counts.json")))


@pytest.mark.parametrize("rec", GOLD, ids=lambda r: "%s-%s-%d-%d-%d" % (r["cfg"], r["op"], r["maxLevel"], r["L"], r["alpha"]))
def test_trace_counts_equal_reference(rec):
    got = hml.trace_counts(rec["op"], rec["N"], rec["batchSize"], rec["maxLevel"], rec["L"], rec["alpha"], 2, 6)
    for opc in ("NTT", "INTT", "MULT", "BCONV_STEP2", "AUTO"):
        assert got[opc] == rec["by_opcode"].get(opc, 0), opc
    assert got["total"] == rec["total"]
    assert got["driverTotal"] == rec["driverTotal"]
    # per stage (label|opcode), as tallied from Instruction::Name by the harness
    mine = {}
    for st in got["stages"]:
        if st["instructions"]:
            key = st["label"] + "|" + st["opcode"]
            mine[key] = mine.get(key, 0) + st["instructions"]
    assert mine == rec["by_stage"]


def test_closed_forms_survey_3_4():
    """SURVEY.md 3.4 closed forms, limb-ops, at the north-star shape."""
    L, a = 35, 15
    beta, E = 3, 50
    c = hml.trace_counts("hmult", 65536, 256, 45, L, a)
    bc = 256
    assert c["INTT"] // bc == (L + 2 * a + 2 * L) + 2
    assert c["NTT"] // bc == beta * E + 2
    assert c["BCONV_STEP2"] // bc == 15 * 35 + 15 * 35 + 5 * 45 + 2 * a * L
    assert c["MULT"] // bc == (L + 2 * E * (beta - 1) + 2 * a + 2 * L) + 3 * L + 2 * L + 4 * (L - 1)


def test_unknown_op_and_bad_level():
    with pytest.raises(hml.HmlError) as e:
        hml.trace_counts("hrot", 65536, 256, 45, 35, 15)
    assert e.value.code == 5  # HML_ERR_OP, reference prints "Error operation requirement..."
    with pytest.raises(hml.HmlError):
        hml.trace_counts("hmult", 65536, 256, 45, 1, 15)  # reference segfaults at L=1; we refuse


def test_library_exports_every_declared_symbol():
    lib = hml.load_library()
    header = open(os.path.join(ROOT, "include", "homulator_b200.h")).read()
    declared = set(re.findall(r"\b(hml_[a-z0-9_]+)\s*\(", header))
    declared -= {"hml_status"}
    assert declared, "no declarations parsed"
    assert declared == set(api.EXPORTS)
    for name in sorted(declared):
        assert hasattr(lib, name), name
        getattr(lib, name)


def test_context_creation_fails_loudly_without_gpu_or_with_bad_config():
    import torch
    lib = hml.load_library()
    h = ctypes.c_void_p()
    rc = lib.hml_ctx_create(b"/nonexistent/config.cfg", 45, 15, 0, ctypes.byref(h))
    assert rc == 2 and b"config" in lib.hml_last_create_error().lower()
    rc = lib.hml_ctx_create_params(65536, 60, 256, 45, 15, 0, ctypes.byref(h))
    assert rc == 4  # elementBitWidth outside the FP64 datapath's range
    if not torch.cuda.is_available():
        rc = lib.hml_ctx_create(os.path.join(ROOT, "config", "config_4.cfg").encode(), 45, 15, 0, ctypes.byref(h))
        assert rc == 3 and b"no cpu fallback" in lib.hml_last_create_error().lower()
        with pytest.raises(hml.HmlError):
            hml.Context(os.path.join(ROOT, "config", "config_4.cfg"), 45, 15)


def test_cli_usage_and_unknown_op(capfd):
    lib = hml.load_library()

    def run(args):
        argv = (ctypes.c_char_p * len(args))(*[a.encode() for a in args])
        return lib.hml_cli_main(len(args), argv)

    assert run(["Homulator.run", "x.cfg"]) == 1  # reference: usage on stderr, exit 1 (bench_micro24.cpp:6-9)
    err = capfd.readouterr().err
    assert "Usage:" in err
    cfg = os.path.join(ROOT, "config", "config_4.cfg")
    assert run(["Homulator.run", cfg, "hrot", "45", "35", "15"]) == 0  # reference: message, exit 0 (:49-51)
    out = capfd.readouterr().out
    assert "Error operation requirement, please double confirm!" in out
    assert "Configuration details are as follow:" in out and "elementBitWidth" in out
    assert run(["Homulator.run", "/nonexistent.cfg", "hmult", "45", "35", "15"]) == 2


def test_bench_reference_arm_prints_exactly_one_json_line():
    """bench.py --impl reference (the CPU arm the driver times beside the GPU arm): stdout is ONE JSON line with the contract's
    keys; under a multi-rank launch only rank 0 works and prints."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--no-extra"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-1000:]
    lines = [x for x in r.stdout.splitlines() if x.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "us" and d["higher_is_better"] is False and d["value"] > 0
    for k in ("metric", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    r1 = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert r1.returncode == 0 and r1.stdout.strip() == ""


def test_bench_dump_outputs_and_steps(tmp_path):
    """bench.py --dump-outputs samples the same positions of every row on every run, exactly and within its byte budget;
    --steps below 1 is refused rather than rounded up"""
    import subprocess
    import sys
    import numpy as np
    import torch
    import bench
    out = torch.randint(0, 1 << 36, (3, 2, 5, 4096), dtype=torch.int64)
    for name in ("a", "b"):
        bench.dump_outputs(str(tmp_path / "d"), name, out, 1 << 16, torch)
    a, b = np.load(tmp_path / "d" / "a.npy"), np.load(tmp_path / "d" / "b.npy")
    assert a.dtype == np.float64 and a.shape == (3, 2, 5, (1 << 16) // (8 * 30)) and a.nbytes <= 1 << 16
    assert np.array_equal(a, b)
    rows, got = out.reshape(30, -1).numpy(), a.reshape(30, -1)
    assert all(np.isin(got[i], rows[i]).all() for i in range(30))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 2 and "--steps" in r.stderr
