"""hml_exec_counts of every op pinned against tests/golden/exec_counts.json (written by tests/golden/gen_exec_counts.py).

The counters are the launch and limb tallies that the profile scripts and the trace comparisons rely on; they follow from
the launch sequence of each op alone.  The golden file records them for the one-GPU, batched, host-buffer and limb-sharded
ops on a single-pass ring, a small two-pass ring and the north-star ring."""
import json
import os
import sys

import pytest

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import gen_exec_counts as gen  # noqa: E402


@pytest.mark.parametrize("shape", list(gen.SHAPES))
def test_exec_counts_match_golden(shape):
    with open(gen.GOLDEN) as f:
        golden = {k: v for k, v in json.load(f).items() if k.split("/")[0] == shape}
    got = gen.run_shape(shape)
    assert sorted(got) == sorted(golden)
    for case in golden:
        assert got[case] == golden[case], case
