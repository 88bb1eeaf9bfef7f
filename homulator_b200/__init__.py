"""homulator_b200 — B200-native RNS-CKKS primitive datapath behind Homulator's operation interface.

The product is the C-ABI shared library (include/homulator_b200.h, built in-tree by homulator_b200.build);
this package is the thin Python host mirror used by tests and bench.py.  There is no CPU fallback: every
compute call goes through libhomulator_b200.so and raises if the library or a CUDA device is missing.
"""
from .api import (Context, HmlError, HMULT, HROTATE, HADD, PMULT, PADD, lib_path, load_library, trace_counts,  # noqa: F401
                  algorithmic_words, shard_layout, Shard, Replay, group_op, group_hrotate_hoisted,
                  group_hrotate_sum_hoisted, group_hmult_sum, KEY_PACKED)

__all__ = ["Context", "HmlError", "HMULT", "HROTATE", "HADD", "PMULT", "PADD", "lib_path", "load_library",
           "trace_counts", "algorithmic_words", "shard_layout", "Shard", "Replay", "group_op", "group_hrotate_hoisted",
           "group_hrotate_sum_hoisted", "group_hmult_sum", "KEY_PACKED"]
