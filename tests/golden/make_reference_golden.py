#!/usr/bin/env python3
"""Writes tests/golden/reference_golden.json: the reference's side of every comparison with the UNMODIFIED reference in the
suite (tests/reference_golden.py).  Needs oracle/_ref (make -C oracle -f ref_build.mk, from the reference sources); the
benched batch is built on a CUDA device, so where there is none its stored entry is kept.
Usage: python tests/golden/make_reference_golden.py [module ...]"""
import importlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path[:0] = [os.path.dirname(TESTS), TESTS]
import ref_lib  # noqa: E402
from reference_golden import PATH  # noqa: E402

MODULES = ["test_ref_vs_oracle", "test_rule_cores_host", "test_cfr_oracle", "test_mcts_oracle_vs_reference", "test_mccfr_oracle",
           "test_os_mccfr_oracle", "test_trajectories_oracle", "test_serialization", "test_gpu_vs_reference", "test_gpu_cfr",
           "test_gpu_serialization", "test_gpu_mcts", "test_gpu_bench_workload"]
NEEDS_CUDA = ["test_gpu_bench_workload"]

assert ref_lib.available(), "build oracle/_ref first (make -C oracle -f ref_build.mk)"
modules = sys.argv[1:] or MODULES
out = json.load(open(PATH)) if os.path.exists(PATH) else {}
for name in modules:
    if name in NEEDS_CUDA:
        import torch
        if not torch.cuda.is_available():
            print("kept", name, "(no CUDA device)")
            continue
    entries = importlib.import_module(name).reference_golden()
    out.update(entries)
    print(name, len(entries), "entries")
with open(PATH, "w") as f:
    json.dump(out, f, indent=0, sort_keys=True)
    f.write("\n")
print("wrote", PATH, os.path.getsize(PATH), "bytes")
