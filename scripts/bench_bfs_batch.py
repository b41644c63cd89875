#!/usr/bin/env python
"""Time the batched breadth-first sweep: all 1190 Miller-Schupp rows at a node budget of 1e6, once
per ``cyclically_reduce_after_moves`` flag, through ``bfs_groups`` (one engine per max_relator_length),
against single ``bfs_device`` calls on a fixed sample of rows timed in the same process.

    python scripts/bench_bfs_batch.py [--budget 1000000] [--sample-step 119] [--out FILE]

Prints one JSON line.  The per-row baseline is a sample; its extrapolation to all rows is labelled.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ac_solver_b200 import _lib  # noqa: E402
from ac_solver_b200.search.breadth_first import bfs_device, bfs_groups  # noqa: E402
from ac_solver_b200.search.miller_schupp import load_presentations_from_text_file  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (x.strip() for x in q.split(","))
    return {"gpu": name, "power_limit": power}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--budget", type=int, default=1_000_000)
    ap.add_argument("--sample-step", type=int, default=119)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rows = load_presentations_from_text_file(
        os.path.join(ROOT, "ac_solver_b200", "search", "miller_schupp", "data", "all_presentations.txt"))
    by_width = {}
    for k, r in enumerate(rows):
        by_width.setdefault(len(r), []).append(k)
    keys = list(by_width.values())
    groups = [np.array([rows[k] for k in ks], np.int8) for ks in keys]
    L = _lib.lib()
    engine_bytes = {}
    for g in groups:
        b, budgets = C.c_int64(0), np.full(g.shape[0], args.budget, np.int64)
        _lib.check(L.acs_bfs_batch_bytes(g.shape[0], g.shape[1] // 2, budgets.ctypes.data, 0, C.byref(b)))
        engine_bytes[str(g.shape[1] // 2)] = {"rows": int(g.shape[0]), "bytes": int(b.value)}
    result = {"bench": "bfs_batch_miller_schupp_sweep", **gpu_info(), "rows": len(rows), "budget": args.budget,
              "engine_bytes_by_mrl": engine_bytes}
    bfs_groups([g[:2] for g in groups], 1000, False)  # warm-up: module load and first launches of every kernel
    bfs_groups([g[:2] for g in groups], 1000, True)
    for cyc in (True, False):
        t0 = time.perf_counter()
        outs = bfs_groups(groups, args.budget, cyc)
        wall = time.perf_counter() - t0
        flat = [r for out in outs for r in out]
        expanded = sum(r[2]["n_expanded"] for r in flat)
        result[f"cyclical_{cyc}"] = {
            "wall_s": wall,
            # engines of different mrl run concurrently; each reports its own device time
            "device_s_per_engine_max": max(out[0][2]["seconds_device"] for out in outs),
            "searches": len(flat), "solved": sum(r[0] for r in flat),
            "visited_total": sum(r[2]["n_visited"] for r in flat), "expanded_total": expanded,
            "expansions_per_s_wall": expanded / wall,
        }
    sample = list(range(0, len(rows), args.sample_step))
    for cyc in (True, False):
        t0 = time.perf_counter()
        for k in sample:
            bfs_device(np.array(rows[k], np.int8), args.budget, cyc)
        wall = time.perf_counter() - t0
        result[f"single_bfs_device_sample_cyclical_{cyc}"] = {
            "rows": sample, "wall_s": wall, "per_row_s": wall / len(sample),
            "extrapolated_to_all_rows_s": wall / len(sample) * len(rows),
        }
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
