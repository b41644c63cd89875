#!/usr/bin/env python
"""Measure batched beam search (csrc/beam.cu) on the 1190 Miller-Schupp rows:

  * one engine run per max_relator_length group (split further only when an engine would exceed
    --max-bytes), for every node budget per row, beam width and cyclic flag of the grid: device time,
    expansions/s, rows solved and the rows solved that greedy search at 1e6 does not solve (listed);
  * bfs_batch on the same rows and budget, as the throughput reference;
  * beam meet-in-the-middle against a symmetric trivial_ball of --ball-nodes nodes per group.

Every solving path is replayed with the device ACMove and must end at total length 2.  A grid point that would
not end within --max-seconds of wall time (estimated from the same width at the smaller budget) is recorded as
not measured.

    python scripts/bench_beam_search.py [--budgets 1000000,10000000] [--widths 100,1000,10000,100000]
        [--ball-nodes 100000000] [--out profiles/beam_search_b200.json]

Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ac_solver_b200 import (beam_meet_in_the_middle, beam_search_batch, bfs_batch, greedy_search_batch,  # noqa: E402
                            trivial_ball)
from ac_solver_b200.envs.ac_moves import ac_moves_batch  # noqa: E402
from ac_solver_b200.search.miller_schupp import load_presentations_from_text_file  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (x.strip() for x in q.split(","))
    return {"gpu": name, "power_limit": power}


def replay_ok(rows, paths, cyclical):
    """Replay every path on the device (one batched move per step): True if each ends at total length 2 with
    every intermediate length as recorded."""
    if not paths:
        return True
    state = np.array(rows, np.int8)
    if any(int(np.count_nonzero(r)) != p[0][1] for r, p in zip(state, paths)):
        return False
    for t in range(1, max(len(p) for p in paths)):
        idx = [i for i, p in enumerate(paths) if len(p) > t]
        nxt, lens, status = ac_moves_batch(state[idx], np.array([paths[i][t][0] for i in idx], np.uint8),
                                           cyclical=cyclical)
        if status.any():
            return False
        state[idx] = nxt
        if any(int(lens[j].sum()) != paths[i][t][1] for j, i in enumerate(idx)):
            return False
    return all(int(np.count_nonzero(s)) == 2 for s in state)


def sweep(groups, fn, cyclical):
    """fn(rows) -> results, per group; -> (global row indices solved, device seconds, expansions, paths ok)."""
    solved, dev, expanded, ok = [], 0.0, 0, True
    for mrl, (idx, P) in groups.items():
        out = fn(P)
        dev += sum({r[2]["seconds_device"] for r in out})  # every engine's time once (a group may be split)
        expanded += sum(r[2]["n_expanded"] for r in out)
        hit = [k for k, r in enumerate(out) if r[0]]
        ok &= replay_ok(P[hit], [out[k][1] for k in hit], cyclical)
        solved += [int(idx[k]) for k in hit]
    return sorted(solved), dev, expanded, bool(ok)


def write(result, out):
    """The result so far to ``out`` (rewritten after every run, so a cut-off run keeps what it measured)."""
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            f.write(json.dumps(result) + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--budgets", default="1000000,10000000")
    ap.add_argument("--widths", default="100,1000,10000,100000")
    ap.add_argument("--ball-nodes", type=int, default=100_000_000)
    ap.add_argument("--mitm-width", type=int, default=1000)
    ap.add_argument("--max-bytes", type=int, default=64 << 30)
    ap.add_argument("--max-seconds", type=float, default=480.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    t_start = time.perf_counter()
    budgets = [int(float(x)) for x in args.budgets.split(",")]
    widths = [int(float(x)) for x in args.widths.split(",")]
    rows = load_presentations_from_text_file(
        os.path.join(ROOT, "ac_solver_b200", "search", "miller_schupp", "data", "all_presentations.txt"))
    by_width = {}
    for k, r in enumerate(rows):
        by_width.setdefault(len(r), []).append(k)
    groups = {w // 2: (np.array(ks), np.array([rows[k] for k in ks], np.int8)) for w, ks in sorted(by_width.items())}
    result = {"bench": "beam_search_miller_schupp", **gpu_info(), "rows": len(rows), "budgets_per_row": budgets,
              "widths": widths}

    beam_search_batch(groups[18][1][:2], 10, 1000)  # warm-up: module load and first launches
    bfs_batch(groups[18][1][:2], 1000)

    greedy, _, _, g_ok = sweep(groups, lambda P: greedy_search_batch(P, 1_000_000), False)
    greedy_set = set(greedy)
    result["greedy_1e6"] = {"solved": len(greedy), "paths_replay_to_length_2": g_ok}

    mitm = {"ball_nodes": args.ball_nodes, "width": args.mitm_width, "budget": budgets[0]}
    solved, via_ball, ok, dev = [], 0, True, 0.0
    for mrl, (idx, P) in groups.items():
        with trivial_ball(mrl, args.ball_nodes, symmetric=True) as ball:
            out = beam_meet_in_the_middle(P, args.mitm_width, budgets[0], ball, max_bytes=args.max_bytes)
        dev += out[0][2]["seconds_device"]
        hit = [k for k, r in enumerate(out) if r[0]]
        ok &= replay_ok(P[hit], [out[k][1] for k in hit], False)
        solved += [int(idx[k]) for k in hit]
        via_ball += sum(out[k][2].get("goal") is not None for k in hit)
    mitm.update({"trivialized": len(solved), "via_ball": via_ball, "forward_device_s": dev,
                 "not_solved_by_greedy_1e6": sorted(k for k in solved if k not in greedy_set),
                 "paths_replay_to_length_2": bool(ok)})
    result["meet_in_the_middle"] = mitm
    write(result, args.out)

    runs, skipped, wall = [], [], {}
    for budget in budgets:
        s, dev, exp, ok = sweep(groups, lambda P: bfs_batch(P, budget, max_bytes=args.max_bytes), False)
        runs.append({"engine": "bfs_batch", "budget": budget, "cyclical": False, "device_s": dev,
                     "expansions_per_s": exp / dev if dev else None, "solved": len(s),
                     "not_solved_by_greedy_1e6": [k for k in s if k not in greedy_set],
                     "paths_replay_to_length_2": ok})
        print(json.dumps(runs[-1]), flush=True)
        for width in sorted(widths, reverse=True):  # fewest levels first
            for cyc in (False, True):
                # a run takes about budget / width levels: skip one that would not end within --max-seconds
                guess = wall.get((width, cyc), (0.0, budget))
                guess = guess[0] * budget / guess[1]
                if time.perf_counter() - t_start + 1.5 * guess > args.max_seconds:
                    skipped.append({"budget": budget, "width": width, "cyclical": cyc})
                    continue
                t0 = time.perf_counter()
                s, dev, exp, ok = sweep(groups, lambda P: beam_search_batch(P, width, budget, None, cyc,
                                                                            max_bytes=args.max_bytes), cyc)
                runs.append({"engine": "beam", "budget": budget, "width": width, "cyclical": cyc, "device_s": dev,
                             "expansions_per_s": exp / dev if dev else None, "solved": len(s),
                             "not_solved_by_greedy_1e6": [k for k in s if k not in greedy_set],
                             "paths_replay_to_length_2": ok})
                wall[(width, cyc)] = (time.perf_counter() - t0, budget)
                print(json.dumps(runs[-1]), flush=True)
                result["runs"], result["not_measured"] = runs, skipped
                write(result, args.out)
    result["runs"] = runs
    result["not_measured"] = skipped

    result["wall_s"] = time.perf_counter() - t_start
    print(json.dumps(result))
    write(result, args.out)


if __name__ == "__main__":
    main()
