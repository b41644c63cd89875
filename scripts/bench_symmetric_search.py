#!/usr/bin/env python
"""Measure orbit search (bfs_batch(symmetric=True), csrc/ac_sym.cuh + csrc/mbfs.cu) on the Miller-Schupp rows:

  * the 1190-row sweep at one node budget, orbit search against exact search, for both
    cyclically_reduce_after_moves flags, alternated over repeats: device seconds per engine run (summed over
    the max_relator_length groups), solved counts, rows solved by only one of the two, and whether every
    row both solve has paths of the same length;
  * every orbit-search path is replayed from its row with the device ACMove and must end at total length 2
    with every recorded intermediate length;
  * symmetric trivial balls (one orbit search from <x, y>) per max_relator_length at several budgets: wall
    time, entries, distinct states and bytes; and BFS (exact and orbit forward search) and greedy
    meet-in-the-middle without cyclic reduction at the sweep budget against each ball: rows trivialized,
    every stitched path replayed.

    python scripts/bench_symmetric_search.py [--budget 1000000] [--repeats 3] [--out FILE]

Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import time  # noqa: E402

from ac_solver_b200 import bfs_batch, bfs_meet_in_the_middle, greedy_meet_in_the_middle, trivial_ball  # noqa: E402
from ac_solver_b200.envs.ac_moves import ac_moves_batch  # noqa: E402
from ac_solver_b200.search.miller_schupp import load_presentations_from_text_file  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (x.strip() for x in q.split(","))
    return {"gpu": name, "power_limit": power}


def replay_ok(rows, paths, cyclical):
    """Replay every path on the device (one batched move per step); True if each ends at total length 2
    with every intermediate length as recorded."""
    if not paths:
        return True
    state = np.array(rows, np.int8)
    for r, p in zip(state, paths):
        if int(np.count_nonzero(r)) != p[0][1]:
            return False
    for t in range(1, max(len(p) for p in paths)):
        idx = [i for i, p in enumerate(paths) if len(p) > t]
        nxt, lens, status = ac_moves_batch(state[idx], np.array([paths[i][t][0] for i in idx], np.uint8),
                                           cyclical=cyclical)
        if status.any():
            return False
        state[idx] = nxt
        for j, i in enumerate(idx):
            if int(lens[j].sum()) != paths[i][t][1]:
                return False
    return all(int(np.count_nonzero(s)) == 2 for s in state)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--budget", type=int, default=1_000_000)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--ball-budgets", default="1000000,10000000,100000000")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rows = load_presentations_from_text_file(
        os.path.join(ROOT, "ac_solver_b200", "search", "miller_schupp", "data", "all_presentations.txt"))
    by_width = {}
    for k, r in enumerate(rows):
        by_width.setdefault(len(r), []).append(k)
    groups = {w // 2: np.array([rows[k] for k in ks], np.int8) for w, ks in sorted(by_width.items())}
    row_index = {w // 2: ks for w, ks in by_width.items()}  # row numbers in all_presentations.txt
    result = {"bench": "symmetric_search_miller_schupp", **gpu_info(), "rows": len(rows), "budget": args.budget,
              "repeats": args.repeats}

    first = next(iter(groups.values()))
    for sym in (False, True):  # warm-up: module load and first launches of both variants
        bfs_batch(first[:2], 1000, symmetric=sym)

    for cyc in (False, True):
        secs = {"exact": [], "symmetric": []}
        answers = {}
        for rep in range(args.repeats):
            order = ("exact", "symmetric") if rep % 2 == 0 else ("symmetric", "exact")
            for name in order:
                tot = 0.0
                for mrl, P in groups.items():
                    out = bfs_batch(P, args.budget, cyc, symmetric=(name == "symmetric"))
                    tot += out[0][2]["seconds_device"]
                    if rep == 0:
                        answers.setdefault(name, {})[mrl] = out
                secs[name].append(tot)
        ex, sy = answers["exact"], answers["symmetric"]
        only_exact, only_sym, both, same_len, all_ok, visited = [], [], 0, True, True, {"exact": 0, "symmetric": 0}
        for mrl, P in groups.items():
            for k in range(len(P)):
                a, b = ex[mrl][k], sy[mrl][k]
                visited["exact"] += a[2]["n_visited"]
                visited["symmetric"] += b[2]["n_visited"]
                if a[0] and b[0]:
                    both += 1
                    same_len &= len(a[1]) == len(b[1])
                elif a[0]:
                    only_exact.append(row_index[mrl][k])
                elif b[0]:
                    only_sym.append(row_index[mrl][k])
            ok = [k for k in range(len(P)) if sy[mrl][k][0]]
            all_ok &= replay_ok(P[ok], [sy[mrl][k][1] for k in ok], cyc)
        result["cyclical" if cyc else "plain"] = {
            "device_s": secs,
            "device_s_median": {n: float(np.median(v)) for n, v in secs.items()},
            "solved": {"exact": sum(r[0] for o in ex.values() for r in o),
                       "symmetric": sum(r[0] for o in sy.values() for r in o)},
            "solved_by_both": both, "same_path_length_on_both": bool(same_len),
            "only_exact": only_exact, "only_symmetric": only_sym,
            "states_visited_total": visited,
            "symmetric_paths_replay_to_length_2": bool(all_ok),
        }
        print(json.dumps({"cyclical": cyc, **result["cyclical" if cyc else "plain"]}), file=sys.stderr)
    balls, mitm = [], []
    for bb in [int(x) for x in args.ball_budgets.split(",")]:
        tot = {"bfs": 0, "bfs_orbit": 0, "greedy": 0}
        ok_all = True
        for mrl, P in groups.items():
            t0 = time.perf_counter()
            ball = trivial_ball(mrl, bb, symmetric=True)
            wall = time.perf_counter() - t0
            try:
                balls.append({"mrl": mrl, "budget": bb, "wall_s": wall, "entries": ball.n_entries,
                              "states": ball.n_states, "goal_set_bytes": ball.nbytes})
                runs = {"bfs": bfs_meet_in_the_middle(P, args.budget, ball),
                        "bfs_orbit": bfs_meet_in_the_middle(P, args.budget, ball, symmetric=True),
                        "greedy": greedy_meet_in_the_middle(P, args.budget, ball)}
            finally:
                ball.close()
            for name, out in runs.items():
                ok = [k for k, r in enumerate(out) if r[0]]
                ok_all &= replay_ok(P[ok], [out[k][1] for k in ok], False)
                tot[name] += len(ok)
        mitm.append({"ball_budget": bb, "trivialized": tot, "all_paths_replay_to_length_2": bool(ok_all)})
        print(json.dumps(mitm[-1]), file=sys.stderr)
    result["symmetric_balls"] = balls
    result["meet_in_the_middle"] = mitm
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
