#!/usr/bin/env python
"""Measure goal-set search on the Miller-Schupp rows (csrc/goalset.cu, the goal test of csrc/mbfs.cu):

  * trivial_ball per max_relator_length at several per-root budgets: wall time, entries, distinct
    states, the exploring engine's bytes and the goal set's bytes;
  * the 1190-row sweep at a forward budget of 1e6, plain against a goal set of the 8 trivial states
    (same answers, so the difference is the lookup kernel), device time per engine, alternated;
  * bfs_meet_in_the_middle at the same forward budget against each ball: rows trivialized against
    plain BFS.  Every stitched path is replayed with the device ACMove and must end at total length 2.

    python scripts/bench_goal_search.py [--budget 1000000] [--ball-budgets 1000000,10000000] [--out FILE]

Prints one JSON line.
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
from ac_solver_b200 import GoalSet, _lib, bfs_batch, bfs_meet_in_the_middle, trivial_ball  # noqa: E402
from ac_solver_b200.envs.ac_moves import ac_moves_batch  # noqa: E402
from ac_solver_b200.envs.utils import generate_trivial_states  # noqa: E402
from ac_solver_b200.search.miller_schupp import load_presentations_from_text_file  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (x.strip() for x in q.split(","))
    return {"gpu": name, "power_limit": power}


def engine_bytes(n, mrl, budget):
    b, budgets = C.c_int64(0), np.full(n, budget, np.int64)
    _lib.check(_lib.lib().acs_bfs_batch_bytes(n, mrl, budgets.ctypes.data, 0, C.byref(b)))
    return int(b.value)


def replay_ok(rows, paths):
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
        nxt, lens, status = ac_moves_batch(state[idx], np.array([paths[i][t][0] for i in idx], np.uint8), cyclical=False)
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
    ap.add_argument("--ball-budgets", default="1000000,10000000,100000000")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ball_budgets = [int(x) for x in args.ball_budgets.split(",")]
    rows = load_presentations_from_text_file(
        os.path.join(ROOT, "ac_solver_b200", "search", "miller_schupp", "data", "all_presentations.txt"))
    by_width = {}
    for k, r in enumerate(rows):
        by_width.setdefault(len(r), []).append(k)
    groups = {w // 2: np.array([rows[k] for k in ks], np.int8) for w, ks in sorted(by_width.items())}
    result = {"bench": "goal_search_miller_schupp", **gpu_info(), "rows": len(rows), "forward_budget": args.budget,
              "ball_budgets_per_root": ball_budgets}

    bfs_batch(groups[18][:2], 1000)  # warm-up: module load and first launches
    with trivial_ball(18, 1000) as b:
        bfs_meet_in_the_middle(groups[18][:2], 1000, b)

    # 1. the sweep, plain against the 8 trivial states as goals (identical answers: the solve wins ties)
    sweep = {"plain": {}, "trivial_goals": {}}
    for rep in range(args.repeats):
        for mrl, P in groups.items():
            with GoalSet.from_rows(generate_trivial_states(mrl)) as g:
                for name, goals in (("plain", None), ("trivial_goals", g)) if rep % 2 == 0 else \
                        (("trivial_goals", g), ("plain", None)):
                    out = bfs_batch(P, args.budget, goals=goals)
                    sweep[name].setdefault(str(mrl), []).append(out[0][2]["seconds_device"])
                    if rep == 0 and name == "plain":
                        sweep.setdefault("plain_solved", {})[str(mrl)] = int(sum(r[0] for r in out))
                    if rep == 0 and name == "trivial_goals":
                        sweep.setdefault("trivial_goals_solved", {})[str(mrl)] = int(sum(r[0] for r in out))
    for name in ("plain", "trivial_goals"):
        sweep[name + "_device_s_total_median"] = float(np.median(
            [sum(sweep[name][str(m)][i] for m in groups) for i in range(args.repeats)]))
    result["sweep"] = sweep
    plain_total = sum(sweep["plain_solved"].values())

    # 2. balls and meet-in-the-middle
    balls, mitm = [], []
    for bb in ball_budgets:
        tot_triv, tot_met, all_ok, mitm_dev = 0, 0, True, 0.0
        for mrl, P in groups.items():
            t0 = time.perf_counter()
            ball = trivial_ball(mrl, bb)
            wall = time.perf_counter() - t0
            try:
                balls.append({"mrl": mrl, "budget_per_root": bb, "wall_s": wall,
                              "device_s": ball.results[0][2]["seconds_device"], "entries": ball.n_entries,
                              "states": ball.n_states, "engine_bytes": engine_bytes(8, mrl, bb),
                              "goal_set_bytes": ball.nbytes,
                              "raising_roots": sum(r[2]["status"] != 0 for r in ball.results)})
                out = bfs_meet_in_the_middle(P, args.budget, ball)
            finally:
                ball.close()
            mitm_dev += out[0][2]["seconds_device"]
            ok = [k for k, r in enumerate(out) if r[0]]
            all_ok &= replay_ok(P[ok], [out[k][1] for k in ok])
            tot_triv += len(ok)
            tot_met += sum(out[k][2].get("goal") is not None for k in ok)
        mitm.append({"ball_budget_per_root": bb, "trivialized": tot_triv, "via_ball": tot_met,
                     "plain_bfs_solved": plain_total, "all_paths_replay_to_length_2": bool(all_ok),
                     "forward_device_s_total": mitm_dev})
    result["balls"] = balls
    result["meet_in_the_middle"] = mitm
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
