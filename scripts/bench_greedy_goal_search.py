#!/usr/bin/env python
"""Measure goal-set greedy search on the Miller-Schupp rows (the GOAL instantiations of csrc/greedy.cu and
csrc/greedy_bucket.cuh):

  * the 1190-row greedy sweep at a budget of 1e6 per max_relator_length group, plain against a goal set of
    the 8 trivial states (same answers, so the difference is the lookup), device time per group, alternated;
  * for each ball budget: one trivial_ball per max_relator_length, greedy_meet_in_the_middle and
    bfs_meet_in_the_middle against it at the same forward budget, then the ball is closed before the next
    group.  Rows trivialized by each and by their union, against plain greedy.  Every stitched path is
    replayed with the device ACMove and must end at total length 2.

    python scripts/bench_greedy_goal_search.py [--budget 1000000] [--ball-budgets 1000000,10000000] [--out FILE]

Prints one JSON line.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from ac_solver_b200 import (GoalSet, bfs_meet_in_the_middle, greedy_meet_in_the_middle,  # noqa: E402
                            greedy_search_batch, trivial_ball)
from ac_solver_b200.envs.utils import generate_trivial_states  # noqa: E402
from ac_solver_b200.search.miller_schupp import load_presentations_from_text_file  # noqa: E402
from bench_goal_search import gpu_info, replay_ok  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--budget", type=int, default=1_000_000)
    ap.add_argument("--ball-budgets", default="1000000,10000000,100000000")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ball_budgets = [int(x) for x in args.ball_budgets.split(",") if x]
    rows = load_presentations_from_text_file(
        os.path.join(ROOT, "ac_solver_b200", "search", "miller_schupp", "data", "all_presentations.txt"))
    by_width = {}
    for k, r in enumerate(rows):
        by_width.setdefault(len(r), []).append(k)
    groups = {w // 2: np.array([rows[k] for k in ks], np.int8) for w, ks in sorted(by_width.items())}
    result = {"bench": "greedy_goal_search_miller_schupp", **gpu_info(), "rows": len(rows), "forward_budget": args.budget,
              "ball_budgets_per_root": ball_budgets}

    greedy_search_batch(groups[18][:2], 1000)  # warm-up: module load and first launches of both instantiations
    with GoalSet.from_rows(generate_trivial_states(18)) as g:
        greedy_search_batch(groups[18][:2], 1000, goals=g)

    # 1. the sweep, plain against the 8 trivial states as goals (identical answers: the solve wins ties)
    sweep = {"plain": {}, "trivial_goals": {}}
    answers = {}
    identical = True
    for rep in range(args.repeats):
        for mrl, P in groups.items():
            with GoalSet.from_rows(generate_trivial_states(mrl)) as g:
                order = (("plain", None), ("trivial_goals", g))
                for name, goals in (order if rep % 2 == 0 else order[::-1]):
                    out = greedy_search_batch(P, args.budget, goals=goals)
                    sweep[name].setdefault(str(mrl), []).append(out[0][2]["seconds_device"])
                    key = [(r[0], r[1], r[2]["n_visited"], r[2]["n_moves"]) for r in out]
                    if goals is not None:
                        identical &= all(r[2]["goal"] is None for r in out)
                    if (rep, mrl) in answers:
                        identical &= answers[(rep, mrl)] == key
                    answers[(rep, mrl)] = key
                    if rep == 0:
                        sweep.setdefault(name + "_solved", {})[str(mrl)] = int(sum(r[0] for r in out))
    for name in ("plain", "trivial_goals"):
        sweep[name + "_device_s_total_median"] = float(np.median(
            [sum(sweep[name][str(m)][i] for m in groups) for i in range(args.repeats)]))
    sweep["answers_identical"] = bool(identical)
    result["sweep"] = sweep
    plain_total = sum(sweep["plain_solved"].values())

    # 2. meet-in-the-middle, greedy and BFS, against one ball per max_relator_length (one at a time)
    mitm = []
    for bb in ball_budgets:
        res = {"ball_budget_per_root": bb, "greedy_mitm": 0, "greedy_via_ball": 0, "bfs_mitm": 0, "bfs_via_ball": 0,
               "union": 0, "plain_greedy_solved": plain_total, "plain_greedy_solved_lost": 0,
               "all_paths_replay_to_length_2": True, "ball_wall_s": 0.0, "greedy_device_s": 0.0, "bfs_device_s": 0.0}
        for mrl, P in groups.items():
            t0 = time.perf_counter()
            ball = trivial_ball(mrl, bb)
            res["ball_wall_s"] += time.perf_counter() - t0
            try:
                gr = greedy_meet_in_the_middle(P, args.budget, ball)
                bf = bfs_meet_in_the_middle(P, args.budget, ball)
            finally:
                ball.close()
            res["greedy_device_s"] += gr[0][2]["seconds_device"]
            res["bfs_device_s"] += bf[0][2]["seconds_device"]
            g_ok = [k for k, r in enumerate(gr) if r[0]]
            b_ok = [k for k, r in enumerate(bf) if r[0]]
            for ok, out in ((g_ok, gr), (b_ok, bf)):
                res["all_paths_replay_to_length_2"] &= bool(replay_ok(P[ok], [out[k][1] for k in ok]))
            res["greedy_mitm"] += len(g_ok)
            res["greedy_via_ball"] += sum(gr[k][2]["goal"] is not None for k in g_ok)
            res["bfs_mitm"] += len(b_ok)
            res["bfs_via_ball"] += sum(bf[k][2]["goal"] is not None for k in b_ok)
            res["union"] += len(set(g_ok) | set(b_ok))
            plain_ok = {k for k, key in enumerate(answers[(0, mrl)]) if key[0]}
            res["plain_greedy_solved_lost"] += len(plain_ok - set(g_ok))
        mitm.append(res)
    result["meet_in_the_middle"] = mitm
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
