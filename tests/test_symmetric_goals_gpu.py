"""Symmetric goal sets on the GPU (csrc/goalset.cu, goalset.cuh; mbfs.cu, greedy.cu) and meet-in-the-middle
through symmetric balls (search/goals.py): a set of canonical forms matches every image of its states, exact
and orbit searches stop where the oracles with a symmetric goal test say, at the same entry and with the
element u that maps the end of the returned path onto the entry's state."""

import numpy as np
import pytest

import sym_oracle as S
from ac_solver_b200 import GoalSet, bfs_batch, bfs_meet_in_the_middle, greedy_meet_in_the_middle, trivial_ball
from ac_solver_b200.search.greedy import greedy_search_batch
from ac_solver_b200.synthetic import random_presentations
from conftest import ms_row
from goal_oracle import bfs_goals
from greedy_goal_oracle import greedy_goals
from oracle import oracle as O
from width_edges import roots

pytestmark = pytest.mark.gpu

KEYS = ("n_visited", "n_expanded", "n_moves", "frontier_left", "budget_hit", "status", "minlen_log")


def _end_state(row, path, cyc):
    s = np.ascontiguousarray(row, np.int8)
    for a, _ in path[1:]:
        s, _ = O.acmove(a, s, s.size // 2, cyclical=cyc)
    return s


def _check_hit(row, got, want, entry_state, cyc):
    assert got[0] == want[0] and got[1] == want[1], row
    for k in KEYS:
        assert got[2][k] == want[2][k], (k, row)
    assert got[2]["goal"] == want[2]["goal"], row
    if got[2]["goal"] is not None:
        c, u = S.canonical(_end_state(row, got[1], cyc))
        assert np.array_equal(c, entry_state(got[2]["goal"])), row
        assert got[2]["goal_element"] == u, row


@pytest.mark.parametrize("cyc", [False, True])
def test_all_images_hit_the_same_entry(cyc):
    rows = random_presentations(20, 12, seed=3)
    with GoalSet.from_rows(rows, cyc, symmetric=True) as gs:
        assert gs.symmetric and gs.n_entries == 20
        canon = [S.canonical(r)[0] for r in rows]
        for k in range(len(rows)):
            assert gs.frame(k) == S.INV[S.canonical(rows[k])[1]]  # end of the root path = the row itself
        q = np.concatenate([np.stack([S.act(g, r) for g in range(16)]) for r in rows])
        for res in (bfs_batch(q, 10, cyc, goals=gs), greedy_search_batch(q, 10, cyc, goals=gs)):
            for i, (ok, path, info) in enumerate(res):
                e = info["goal"]
                assert ok and path == [(-1, int(np.count_nonzero(q[i])))]
                assert e == min(j for j in range(len(rows)) if np.array_equal(canon[j], canon[i // 16]))
                assert np.array_equal(S.act(info["goal_element"], q[i]), canon[e])
                assert info["goal_element"] == S.canonical(q[i])[1]


@pytest.mark.parametrize("cyc", [False, True])
def test_searches_stop_at_symmetric_sets_like_the_oracle(cyc):
    rng = np.random.default_rng(7)
    for mrl in (4, 16, 30):
        R = roots(mrl)
        R = R[[all(np.count_nonzero(r[h * mrl:(h + 1) * mrl]) for h in (0, 1)) for r in R]]
        # goals: images of states deep in the roots' orbit searches, and an explored set from other rows
        deep = []
        for r in R[:3]:
            _, _, info = S.orbit_bfs(r, 400, cyc, want_visited=True)
            if info["status"] == 0 and len(info["visited"]) > 50:
                deep += [S.act(int(rng.integers(16)), v) for v in info["visited"][[40, -1]]]
        sets = []
        if deep:
            D = np.array(deep, np.int8)
            sets.append((GoalSet.from_rows(D, cyc, symmetric=True), [S.canonical(d)[0] for d in D]))
        E = random_presentations(2, mrl, seed=50 + mrl)
        ex = GoalSet.explore(E, 300, cyc, symmetric=True)
        ent = np.concatenate([S.orbit_bfs(e, 300, cyc, want_visited=True, stop_at_trivial=False)[2]["visited"]
                              for e in E])
        assert ex.n_entries == len(ent)
        for j in range(0, len(ent), 37):  # frames: the entry's path ends at frame(j).(stored state)
            root, path = ex.path(j)
            assert np.array_equal(_end_state(E[root], path, cyc), S.act(ex.frame(j), ent[j]))
        sets.append((ex, list(ent)))
        for gs, states in sets:
            d = {}
            for j, st in enumerate(states):
                d.setdefault(st.tobytes(), j)
            goals = S.SymGoals(d)
            B = np.array([(300, 2000)[k % 2] for k in range(len(R))], np.int64)
            for sym in (False, True):
                got = bfs_batch(R, B, cyc, goals=gs, symmetric=sym)
                for r, b, g in zip(R, B, got):
                    want = (S.orbit_bfs(r, int(b), cyc, goals=goals) if sym else
                            bfs_goals(r, int(b), cyc, goals=goals))
                    _check_hit(r, g, want, lambda e: states[e], cyc)
            got = greedy_search_batch(R, 2000, cyc, goals=gs)
            for r, g in zip(R, got):
                want = greedy_goals(r, 2000, cyc, goals=goals)
                assert g[0] == want[0] and g[1] == want[1] and g[2]["goal"] == want[2]["goal"], r
                if g[2]["goal"] is not None:
                    c, u = S.canonical(_end_state(r, g[1], cyc))
                    assert np.array_equal(c, states[g[2]["goal"]]) and g[2]["goal_element"] == u
            gs.close()


def _replays(row, path):
    return S.replay(row, path, False) == 2


def test_meet_in_the_middle_through_symmetric_balls(miller_schupp):
    ks = [k for k in range(0, 1190, 7) if int(miller_schupp["mrl"][k]) == int(miller_schupp["mrl"][0])]
    rows = np.array([ms_row(miller_schupp, k) for k in ks], np.int8)
    mrl = rows.shape[1] // 2
    plain = greedy_search_batch(rows, 20_000, False)
    with trivial_ball(mrl, 200_000, symmetric=True) as ball:
        assert ball.symmetric
        met = 0
        for sym in (False, True):
            for r, (ok, path, info) in zip(rows, bfs_meet_in_the_middle(rows, 20_000, ball, symmetric=sym)):
                if ok:
                    assert _replays(r, path)
                    met += info.get("goal") is not None
        out = greedy_meet_in_the_middle(rows, 20_000, ball)
        for r, p, (ok, path, info) in zip(rows, plain, out):
            if p[0]:
                assert ok
            if ok:
                assert _replays(r, path)
                met += info.get("goal") is not None
        assert met > 0
