"""Goal-set greedy search on the GPU (the GOAL instantiations of csrc/greedy.cu and csrc/greedy_bucket.cuh):
checked against plain greedy_search_batch where the answer is known, and against the CPU greedy goal
oracle (tests/greedy_goal_oracle.py) everywhere else.  Every check runs under the bucket kernel and under the
one-warp heap kernel (ACS_GREEDY_KERNEL=heap)."""

import numpy as np
import pytest

import goal_oracle as G
from greedy_goal_oracle import greedy_goals
from conftest import ms_row
from oracle import oracle as O

pytestmark = pytest.mark.gpu

AK2 = np.array([1, 1, -2, -2, -2, 0, 0, 1, 2, 1, -2, -1, -2, 0], np.int8)
KEYS = ("n_visited", "n_expanded", "n_moves", "frontier_left", "budget_hit", "status", "minlen_log")


@pytest.fixture(params=["bucket", "heap"])
def kernel(request, monkeypatch):
    """The engine reads ACS_GREEDY_KERNEL when it is created."""
    if request.param == "heap":
        monkeypatch.setenv("ACS_GREEDY_KERNEL", "heap")
    else:
        monkeypatch.delenv("ACS_GREEDY_KERNEL", raising=False)
    return request.param


def _same(a, b, visited=True):
    assert (a[0], a[1]) == (b[0], b[1])
    for k in KEYS:
        assert a[2][k] == b[2][k], k
    if visited:
        assert np.array_equal(a[2]["visited"], b[2]["visited"])


def _replay(state, path, cyc):
    state = np.asarray(state, np.int8)
    mrl = state.size // 2
    assert int(np.count_nonzero(state)) == path[0][1]
    for a, length in path[1:]:
        state = np.asarray(O.acmove(int(a), state, mrl, cyclical=cyc)[0], np.int8)
        assert int(np.count_nonzero(state)) == length
    return state


def _ms_groups(ms, step=1):
    by_width = {}
    for k in range(0, 1190, step):
        by_width.setdefault(len(ms_row(ms, k)), []).append(k)
    return by_width


def test_empty_goal_set_changes_nothing(search_cases, kernel):
    from ac_solver_b200 import GoalSet, greedy_search_batch

    groups = {}
    for c in search_cases["greedy"]:
        groups.setdefault((len(c["presentation"]), bool(c["cyclical"]), c["budget"]), []).append(c)
    for (w, cyc, budget), cases in groups.items():
        rows = np.array([c["presentation"] for c in cases], np.int8)
        with GoalSet.from_rows(np.zeros((0, w), np.int8), cyc) as g:
            got = greedy_search_batch(rows, budget, cyc, want_visited=True, goals=g)
        for a, b in zip(got, greedy_search_batch(rows, budget, cyc, want_visited=True)):
            _same(a, b)
            assert a[2]["goal"] is None and "goal" not in b[2]


def test_trivial_goals_equal_plain_search(miller_schupp, kernel):
    """The 8 trivial states as goals: identical answers, and no row stops at a goal -- every state of total
    length 2 is one of them, and the solve wins on the same child."""
    from ac_solver_b200 import GoalSet, greedy_search_batch
    from ac_solver_b200.envs.utils import generate_trivial_states

    n_solved = 0
    for mrl2, ks in _ms_groups(miller_schupp).items():
        rows = np.array([ms_row(miller_schupp, k) for k in ks], np.int8)
        with GoalSet.from_rows(generate_trivial_states(mrl2 // 2)) as g:
            got = greedy_search_batch(rows, 10_000, goals=g)
        for a, b in zip(got, greedy_search_batch(rows, 10_000)):
            _same(a, b, visited=False)
            assert a[2]["goal"] is None
            n_solved += a[0]
    assert n_solved > 0


def _one_goal_rows(ms):
    return [AK2] + [ms_row(ms, k) for k in (0, 5, 40, 200, 700)]


@pytest.mark.parametrize("cyc", [False, True])
def test_one_goal_per_row_matches_the_goal_oracle(miller_schupp, cyc, kernel):
    """Goal = a state of the row's own plain visited array at several positions; every row of the batch sees
    the goals of the others too.  Hit, path, counters, minimal-length log and visited array equal the goal
    oracle's; the visited array is a prefix of the plain run's; the path replays to the goal state."""
    from ac_solver_b200 import GoalSet, greedy_search_batch

    budget = 3000
    for mrl2 in sorted({len(r) for r in _one_goal_rows(miller_schupp)}):
        rows = np.array([r for r in _one_goal_rows(miller_schupp) if len(r) == mrl2], np.int8)
        plain = greedy_search_batch(rows, budget, cyc, want_visited=True)
        for frac in (0.0, 0.3, 0.7, 1.0):
            goals = []
            for p in plain:
                vis = p[2]["visited"]
                goals.append(vis[min(len(vis) - 1, max(1, int(frac * (len(vis) - 1))))])
            goals = np.array(goals, np.int8)
            with GoalSet.from_rows(goals, cyc) as g:
                got = greedy_search_batch(rows, budget, cyc, want_visited=True, goals=g)
            for r, p, a in zip(rows, plain, got):
                ref = greedy_goals(r, budget, cyc, goals=G.goal_dict(goals), want_visited=True)
                _same(a, ref)
                assert a[2]["goal"] == ref[2]["goal"]
                assert np.array_equal(a[2]["visited"], p[2]["visited"][: a[2]["n_visited"]])
                if a[0]:
                    end = _replay(r, a[1], cyc)
                    if a[2]["goal"] is not None:
                        assert np.array_equal(end, goals[a[2]["goal"]])


def test_roots_in_the_goal_set_hit_at_depth_zero(miller_schupp, kernel):
    from ac_solver_b200 import GoalSet, greedy_search_batch

    rows = np.array([ms_row(miller_schupp, k) for k in range(0, 170, 7)], np.int8)
    goals = rows[::-1].copy()
    with GoalSet.from_rows(goals) as g:
        got = greedy_search_batch(rows, 1000, want_visited=True, goals=g)
    for j, (r, a) in enumerate(zip(rows, got)):
        assert a[0] and a[1] == [(-1, int(np.count_nonzero(r)))]
        assert a[2]["goal"] == len(rows) - 1 - j
        assert (a[2]["n_visited"], a[2]["n_expanded"], a[2]["n_moves"], a[2]["frontier_left"]) == (1, 0, 0, 1)
        _same(a, greedy_goals(r, 1000, goals=G.goal_dict(goals), want_visited=True))


def test_explored_goal_set_hits_the_smallest_entry(kernel):
    """A GoalSet.explore set whose balls share states: a greedy search rooted at a state stops at depth 0 on
    the smallest entry holding it."""
    from ac_solver_b200 import GoalSet, bfs_batch, greedy_search_batch
    from ac_solver_b200.envs.utils import generate_trivial_states

    mrl, budget = 7, 2000
    roots = np.concatenate([generate_trivial_states(mrl).astype(np.int8), AK2[None, :], AK2[None, :]])
    plain = bfs_batch(roots, budget, want_visited=True, stop_at_trivial=False)
    vis = np.concatenate([p[2]["visited"] for p in plain])
    first = G.goal_dict(vis)
    assert sum(1 for e in range(len(vis)) if first[vis[e].tobytes()] != e) > 0
    rng = np.random.default_rng(5)
    probe = vis[rng.choice(len(vis), 200, replace=False)]
    with GoalSet.explore(roots, budget) as g:
        hits = greedy_search_batch(probe, 10, goals=g)
    for p, h in zip(probe, hits):
        assert h[0] and h[2]["goal"] == first[p.tobytes()]


def test_path_overflow_rerun_keeps_goal_hits(miller_schupp, kernel):
    """Goals deep in the search (the node each plain search expanded last, from its path replayed without
    the final pair): the goal paths are longer than a path_cap of 4, so the search is re-run with room,
    and the re-run keeps the goal set."""
    from ac_solver_b200 import GoalSet, greedy_search_batch

    rows = np.array([ms_row(miller_schupp, k) for k in (5, 40, 200)], np.int8)
    plain = greedy_search_batch(rows, 3000)
    goals = np.array([_replay(r, p[1][:-1], False) for r, p in zip(rows, plain)], np.int8)
    with GoalSet.from_rows(goals) as g:
        ref = greedy_search_batch(rows, 3000, goals=g)
        small = greedy_search_batch(rows, 3000, goals=g, path_cap=4)
    assert max(len(r[1]) for r in ref) > 4
    for r, a, b in zip(rows, small, ref):
        _same(a, b, visited=False)
        assert a[2]["goal"] == b[2]["goal"] is not None
        _same(a, greedy_goals(r, 3000, goals=G.goal_dict(goals)), visited=False)


def test_greedy_meet_in_the_middle_on_miller_schupp_rows(miller_schupp, kernel):
    """Stitched paths replay to total length 2, every row plain greedy solves is trivialized, and at least
    one row meets the ball."""
    from ac_solver_b200 import greedy_meet_in_the_middle, greedy_search_batch, trivial_ball

    budget, ball_budget = 5000, 20_000
    n_plain = n_mitm = n_met = 0
    for mrl2, ks in _ms_groups(miller_schupp, 3).items():
        rows = np.array([ms_row(miller_schupp, k) for k in ks], np.int8)
        plain = greedy_search_batch(rows, budget)
        with trivial_ball(mrl2 // 2, ball_budget) as ball:
            got = greedy_meet_in_the_middle(rows, budget, ball)
        for r, p, (ok, path, info) in zip(rows, plain, got):
            if p[0]:
                assert ok
            if ok:
                assert path[-1][1] == 2
                end = _replay(r, path, False)
                assert int(np.count_nonzero(end)) == 2
                n_met += info["goal"] is not None
            else:
                assert (ok, path) == (p[0], p[1])  # greedy's failure path
            n_plain += p[0]
            n_mitm += ok
    assert n_mitm >= n_plain and n_met > 0
