"""Goal-set search on the GPU (csrc/goalset.cu, the goal test and exploration mode of csrc/mbfs.cu):
checked against plain bfs_batch where the answer is known, and against the CPU goal oracle
(tests/goal_oracle.py) everywhere else."""

import numpy as np
import pytest

import goal_oracle as G
from conftest import ms_row
from oracle import oracle as O

pytestmark = pytest.mark.gpu

AK2 = np.array([1, 1, -2, -2, -2, 0, 0, 1, 2, 1, -2, -1, -2, 0], np.int8)
KEYS = ("n_visited", "n_expanded", "n_moves", "frontier_left", "budget_hit", "status", "minlen_log")


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


def test_empty_goal_set_changes_nothing(search_cases):
    """The reference fixtures as batches with an empty goal set equal plain bfs_batch."""
    from ac_solver_b200 import GoalSet, bfs_batch

    groups = {}
    for c in search_cases["bfs"]:
        groups.setdefault((len(c["presentation"]), bool(c["cyclical"])), []).append(c)
    for (w, cyc), cases in groups.items():
        rows, budgets = np.array([c["presentation"] for c in cases]), [c["budget"] for c in cases]
        with GoalSet.from_rows(np.zeros((0, w), np.int8), cyc) as g:
            assert (g.n_entries, g.n_states) == (0, 0)
            got = bfs_batch(rows, budgets, cyc, want_visited=True, goals=g)
        for a, b in zip(got, bfs_batch(rows, budgets, cyc, want_visited=True)):
            _same(a, b)
            assert a[2]["goal"] is None


@pytest.mark.parametrize("cyc", [False, True])
def test_trivial_goals_in_exploration_mode_equal_plain_search(miller_schupp, cyc):
    """Every Miller-Schupp row: with the 8 trivial states as goals and the length-2 rule off, a search
    stops exactly where the plain search solves (the groups are trivial, so every state of total
    length 2 is one of the 8)."""
    from ac_solver_b200 import GoalSet, bfs_batch
    from ac_solver_b200.envs.utils import generate_trivial_states

    n_solved = 0
    for mrl2, ks in _ms_groups(miller_schupp).items():
        rows = np.array([ms_row(miller_schupp, k) for k in ks], np.int8)
        with GoalSet.from_rows(generate_trivial_states(mrl2 // 2), cyc) as g:
            got = bfs_batch(rows, 10_000, cyc, want_visited=True, goals=g, stop_at_trivial=False)
        for a, b in zip(got, bfs_batch(rows, 10_000, cyc, want_visited=True)):
            _same(a, b)
            assert (a[2]["goal"] is not None) == a[0]
            n_solved += a[0]
    assert n_solved > 0 or not cyc


def _one_goal_rows(ms):
    return [AK2] + [ms_row(ms, k) for k in (0, 5, 40, 200)]


@pytest.mark.parametrize("cyc", [False, True])
def test_one_goal_per_row_matches_the_goal_oracle(miller_schupp, cyc):
    """Goal = a state of the row's own visited array at several positions; every row of the batch sees
    the goals of the others too.  Hit, path, counters and visited array equal the goal oracle's, and the
    visited array is a prefix of the plain run's."""
    from ac_solver_b200 import GoalSet, bfs_batch
    from ac_solver_b200.search.breadth_first import bfs_device

    budget = 3000
    for mrl2 in sorted({len(r) for r in _one_goal_rows(miller_schupp)}):
        rows = np.array([r for r in _one_goal_rows(miller_schupp) if len(r) == mrl2], np.int8)
        plain = [bfs_device(r, budget, cyc, want_visited=True) for r in rows]
        for frac in (0.0, 0.3, 0.7, 1.0):
            goals = []
            for r, p in zip(rows, plain):
                vis = p[2]["visited"]
                goals.append(vis[min(len(vis) - 1, max(1, int(frac * (len(vis) - 1))))])
            goals = np.array(goals, np.int8)
            with GoalSet.from_rows(goals, cyc) as g:
                got = bfs_batch(rows, budget, cyc, want_visited=True, goals=g)
            for r, p, a in zip(rows, plain, got):
                ref = G.bfs_goals(r, budget, cyc, goals=G.goal_dict(goals), want_visited=True)
                _same(a, ref)
                assert a[2]["goal"] == ref[2]["goal"]
                assert np.array_equal(a[2]["visited"], p[2]["visited"][: a[2]["n_visited"]])
                if a[0]:
                    end = _replay(r, a[1], cyc)
                    if a[2]["goal"] is not None:
                        assert np.array_equal(end, goals[a[2]["goal"]])


def test_roots_in_the_goal_set_hit_at_depth_zero(miller_schupp):
    from ac_solver_b200 import GoalSet, bfs_batch

    rows = np.array([ms_row(miller_schupp, k) for k in range(0, 170, 7)], np.int8)
    goals = rows[::-1].copy()
    with GoalSet.from_rows(goals) as g:
        got = bfs_batch(rows, 1000, want_visited=True, goals=g)
    for j, (r, a) in enumerate(zip(rows, got)):
        assert a[0] and a[1] == [(-1, int(np.count_nonzero(r)))]
        assert a[2]["goal"] == len(rows) - 1 - j
        assert (a[2]["n_visited"], a[2]["n_expanded"], a[2]["n_moves"]) == (1, 0, 0)
        _same(a, G.bfs_goals(r, 1000, goals=G.goal_dict(goals), want_visited=True))


@pytest.mark.parametrize("cyc", [False, True])
def test_exploration_from_the_trivial_roots(cyc):
    """Exploration mode equals the goal oracle with the length-2 rule off, and no row raises."""
    from ac_solver_b200 import bfs_batch
    from ac_solver_b200.envs.utils import generate_trivial_states

    for mrl, budget in ((5, 4000), (11, 3000), (30, 1500)):
        roots = generate_trivial_states(mrl).astype(np.int8)
        got = bfs_batch(roots, budget, cyc, want_visited=True, stop_at_trivial=False)
        for r, a in zip(roots, got):
            assert a[2]["status"] == 0 and not a[0]
            _same(a, G.bfs_goals(r, budget, cyc, stop_at_trivial=False, want_visited=True))


def test_goal_set_from_a_run():
    """Entries are the visited states of every search in (search, FIFO) order; n_states counts distinct
    states; the smallest entry index represents a shared state; paths replay from the entry's root."""
    from ac_solver_b200 import GoalSet, bfs_batch
    from ac_solver_b200.envs.utils import generate_trivial_states

    mrl, budget = 7, 2000
    roots = np.concatenate([generate_trivial_states(mrl).astype(np.int8), AK2[None, :], AK2[None, :]])
    plain = bfs_batch(roots, budget, want_visited=True, stop_at_trivial=False)
    vis = np.concatenate([p[2]["visited"] for p in plain])
    root_of = np.concatenate([np.full(len(p[2]["visited"]), s) for s, p in enumerate(plain)])
    first = G.goal_dict(vis)
    with GoalSet.explore(roots, budget) as g:
        assert g.n_entries == len(vis) and g.n_states == len(first)
        assert [r[2]["n_visited"] for r in g.results] == [p[2]["n_visited"] for p in plain]
        rng = np.random.default_rng(3)
        for e in rng.choice(len(vis), 40, replace=False).tolist() + [0, len(vis) - 1]:
            root, path = g.path(e)
            assert root == root_of[e]
            assert np.array_equal(_replay(roots[root], path, False), vis[e])
        # the smallest index wins: a search rooted at a state stops at depth 0 on its first entry
        probe = vis[rng.choice(len(vis), 200, replace=False)]
        hits = bfs_batch(probe, 10, goals=g)
        for p, h in zip(probe, hits):
            assert h[2]["goal"] == first[p.tobytes()]
        shared = sum(1 for e in range(len(vis)) if first[vis[e].tobytes()] != e)
        assert shared > 0  # the AK2 copies and the trivial balls share states


def test_meet_in_the_middle_on_miller_schupp_rows(miller_schupp):
    """Stitched paths replay to total length 2, and every row plain bfs_batch solves is trivialized."""
    from ac_solver_b200 import bfs_batch, bfs_meet_in_the_middle, trivial_ball

    budget, ball_budget = 5000, 20_000
    n_plain = n_mitm = n_met = 0
    for mrl2, ks in _ms_groups(miller_schupp, 3).items():
        rows = np.array([ms_row(miller_schupp, k) for k in ks], np.int8)
        plain = bfs_batch(rows, budget)
        with trivial_ball(mrl2 // 2, ball_budget) as ball:
            assert all(r[2]["status"] == 0 and not r[0] for r in ball.results)
            got = bfs_meet_in_the_middle(rows, budget, ball)
        for r, p, (ok, path, info) in zip(rows, plain, got):
            if p[0]:
                assert ok
            if ok:
                assert path[-1][1] == 2
                end = _replay(r, path, False)
                assert int(np.count_nonzero(end)) == 2
                n_met += info["goal"] is not None
            n_plain += p[0]
            n_mitm += ok
    assert n_mitm >= n_plain and n_met > 0


@pytest.mark.parametrize("chunk_parents", [1, 7, 64])
def test_goal_results_do_not_depend_on_chunks_or_splits(miller_schupp, chunk_parents):
    from ac_solver_b200 import bfs_batch, trivial_ball

    rows = np.array([ms_row(miller_schupp, k) for k in range(0, 170, 9)], np.int8)
    mrl = rows.shape[1] // 2
    with trivial_ball(mrl, 3000, chunk_parents=chunk_parents) as ball, trivial_ball(mrl, 3000) as ref_ball:
        assert ball.n_entries == ref_ball.n_entries and ball.n_states == ref_ball.n_states
        assert [ball.path(e) for e in (1, 100, 5000)] == [ref_ball.path(e) for e in (1, 100, 5000)]
        ref = bfs_batch(rows, 3000, want_visited=True, goals=ref_ball)
        got = bfs_batch(rows, 3000, want_visited=True, goals=ref_ball, chunk_parents=chunk_parents)
        split = bfs_batch(rows, 3000, want_visited=True, goals=ref_ball, max_bytes=1)  # one row per engine
        for a, b, c in zip(got, ref, split):
            _same(a, b)
            _same(c, b)
            assert a[2]["goal"] == b[2]["goal"] == c[2]["goal"]
        assert any(b[2]["goal"] is not None for b in ref)
