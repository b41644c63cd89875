"""Batched beam search on the GPU (csrc/beam.cu) against its CPU statement (tests/beam_oracle.py) in
everything it reports: solved flag, path, counters, minimal-length log, goal entry and the visited rows in
order."""

import numpy as np
import pytest

import beam_oracle as B
import goal_oracle as G
import sym_oracle as SO
import width_edges as WE
from conftest import ms_row
from oracle import oracle as O

pytestmark = pytest.mark.gpu

AK2 = np.array([1, 1, -2, -2, -2, 0, 0, 1, 2, 1, -2, -1, -2, 0], np.int8)
AK3 = np.array([1, 1, 1, -2, -2, -2, -2] + [0] * 17 + [1, 2, 1, -2, -1, -2] + [0] * 18, np.int8)
KEYS = ("n_visited", "n_expanded", "n_moves", "frontier_left", "budget_hit", "levels", "status", "minlen_log")


def _same(dev, orc, goals=False):
    assert (dev[0], dev[1]) == (orc[0], orc[1])
    for k in KEYS:
        assert dev[2][k] == orc[2][k], (k, dev[2][k], orc[2][k])
    if goals:
        assert dev[2]["goal"] == orc[2]["goal"]
    if orc[2]["status"] == 0:
        assert np.array_equal(dev[2]["visited"], orc[2]["visited"])


def _check(rows, width, budget, depth=None, cyc=False, goals=None, orc_goals=None):
    from ac_solver_b200 import beam_search_batch

    rows = np.ascontiguousarray(rows, dtype=np.int8)
    res = beam_search_batch(rows, width, budget, depth, cyc, want_visited=True, goals=goals)
    assert len(res) == len(rows)
    budgets = np.broadcast_to(np.asarray(budget), (len(rows),))
    for k, row in enumerate(rows):
        orc = B.beam_search(row, width, int(budgets[k]), depth, cyc, goals=orc_goals, want_visited=True)
        _same(res[k], orc, goals is not None)
    return res


def _one_mrl(ms, n, step=7):
    """n Miller-Schupp rows of one max_relator_length (that of row 0), every step-th of them."""
    m = ms_row(ms, 0).size
    rows = [ms_row(ms, k) for k in range(1190) if ms_row(ms, k).size == m]
    return np.array(rows[::step][:n])


def _ms(ms, mrls, per=2, start=0):
    rows = {}
    for k in range(start, 1190, 7):
        row = ms_row(ms, k)
        m = row.size // 2
        if m in mrls and len(rows.setdefault(m, [])) < per:
            rows[m].append(row)
    return rows


@pytest.mark.parametrize("cyc", [False, True])
@pytest.mark.parametrize("width", [1, 2, 7, 64, 1000])
def test_ak_rows_match_the_oracle(width, cyc):
    for row in (AK2, AK3):
        _check(row[None, :], width, 3000, cyc=cyc)


@pytest.mark.parametrize("cyc", [False, True])
@pytest.mark.parametrize("width", [1, 7, 64, 1000])
def test_miller_schupp_rows_of_both_key_widths(miller_schupp, width, cyc):
    """mrl 18-28 (one key word per relator) and 32-36 (two), one engine per mrl; budgets that cut a level in
    the middle (7 * 64 + 1, and 1000 + 1 below the second level of width 1000)."""
    for m, rows in _ms(miller_schupp, (18, 24, 28, 32, 36)).items():
        _check(np.array(rows), width, [449, 1001] * (len(rows) // 2) + [449] * (len(rows) % 2), cyc=cyc)


@pytest.mark.parametrize("depth", [1, 3, 10])
def test_depth_limits(miller_schupp, depth):
    rows = np.array(_ms(miller_schupp, (20,), per=3)[20])
    _check(rows, 7, 5000, depth=depth)
    _check(AK2[None, :], 64, 100_000, depth=depth, cyc=True)


def test_budget_one_and_budget_at_the_root_level():
    """Budget 1: the root level is expanded, nothing is kept.  Budget 2 and width 5: one node of level 1."""
    for budget in (1, 2, 13):
        _check(np.array([AK2, AK2]), 5, budget)


def test_batch_equals_one_run_per_row(miller_schupp):
    from ac_solver_b200 import beam_search, beam_search_batch

    rows = _one_mrl(miller_schupp, 15, 23)
    budgets = np.arange(len(rows)) * 97 + 200
    batch = beam_search_batch(rows, 16, budgets, want_visited=True)
    for k, row in enumerate(rows):
        one = beam_search(row, 16, int(budgets[k]), want_visited=True)
        assert (one[0], one[1]) == (batch[k][0], batch[k][1])
        for key in KEYS:
            assert one[2][key] == batch[k][2][key]
        assert np.array_equal(one[2]["visited"], batch[k][2]["visited"])


def test_split_batches_equal_one_engine(miller_schupp):
    from ac_solver_b200 import beam_search_batch

    rows = _one_mrl(miller_schupp, 11, 31)
    whole = beam_search_batch(rows, 8, 500)
    parts = beam_search_batch(rows, 8, 500, max_bytes=1)  # one row per engine
    for a, b in zip(whole, parts):
        assert (a[0], a[1]) == (b[0], b[1]) and all(a[2][k] == b[2][k] for k in KEYS)


@pytest.mark.parametrize("mrl", [1, 2, 3, 4, 15, 16, 17, 28, 29, 30, 31, 32, 33, 60, 61])
def test_packed_key_edges(mrl):
    """The rows of tests/width_edges.py at the edges of the packed key layout, including rows that raise
    and rows that solve at the first level."""
    rows = WE.roots(mrl)
    for cyc in (False, True):
        _check(rows, 7, 300, cyc=cyc)


def test_a_row_that_raises_ends_only_its_search():
    rows = np.array(WE.HAND_PICKED[2], np.int8)
    res = _check(rows, 4, 100)
    assert res[0][2]["status"] != 0 or res[1][2]["status"] != 0
    rows = np.concatenate([WE.roots(4), WE.roots(4)])
    _check(rows, 3, 200, cyc=True)


def _goal_rows(row, cyc, width=7, budget=400):
    """States a beam of another width reaches: likely goals of the searches under test."""
    V = B.beam_search(row, width, budget, cyclically_reduce_after_moves=cyc, want_visited=True)[2]["visited"]
    return V[-6:]


@pytest.mark.parametrize("cyc", [False, True])
def test_exact_goal_sets(miller_schupp, cyc):
    from ac_solver_b200 import GoalSet

    row = ms_row(miller_schupp, 14)
    goal_rows = np.concatenate([_goal_rows(row, cyc), _goal_rows(row, cyc, 3, 300)])
    hits = 0
    with GoalSet.from_rows(goal_rows, cyc) as gs:
        for width in (2, 7, 16, 64):
            res = _check(row[None, :], width, 3000, cyc=cyc, goals=gs, orc_goals=G.goal_dict(goal_rows))
            hits += res[0][2]["goal"] is not None
    assert hits > 0


def test_root_in_goal_set_and_solve_beats_goal():
    from ac_solver_b200 import GoalSet, beam_search_batch

    rows = np.array([[1, 2, 0, 2, 0, 0], [2, 1, 1, 1, 0, 0]], np.int8)  # xy, y (move 1 gives x, y); yx, xx
    child, _ = O.acmove(1, rows[0], 3, cyclical=False)
    goal_rows = np.array([child, rows[1]], np.int8)  # a trivial child of row 0, and row 1 itself
    with GoalSet.from_rows(goal_rows) as gs:
        res = _check(rows, 4, 100, goals=gs, orc_goals=G.goal_dict(goal_rows))
        assert res[0][0] and res[0][2]["goal"] is None and res[0][1][-1][1] == 2
        assert res[1][0] and res[1][1] == [(-1, 4)] and res[1][2]["goal"] == 1
        full = beam_search_batch(rows, 4, 100, goals=gs)
        assert full[1][2]["goal_element"] == 0


@pytest.mark.parametrize("cyc", [False, True])
def test_symmetric_goal_sets(miller_schupp, cyc):
    from ac_solver_b200 import GoalSet

    rows = _one_mrl(miller_schupp, 3)
    goal_rows = np.concatenate([_goal_rows(r, cyc) for r in rows])
    images = np.array([SO.act((3 + i) % 16, r) for i, r in enumerate(goal_rows)], np.int8)
    entries = {}
    for i, r in enumerate(images):
        entries.setdefault(SO.canonical(r)[0].tobytes(), i)
    with GoalSet.from_rows(images, cyc, symmetric=True) as gs:
        res = _check(rows, 16, 2000, cyc=cyc, goals=gs, orc_goals=SO.SymGoals(entries))
    assert any(info["goal"] is not None for _, _, info in res)
    for solved, path, info in res:
        if info["goal"] is not None:
            assert 0 <= info["goal_element"] < 16


@pytest.mark.parametrize("symmetric", [False, True])
def test_meet_in_the_middle_paths_replay_to_trivial(miller_schupp, symmetric):
    from ac_solver_b200 import beam_meet_in_the_middle, trivial_ball

    rows = [ms_row(miller_schupp, k) for k in range(0, 1190, 13)]
    by = {}
    for r in rows:
        by.setdefault(r.size // 2, []).append(r)
    n_ball = 0
    for m, rs in by.items():
        ball = trivial_ball(m, 20_000, symmetric=symmetric)
        try:
            res = beam_meet_in_the_middle(np.array(rs), 64, 20_000, ball)
            for r, (triv, path, info) in zip(rs, res):
                if triv:
                    assert SO.replay(r, path, False) == 2
                    n_ball += info.get("goal") is not None
        finally:
            ball.close()
    assert n_ball > 0


def test_long_paths_are_fetched_again(miller_schupp):
    """A path longer than the first buffer is fetched through acs_beam_paths without searching again."""
    from ac_solver_b200.search.beam import beam_search_batch

    rows = _one_mrl(miller_schupp, 20, 17)
    orc = [B.beam_search(r, 4, 3000) for r in rows]
    assert any(o[0] and len(o[1]) > 3 for o in orc)
    short = beam_search_batch(rows, 4, 3000, _path_cap=3)
    full = beam_search_batch(rows, 4, 3000)
    for s, o in enumerate(orc):
        assert short[s][1] == full[s][1] == o[1]
