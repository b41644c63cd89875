"""Goal sets and goal-set search without a GPU: the CPU goal oracle is anchored to the pinned oracle,
every argument is validated on the host before any device work, and without a GPU the entry points
fail loudly instead of falling back to the CPU."""

import ctypes as C
import types

import numpy as np
import pytest

import goal_oracle as G
from oracle import oracle as O

AK2 = np.array([1, 1, -2, -2, -2, 0, 0, 1, 2, 1, -2, -1, -2, 0], np.int8)


def _no_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present: the loud-failure path is for CPU-only hosts")


def test_goal_oracle_without_goals_is_the_oracle(search_cases):
    """The anchor: no goal set and the length-2 rule on give oracle.bfs, visited array included
    (every reference fixture up to a budget of 20000)."""
    n = 0
    for c in search_cases["bfs"]:
        if c["budget"] > 20000:
            continue
        p, cyc = np.array(c["presentation"], np.int8), bool(c["cyclical"])
        ref = O.bfs(p, c["budget"], cyclically_reduce_after_moves=cyc, want_visited=True)
        got = G.bfs_goals(p, c["budget"], cyc, want_visited=True)
        assert (got[0], got[1]) == (ref[0], ref[1]), c
        for k in ("n_visited", "n_expanded", "n_moves", "frontier_left", "budget_hit", "minlen_log", "status"):
            assert got[2][k] == ref[2][k], (k, c)
        assert np.array_equal(got[2]["visited"], ref[2]["visited"])
        n += 1
    assert n == 19


def test_goal_oracle_stops_at_a_visited_state():
    ref = G.bfs_goals(AK2, 3000, want_visited=True)
    vis = ref[2]["visited"]
    for pos in (1, 17, len(vis) - 1):
        solved, path, info = G.bfs_goals(AK2, 3000, goals=G.goal_dict(vis[pos:pos + 1]), want_visited=True)
        assert solved and info["goal"] == 0
        assert path[-1][1] == int(np.count_nonzero(vis[pos]))
        assert np.array_equal(info["visited"], vis[: info["n_visited"]])
        state = AK2.copy()
        for a, length in path[1:]:
            state = O.acmove(a, state, 7, cyclical=False)[0]
            assert int(np.count_nonzero(state)) == length
        assert np.array_equal(state, vis[pos])
    root_hit = G.bfs_goals(AK2, 3000, goals=G.goal_dict(AK2[None, :]))
    assert root_hit[0] and root_hit[1] == [(-1, 11)] and root_hit[2]["n_expanded"] == 0


def test_goal_rows_are_validated_before_any_device_work():
    from ac_solver_b200 import GoalSet

    with pytest.raises(ValueError, match="must be"):
        GoalSet.from_rows(np.array([1, 0, 2, 0]))  # one row, not [n, 2*mrl]
    with pytest.raises(ValueError, match="alphabet"):
        GoalSet.from_rows(np.array([[1, 3, 2, 0]]))
    with pytest.raises(ValueError, match="row 1"):
        GoalSet.from_rows(np.array([[1, 0, 2, 0], [1, 0, 0, 0]]))  # an empty relator
    with pytest.raises(ValueError, match="row 0"):
        GoalSet.from_rows(np.array([[0, 1, 2, 0]]))  # padding on the left
    with pytest.raises(ValueError, match="freely reduced"):
        GoalSet.from_rows(np.array([[1, -1, 0, 2, 0, 0]]))
    with pytest.raises(ValueError, match="cyclically reduced"):
        GoalSet.from_rows(np.array([[1, 2, -1, 2, 0, 0]]), cyclically_reduce_after_moves=True)


def test_goal_options_are_validated_before_any_device_work():
    from ac_solver_b200 import bfs_batch, bfs_meet_in_the_middle

    rows = np.array([AK2, AK2])
    fake = dict(closed=False, max_relator_length=7, cyclical=False, device=0)
    with pytest.raises(ValueError, match="max_relator_length"):
        bfs_batch(rows, 10, goals=types.SimpleNamespace(**{**fake, "max_relator_length": 8}), device=0)
    with pytest.raises(ValueError, match="cyclically_reduce_after_moves"):
        bfs_batch(rows, 10, True, goals=types.SimpleNamespace(**fake), device=0)
    with pytest.raises(ValueError, match="device"):
        bfs_batch(rows, 10, goals=types.SimpleNamespace(**fake), device=1)
    with pytest.raises(ValueError, match="closed"):
        bfs_batch(rows, 10, goals=types.SimpleNamespace(**{**fake, "closed": True}), device=0)
    with pytest.raises(ValueError, match="cyclically_reduce_after_moves=False"):
        bfs_meet_in_the_middle(rows, 10, types.SimpleNamespace(**{**fake, "cyclical": True}))
    with pytest.raises(AssertionError, match="row 1"):
        bfs_batch(np.array([AK2, np.roll(AK2, 1)]), 10, goals=types.SimpleNamespace(**fake), device=0)


def test_c_abi_rejects_rows_before_looking_for_a_device():
    from ac_solver_b200 import _lib

    L = _lib.lib()
    h = C.c_void_p()
    bad = np.array([[1, -1, 0, 2, 0, 0]], np.int8)
    assert L.acs_goalset_from_rows(0, 3, 0, bad.ctypes.data, 1, C.byref(h)) == _lib.ACS_ERR_INVALID
    assert b"row 0" in L.acs_last_error() and not h
    assert L.acs_goalset_from_rows(0, 62, 0, None, 0, C.byref(h)) == _lib.ACS_ERR_UNSUPPORTED
    assert L.acs_bfs_batch_set_goals(None, None, 1) == _lib.ACS_ERR_INVALID
    assert L.acs_goalset_size(None, None, None, None) == _lib.ACS_ERR_INVALID
    L.acs_goalset_destroy(None)


def test_goal_search_without_gpu_raises():
    _no_gpu()
    from ac_solver_b200 import GoalSet, trivial_ball
    from ac_solver_b200._lib import AcsError

    with pytest.raises(AcsError):
        GoalSet.from_rows(np.array([[1, 0, 2, 0]]))
    with pytest.raises(AcsError):
        trivial_ball(7, 100)
