"""Goal-set greedy search without a GPU: the CPU greedy goal oracle is anchored to the pinned oracle,
every goal option is validated on the host before any device work, and without a GPU the entry points
fail loudly instead of falling back to the CPU."""

import types

import numpy as np
import pytest

import goal_oracle as G
from greedy_goal_oracle import greedy_goals
from oracle import oracle as O

AK2 = np.array([1, 1, -2, -2, -2, 0, 0, 1, 2, 1, -2, -1, -2, 0], np.int8)
AK3 = np.array([1, 1, 1, -2, -2, -2, -2] + [0] * 17 + [1, 2, 1, -2, -1, -2] + [0] * 18, np.int8)
KEYS = ("n_visited", "n_expanded", "n_moves", "frontier_left", "budget_hit", "minlen_log", "status")


def _no_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present: the loud-failure path is for CPU-only hosts")


def _same_as_oracle(p, budget, cyc):
    ref = O.greedy_search(p, budget, cyclically_reduce_after_moves=cyc, want_visited=True)
    got = greedy_goals(p, budget, cyc, want_visited=True)
    assert (got[0], got[1]) == (ref[0], ref[1])
    for k in KEYS:
        assert got[2][k] == ref[2][k], k
    assert np.array_equal(got[2]["visited"], ref[2]["visited"])
    assert got[2]["goal"] is None


def test_greedy_goal_oracle_without_goals_is_the_oracle(search_cases):
    """The anchor: no goal set gives oracle.greedy_search -- path or failure path, counters, minimal-length
    log and the visited array in order -- on every greedy fixture."""
    for c in search_cases["greedy"]:
        _same_as_oracle(np.array(c["presentation"], np.int8), c["budget"], bool(c["cyclical"]))
    assert len(search_cases["greedy"]) == 11


@pytest.mark.parametrize("budget", [50, 777, 20000])
def test_greedy_goal_oracle_without_goals_on_ak3(budget):
    _same_as_oracle(AK3, budget, False)


def _replay(p, path, cyc):
    state = p.copy()
    assert int(np.count_nonzero(state)) == path[0][1]
    for a, length in path[1:]:
        state = O.acmove(a, state, p.size // 2, cyclical=cyc)[0]
        assert int(np.count_nonzero(state)) == length
    return state


@pytest.mark.parametrize("cyc", [False, True])
def test_greedy_goal_oracle_stops_at_a_visited_state(cyc):
    plain = greedy_goals(AK2, 3000, cyc, want_visited=True)
    vis = plain[2]["visited"]
    for pos in (1, 17, 400, len(vis) - 1):
        solved, path, info = greedy_goals(AK2, 3000, cyc, goals=G.goal_dict(vis[pos:pos + 1]), want_visited=True)
        assert solved and info["goal"] == 0 and not info["budget_hit"]
        assert path[-1][1] == int(np.count_nonzero(vis[pos]))
        assert np.array_equal(info["visited"], vis[: info["n_visited"]])
        assert info["n_visited"] <= pos  # the goal child itself is not inserted
        assert info["minlen_log"] == plain[2]["minlen_log"][: len(info["minlen_log"])]
        assert np.array_equal(_replay(AK2, path, cyc), vis[pos])


def test_greedy_goal_oracle_root_hit():
    solved, path, info = greedy_goals(AK2, 3000, goals=G.goal_dict(AK2[None, :]), want_visited=True)
    assert solved and path == [(-1, 11)] and info["goal"] == 0
    assert (info["n_visited"], info["n_expanded"], info["n_moves"], info["frontier_left"]) == (1, 0, 0, 1)
    assert info["minlen_log"] == [] and not info["budget_hit"]


def test_greedy_goal_oracle_solve_wins_on_the_same_child():
    """A goal set holding every state of total length 2: the search ends exactly where the plain one solves,
    as a solve, not a goal."""
    from ac_solver_b200.envs.utils import generate_trivial_states

    plain = greedy_goals(AK2, 5000)
    got = greedy_goals(AK2, 5000, goals=G.goal_dict(generate_trivial_states(7)))
    assert plain[0] and (got[0], got[1]) == (plain[0], plain[1]) and got[2]["goal"] is None


def test_greedy_goal_options_are_validated_before_any_device_work():
    from ac_solver_b200 import greedy_meet_in_the_middle, greedy_search_batch

    rows = np.array([AK2, AK2])
    fake = dict(closed=False, max_relator_length=7, cyclical=False, device=0)
    with pytest.raises(ValueError, match="max_relator_length"):
        greedy_search_batch(rows, 10, goals=types.SimpleNamespace(**{**fake, "max_relator_length": 8}), device=0)
    with pytest.raises(ValueError, match="cyclically_reduce_after_moves"):
        greedy_search_batch(rows, 10, True, goals=types.SimpleNamespace(**fake), device=0)
    with pytest.raises(ValueError, match="device"):
        greedy_search_batch(rows, 10, goals=types.SimpleNamespace(**fake), device=1)
    with pytest.raises(ValueError, match="closed"):
        greedy_search_batch(rows, 10, goals=types.SimpleNamespace(**{**fake, "closed": True}), device=0)
    with pytest.raises(ValueError, match="cyclically_reduce_after_moves=False"):
        greedy_meet_in_the_middle(rows, 10, types.SimpleNamespace(**{**fake, "cyclical": True}))


def test_c_abi_greedy_goal_calls_reject_null_engines():
    from ac_solver_b200 import _lib

    L = _lib.lib()
    assert L.acs_greedy_set_goals(None, None) == _lib.ACS_ERR_INVALID
    assert L.acs_greedy_goal_hits(None, None) == _lib.ACS_ERR_INVALID


def test_greedy_goal_search_without_gpu_raises():
    _no_gpu()
    from ac_solver_b200 import greedy_meet_in_the_middle, greedy_search_batch
    from ac_solver_b200._lib import AcsError

    with pytest.raises(AcsError):
        greedy_search_batch(AK2[None, :], 100, goals=None)
    ball = types.SimpleNamespace(closed=False, max_relator_length=7, cyclical=False, device=0, handle=None)
    with pytest.raises(AcsError):
        greedy_meet_in_the_middle(AK2[None, :], 100, ball)
