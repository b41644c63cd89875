"""Orbit search and canonical forms on the GPU (csrc/ac_sym.cuh, csrc/sym.cu, csrc/mbfs.cu): the device
canonical form equals tests/sym_oracle.py's, and ``bfs_batch(symmetric=True)`` equals the orbit-BFS oracle
in everything it reports -- visited array in insertion order, counters, budget cut, status and the path
in moves of the input row -- which replays to a trivial presentation and is as short as exact search's."""

import numpy as np
import pytest

import sym_oracle as S
from ac_solver_b200 import GoalSet, _lib, bfs_batch, bfs_groups, canonical_form
from ac_solver_b200.synthetic import random_presentations
from conftest import ms_row
from width_edges import WIDTHS, roots

pytestmark = pytest.mark.gpu

KEYS = ("n_visited", "n_expanded", "n_moves", "frontier_left", "budget_hit", "status", "minlen_log")


def test_canonical_form_matches_oracle():
    rng = np.random.default_rng(1)
    for mrl in WIDTHS:
        R = np.concatenate([roots(mrl), random_presentations(40, mrl, seed=mrl)])
        el = rng.integers(0, 16, size=len(R))
        R = np.concatenate([R, np.stack([S.act(int(g), r) for g, r in zip(el, R)])])  # and images of them
        c, g = canonical_form(R)
        want_c, want_g = S.canonical_batch(R)
        assert np.array_equal(c, want_c), mrl
        assert np.array_equal(g, want_g), mrl
    with pytest.raises(_lib.AcsError):
        canonical_form(np.array([[0, 1, 2, 0]], np.int8))  # relator 0 not right-padded


def _same(got, want, row, cyc):
    assert got[0] == want[0], row
    assert got[1] == want[1], row
    for k in KEYS:
        assert got[2][k] == want[2][k], (k, row)
    if want[2]["status"] == 0:
        assert np.array_equal(got[2]["visited"], want[2]["visited"]), row
    if got[0]:
        assert S.replay(row, got[1], cyc) == 2


@pytest.mark.parametrize("cyc", [False, True])
def test_orbit_bfs_matches_oracle(cyc):
    """Visited order, counters, paths, budget cuts and raising rows of the orbit-BFS oracle, across the
    W = 1 / 2 switch, with budgets that cut inside the first levels and chunks of 7 parents."""
    budgets = (1, 7, 150, 1500)
    for mrl in (2, 3, 4, 16, 28, 29, 30, 33):
        R = roots(mrl)
        B = np.array([budgets[k % len(budgets)] for k in range(len(R))], np.int64)
        want = [S.orbit_bfs(r, int(b), cyc, want_visited=True) for r, b in zip(R, B)]
        for chunk in (0, 7):
            got = bfs_batch(R, B, cyc, want_visited=True, symmetric=True, chunk_parents=chunk)
            for r, g, w in zip(R, got, want):
                _same(g, w, r, cyc)


@pytest.mark.parametrize("cyc", [False, True])
def test_orbit_bfs_miller_schupp(miller_schupp, cyc):
    """The shortest Miller-Schupp rows at budget 3000 against the oracle; at budget 20 000, every row solved
    by both exact and orbit search has the same path length, and every orbit path replays."""
    mrls = np.asarray(miller_schupp["mrl"])
    order = [int(k) for k in np.argsort(mrls, kind="stable")[:24]]
    by_width = {}
    for k in order:
        by_width.setdefault(len(ms_row(miller_schupp, k)), []).append(k)
    groups = [np.array([ms_row(miller_schupp, k) for k in ks], np.int8) for ks in by_width.values()]
    for rows in groups:
        got = bfs_batch(rows, 3000, cyc, want_visited=True, symmetric=True)
        for r, g in zip(rows, got):
            _same(g, S.orbit_bfs(r, 3000, cyc, want_visited=True), r, cyc)
    sym = [bfs_batch(rows, 20_000, cyc, symmetric=True) for rows in groups]
    exact = bfs_groups(groups, 20_000, cyc)
    both = 0
    for rows, gs, ge in zip(groups, sym, exact):
        for r, a, b in zip(rows, gs, ge):
            if a[0]:
                assert S.replay(r, a[1], cyc) == 2
            if a[0] and b[0]:
                both += 1
                assert len(a[1]) == len(b[1]), r
    assert both >= 1


def test_orbit_states_are_canonical_and_distinct():
    R = roots(17)
    for (ok, _, info) in bfs_batch(R, 5000, False, want_visited=True, symmetric=True):
        V = info["visited"]
        c, _ = canonical_form(V)
        assert np.array_equal(c, V)
        assert len({v.tobytes() for v in V}) == len(V)


def test_orbit_search_refuses_exact_goal_sets():
    rows = roots(4)
    gs = GoalSet.from_rows(rows[:1], cyclically_reduce_after_moves=False)
    try:
        with pytest.raises(ValueError):
            bfs_batch(rows, 100, False, goals=gs, symmetric=True)
    finally:
        gs.close()
