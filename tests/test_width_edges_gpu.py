"""Every device search at the edges of the packed key layout (csrc/ac_keys.cuh), against the oracle bit for
bit: the roots of tests/width_edges.py at max_relator_length 1-4, 15-17, 28-33 and 60-61, both
``cyclical`` flags.  Each engine packs, unpacks and hashes ``Key<W>`` on its own, so each one is compared:
solved flag and path, counters, minimal-length log and the visited array in insertion order.  A row on
which the reference raises is compared through the status it reports or the exception it raises."""

import functools
import hashlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import goal_oracle as G
from ac_solver_b200 import _lib
from greedy_goal_oracle import greedy_goals
from oracle import oracle as O
from width_edges import BUDGET, WIDTHS, full_length_count, oracle_or_status, relator_lengths, roots

pytestmark = pytest.mark.gpu

KEYS = ("n_visited", "n_expanded", "n_moves", "frontier_left", "budget_hit", "minlen_log")
CYC = [False, True]
GOAL_BUDGET = 5000  # the goal oracles are Python loops
ORACLES = {"bfs": O.bfs, "greedy": O.greedy_search}


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.int8).tobytes()).hexdigest()


@functools.lru_cache(maxsize=None)
def _refs(search, mrl, cyc, budget):
    """Oracle runs of every root -> list of a row status or (solved, path, info); the visited array is kept
    as its hash (``info["visited_sha"]``) so that the whole table stays cached across the tests."""

    def one(r):
        out = oracle_or_status(ORACLES[search], r, budget, cyc, want_visited=True)
        if not isinstance(out, int):
            out[2]["visited_sha"] = _sha(out[2].pop("visited"))
        return out

    O.lib()  # build and load the oracle here: oracle.lib() is not safe to enter from several threads at once
    with ThreadPoolExecutor(8) as pool:
        return list(pool.map(one, roots(mrl)))


def _same(got, ref, what):
    """``got``: an engine's (solved, path, info), or the status of the exception it raised."""
    if isinstance(ref, int):  # the reference raises on this row
        assert (got if isinstance(got, int) else got[2]["status"]) == ref, what
        return
    assert not isinstance(got, int), f"{what}: the engine raised status {got}, the oracle did not"
    assert got[2]["status"] == 0, what
    assert (got[0], got[1]) == (ref[0], ref[1]), what
    for k in KEYS:
        assert got[2][k] == ref[2][k], (what, k)
    vis = got[2]["visited"]
    if "visited_sha" in ref[2]:
        if _sha(vis) != ref[2]["visited_sha"]:  # recompute the oracle's array to say where they part
            r, budget, cyc, fn = what[-1]
            want = fn(r, budget, cyc, want_visited=True)[2]["visited"]
            bad = next((i for i in range(min(len(vis), len(want))) if not np.array_equal(vis[i], want[i])), None)
            pytest.fail(f"{what[:-1]}: visited arrays differ at row {bad} of {len(vis)} / {len(want)}")
    else:
        assert np.array_equal(vis, ref[2]["visited"]), what


def _check_all(got_rows, search, mrl, cyc, budgets, label):
    """Row s of ``got_rows`` against the oracle run of root s at ``budgets[s]``."""
    R = roots(mrl)
    for s, (got, budget) in enumerate(zip(got_rows, budgets)):
        ref = _refs(search, mrl, cyc, budget)[s % len(R)]
        _same(got, ref, (label, mrl, cyc, s, budget, (R[s % len(R)], budget, cyc, ORACLES[search])))


# ---- breadth-first engines -------------------------------------------------------------------------------


@pytest.mark.parametrize("cyc", CYC)
@pytest.mark.parametrize("mrl", WIDTHS)
def test_bfs_device(mrl, cyc):
    from ac_solver_b200.search.breadth_first import bfs_device

    R = roots(mrl)
    for budget in (0, 1, BUDGET):
        got = [oracle_or_status(bfs_device, r, budget, cyc, want_visited=True) for r in R]
        _check_all(got, "bfs", mrl, cyc, [budget] * len(R), "bfs_device")


@pytest.mark.parametrize("cyc", CYC)
@pytest.mark.parametrize("mrl", [29, 61])
def test_bfs_device_large_budget(mrl, cyc):
    """200 000 nodes from a long relator 0 beside a short relator 1 (tens of thousands of full-length states)."""
    from ac_solver_b200.search.breadth_first import bfs_device

    r = roots(mrl)[0]
    got = bfs_device(r, 200_000, cyc, want_visited=True)
    ref = O.bfs(r, 200_000, cyc, want_visited=True)
    assert got[2]["budget_hit"] and full_length_count(ref[2]["visited"], mrl) > 20_000
    _same(got, ref, ("bfs_device", mrl, cyc, 0, 200_000))


@pytest.mark.parametrize("world,stage", [(1, None), (3, None), (3, "0")])
@pytest.mark.parametrize("cyc", CYC)
@pytest.mark.parametrize("mrl", WIDTHS)
def test_bfs_partitioned(mrl, cyc, world, stage, monkeypatch):
    """Levels of many chunks; at world 3 both expansion paths (block-staged records, and ACS_PBFS_CTA_STAGE=0:
    warp-staged), read when the engine is created."""
    from ac_solver_b200.search.partitioned import bfs_partitioned

    if stage is None:
        monkeypatch.delenv("ACS_PBFS_CTA_STAGE", raising=False)
    else:
        monkeypatch.setenv("ACS_PBFS_CTA_STAGE", stage)
    R = roots(mrl)
    got = [oracle_or_status(bfs_partitioned, r, BUDGET, cyc, want_visited=True, chunk_parents=1000, sim_world=world,
                            verbose=None) for r in R]
    _check_all(got, "bfs", mrl, cyc, [BUDGET] * len(R), f"bfs_partitioned world {world} stage {stage}")


@pytest.mark.parametrize("cyc", CYC)
@pytest.mark.parametrize("mrl", [16, 29, 30, 32, 61])
def test_bfs_sharded_world1(mrl, cyc):
    from ac_solver_b200.search.sharded import bfs_sharded

    R = roots(mrl)
    got = [oracle_or_status(bfs_sharded, r, BUDGET, cyc, want_visited=True, chunk_parents=1000) for r in R]
    _check_all(got, "bfs", mrl, cyc, [BUDGET] * len(R), "bfs_sharded")


@pytest.mark.parametrize("cyc", CYC)
@pytest.mark.parametrize("mrl", WIDTHS)
def test_bfs_batch(mrl, cyc):
    """Every root at 20 000 and again at 0 or 1 in one batch; each row equals its own oracle run, however
    the parents are chunked."""
    from ac_solver_b200 import bfs_batch

    R = roots(mrl)
    rows = np.concatenate([R, R])
    budgets = [BUDGET] * len(R) + [k % 2 for k in range(len(R))]
    for chunk in (0, 7):
        got = bfs_batch(rows, budgets, cyc, want_visited=True, chunk_parents=chunk)
        _check_all(got, "bfs", mrl, cyc, budgets, f"bfs_batch chunk_parents {chunk}")


# ---- greedy ----------------------------------------------------------------------------------------------


@pytest.mark.parametrize("kernel", ["bucket", "heap"])
@pytest.mark.parametrize("cyc", CYC)
@pytest.mark.parametrize("mrl", WIDTHS)
def test_greedy(mrl, cyc, kernel, monkeypatch):
    """The pop order (rel_cmp / key_less on full relators) is pinned by the visited order; the failure path
    by the path."""
    from ac_solver_b200 import greedy_search_batch

    if kernel == "heap":
        monkeypatch.setenv("ACS_GREEDY_KERNEL", "heap")
    else:
        monkeypatch.delenv("ACS_GREEDY_KERNEL", raising=False)
    R = roots(mrl)
    for budget in (0, BUDGET):
        got = greedy_search_batch(R, budget, cyc, want_visited=True)
        _check_all(got, "greedy", mrl, cyc, [budget] * len(R), f"greedy {kernel}")
        # info["rounds"]: bucket rounds of a search the bucket kernel served, -1 for one the heap kernel served
        if kernel == "heap":
            assert all(a[2]["rounds"] == -1 for a in got if a[2]["status"] == 0)
        else:
            assert any(a[2]["rounds"] >= 0 for a in got if a[2]["status"] == 0)


# ---- goal sets -------------------------------------------------------------------------------------------


def _deep_full_state(visited, mrl, frac):
    """The first state with a full-length relator at or after position frac of the FIFO, or None."""
    l0, l1 = relator_lengths(visited, mrl)
    full = np.flatnonzero((l0 == mrl) | (l1 == mrl))
    full = full[full >= max(1, int(frac * len(visited)))]
    return visited[full[0]] if len(full) else None


def _goal_rows(search, mrl, cyc, fracs):
    fn = ORACLES[search]
    out = []
    for r in roots(mrl):
        ref = oracle_or_status(fn, r, GOAL_BUDGET, cyc, want_visited=True)
        if isinstance(ref, int):
            continue
        for frac in fracs:
            s = _deep_full_state(ref[2]["visited"], mrl, frac)
            if s is not None:
                out.append(s)
    return np.array(out, np.int8).reshape(len(out), 2 * mrl)


def _same_goal(got, ref, what):
    if ref[2]["status"]:
        assert got[2]["status"] == ref[2]["status"], what
        return
    _same(got, ref, what)
    assert got[2]["goal"] == ref[2]["goal"], what


@pytest.mark.parametrize("cyc", CYC)
@pytest.mark.parametrize("mrl", WIDTHS)
def test_goal_membership(mrl, cyc):
    """Goal sets of full-length states deep in the oracle's own FIFO: bfs_batch equals the goal oracle for
    goals halfway and nine tenths in; greedy_search_batch for goals from its own visited arrays and from
    the breadth-first ones.  Hit entry, path, counters and visited array all match.

    At mrl 1 no search generates a new state (the first child has total length 2, or a move raises), so
    the goals there are the roots themselves: every search, a raising one included, stops at depth 0."""
    from ac_solver_b200 import GoalSet, bfs_batch, greedy_search_batch

    R = roots(mrl)
    hits = 0
    if mrl == 1:
        runs = [("bfs", R), ("greedy", R)]
    else:
        runs = [("bfs", _goal_rows("bfs", mrl, cyc, [f])) for f in (0.5, 0.9)]
        runs.append(("greedy", np.concatenate([_goal_rows("greedy", mrl, cyc, [0.5, 0.9]), runs[0][1]])))
    for search, goals in runs:
        gd = G.goal_dict(goals)
        with GoalSet.from_rows(goals, cyc) as g:
            assert g.n_entries == len(goals) and g.n_states == len(gd)
            if search == "bfs":
                got = bfs_batch(R, GOAL_BUDGET, cyc, want_visited=True, goals=g)
            else:
                got = greedy_search_batch(R, GOAL_BUDGET, cyc, want_visited=True, goals=g)
        for s, (r, a) in enumerate(zip(R, got)):
            if search == "bfs":
                ref = G.bfs_goals(r, GOAL_BUDGET, cyc, goals=gd, want_visited=True)
            else:
                ref = greedy_goals(r, GOAL_BUDGET, cyc, goals=gd, want_visited=True)
            _same_goal(a, ref, (f"{search} goals", mrl, cyc, s))
            hits += ref[2]["goal"] is not None
    assert hits == 2 * len(R) if mrl == 1 else hits >= 3


@pytest.mark.parametrize("cyc", CYC)
@pytest.mark.parametrize("mrl", WIDTHS)
def test_goal_set_from_exploration(mrl, cyc):
    """GoalSet.explore: the entries are the oracle's visited arrays in (search, FIFO) order; sampled entries,
    every full-length one among them, replay from their root and are found at depth 0 under their smallest
    index."""
    from ac_solver_b200 import GoalSet, bfs_batch

    budget = 3000
    plain = [G.bfs_goals(r, budget, cyc, stop_at_trivial=False, want_visited=True) for r in roots(mrl)]
    keep = [s for s, p in enumerate(plain) if p[2]["status"] == 0]  # a raising search has no exploration
    R = roots(mrl)[keep]
    vis = np.concatenate([plain[s][2]["visited"] for s in keep])
    root_of = np.concatenate([np.full(len(plain[s][2]["visited"]), j) for j, s in enumerate(keep)])
    first = G.goal_dict(vis)
    with GoalSet.explore(R, budget, cyc) as g:
        assert g.n_entries == len(vis) and g.n_states == len(first)
        assert [r[2]["n_visited"] for r in g.results] == [plain[s][2]["n_visited"] for s in keep]
        l0, l1 = relator_lengths(vis, mrl)
        full = np.flatnonzero((l0 == mrl) | (l1 == mrl))
        assert len(full) > 0
        rng = np.random.default_rng(mrl)
        ends = np.cumsum([0] + [len(plain[s][2]["visited"]) for s in keep])
        picks = set(rng.choice(full, min(len(full), 48), replace=False).tolist())
        picks |= set(rng.choice(len(vis), min(len(vis), 16), replace=False).tolist())
        picks |= set(ends[:-1].tolist()) | set((ends[1:] - 1).tolist())
        for e in sorted(picks):
            root, path = g.path(e)
            assert root == root_of[e], e
            state = np.asarray(R[root], np.int8)
            assert path[0] == (-1, int(np.count_nonzero(state))), e
            for a, length in path[1:]:
                state = np.asarray(O.acmove(int(a), state, mrl, cyclical=cyc)[0], np.int8)
                assert int(np.count_nonzero(state)) == length, e
            assert np.array_equal(state, vis[e]), e
        probe = sorted(set(rng.choice(full, min(len(full), 200), replace=False).tolist()))
        for e, h in zip(probe, bfs_batch(vis[probe], 10, cyc, goals=g)):
            assert h[0] and h[2]["goal"] == first[vis[e].tobytes()], e


# ---- the refusal past the last two-word width --------------------------------------------------------------


def test_searches_refuse_widths_past_61():
    """Every search, goal set and ball refuses mrl 62-64 with an error (the step kernel serves them; a key
    holds at most 61 letters per relator), and the library goes on working.  The step kernel at 62 and 63,
    in its byte path, equals the oracle on rows that fill the width."""
    from ac_solver_b200 import GoalSet, ac_moves_batch, bfs_batch, greedy_search_batch, trivial_ball
    from ac_solver_b200.search.breadth_first import bfs_device
    from ac_solver_b200.search.partitioned import bfs_partitioned
    from ac_solver_b200.synthetic import random_actions, random_presentations

    msg = "1 <= max_relator_length <= 61"
    for mrl in (62, 63, 64):
        r = random_presentations(1, mrl, seed=mrl, min_len=mrl - 2)
        calls = [lambda: bfs_device(r[0], 100), lambda: bfs_batch(r, 100),
                 lambda: bfs_partitioned(r[0], 100, sim_world=1, verbose=None),
                 lambda: greedy_search_batch(r, 100), lambda: GoalSet.from_rows(r), lambda: trivial_ball(mrl, 100)]
        for call in calls:
            with pytest.raises(_lib.AcsError, match=msg):
                call()
    for mrl in (62, 63):
        S = np.concatenate([random_presentations(2000, mrl, seed=mrl, min_len=mrl - 3),
                            random_presentations(2000, mrl, seed=mrl + 1, max_len=4)])
        S[2000:, :mrl] = S[:2000, :mrl]  # full-length relator 0 beside a short relator 1
        A = random_actions(len(S), seed=mrl)
        for cyc in CYC:
            out, lens, status = ac_moves_batch(S, A, cyclical=cyc)
            eo, el, es = O.moves_batch(S, A, cyclical=cyc)
            assert np.array_equal(status, es) and np.array_equal(out, eo)
            assert np.array_equal(lens[es == 0], el[es == 0])
            assert (lens[es == 0] == mrl).any()
    r = roots(61)[0]
    _same(bfs_device(r, 1000, want_visited=True), O.bfs(r, 1000, want_visited=True), ("bfs_device after", 61))
