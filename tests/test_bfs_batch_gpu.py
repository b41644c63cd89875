"""Batched breadth-first search (csrc/mbfs.cu) on the GPU: every row of a batch equals its own
single search (bfs_device, the reference fixtures, the oracle), whatever else shares the batch,
however the work is chunked and however the rows are split into engine runs."""

import contextlib
import hashlib
import io
import os

import numpy as np
import pytest

from conftest import ms_row
from oracle import oracle as O

pytestmark = pytest.mark.gpu

AK2 = np.array([1, 1, -2, -2, -2, 0, 0, 1, 2, 1, -2, -1, -2, 0])
KEYS = ("n_visited", "n_expanded", "n_moves", "frontier_left", "budget_hit", "status", "minlen_log", "n_levels")


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.int8).tobytes()).hexdigest()


def _same(a, b, visited=True):
    assert a[0] == b[0] and a[1] == b[1]
    for k in KEYS:
        assert a[2][k] == b[2][k], k
    if visited:
        assert ("visited" in a[2]) == ("visited" in b[2])
        if "visited" in a[2]:
            assert np.array_equal(a[2]["visited"], b[2]["visited"])


def _single(p, budget, cyc):
    from ac_solver_b200.search.breadth_first import bfs_device

    try:
        return bfs_device(np.asarray(p, np.int8), budget, cyc, want_visited=True)
    except (AssertionError, IndexError):
        return None  # the row raises: compared through its status


def _pad(p, mrl):
    p = np.asarray(p, np.int8)
    m = p.size // 2
    out = np.zeros(2 * mrl, np.int8)
    out[:m], out[mrl:mrl + m] = p[:m], p[m:]
    return out


def test_golden_cases_in_batches(search_cases, search_visited):
    """All reference bfs fixtures, run as one batch per (mrl, cyclical) with per-row budgets."""
    from ac_solver_b200 import bfs_batch

    groups = {}
    for c in search_cases["bfs"]:
        groups.setdefault((len(c["presentation"]), bool(c["cyclical"])), []).append(c)
    assert sum(len(g) for g in groups.values()) == len(search_cases["bfs"])
    for (_, cyc), cases in groups.items():
        out = bfs_batch(np.array([c["presentation"] for c in cases]), [c["budget"] for c in cases], cyc,
                        want_visited=True)
        for c, (solved, path, info) in zip(cases, out):
            assert solved == c["solved"], c
            assert path == (None if c["path"] is None else [tuple(x) for x in c["path"]]), c
            assert info["n_visited"] == c["n_visited"] and info["n_moves"] == c["n_moves"], c
            assert _sha(info["visited"]) == c["visited_sha256"], c
            if "visited_key" in c:
                assert np.array_equal(info["visited"], search_visited[c["visited_key"]])
            mins = [int(l.rsplit(" ", 1)[1]) for l in c["stdout"].splitlines() if l.startswith("New minimal")]
            assert info["minlen_log"] == mins, c
            assert info["budget_hit"] == ("Exiting search" in c["stdout"]), c


@pytest.mark.parametrize("budget", [10_000, 100_000])
@pytest.mark.parametrize("cyc", [False, True])
def test_batch_equals_single_on_miller_schupp_rows(miller_schupp, budget, cyc):
    """Rows of every mrl of the dataset: each row of a batch equals its single search, visited array included."""
    from ac_solver_b200 import bfs_groups

    by_width = {}
    for k in range(0, 1190, 37):
        by_width.setdefault(len(ms_row(miller_schupp, k)), []).append(k)
    assert len(by_width) == 6
    keys = list(by_width.values())
    outs = bfs_groups([np.array([ms_row(miller_schupp, k) for k in ks], np.int8) for ks in keys], budget, cyc,
                      want_visited=True)
    for ks, out in zip(keys, outs):
        for j, (k, got) in enumerate(zip(ks, out)):
            _same(got, _single(ms_row(miller_schupp, k), budget, cyc))
            if budget == 10_000 and j == 0:  # a subset against the oracle as well
                es, ep, ei = O.bfs(ms_row(miller_schupp, k), budget, cyclically_reduce_after_moves=cyc, want_visited=True)
                assert (got[0], got[1]) == (es, ep) and np.array_equal(got[2]["visited"], ei["visited"]), k


def _isolation_rows():
    """(mrl-8 rows, budgets): repeats, a raising row, tiny budgets, a first-level solve."""
    ak2 = _pad(AK2, 8)
    raising = _pad(np.array([1, 2, 0, 0, 1, 2, 0, 0]), 8)  # r0 == r1: move 1 empties r0
    first_level = _pad(np.array([1, 2, 0, 0, 2, 0, 0, 0]), 8)  # r0 r1^-1 -> length 2 in one move
    rows = [ak2, raising, ak2, first_level, ak2, ak2, ak2, _pad(np.array([1, 1, 2, 0, 2, 2, 1, 0]), 8)]
    budgets = [5000, 1000, 5000, 100, 1, 2, 13, 3000]
    return np.array(rows), budgets


def test_isolation_and_permutation():
    from ac_solver_b200 import bfs_batch

    rows, budgets = _isolation_rows()
    out = bfs_batch(rows, budgets, want_visited=True)
    assert out[1][2]["status"] == 1  # the reference raises AssertionError on this row
    assert out[3][0] and out[3][1][-1][1] == 2
    for r, b, got in zip(rows, budgets, out):
        ref = _single(r, b, False)
        if ref is None:
            assert got[2]["status"] != 0
        else:
            _same(got, ref)
    perm = np.random.default_rng(7).permutation(len(rows))
    out_p = bfs_batch(rows[perm], [budgets[i] for i in perm], want_visited=True)
    for j, i in enumerate(perm):
        _same(out_p[j], out[i])
    # wide keys: mrl 30 / 36 / 48 (two words per relator), repeated rows in one batch
    for mrl in (30, 36, 48):
        wide = np.array([_pad(AK2, mrl)] * 3 + [_pad(np.array([1, 2, 0, 0, 2, 0, 0, 0]), mrl)])
        outw = bfs_batch(wide, [20000, 13, 20000, 50], want_visited=True)
        for r, b, got in zip(wide, [20000, 13, 20000, 50], outw):
            _same(got, _single(r, b, False))


@pytest.mark.parametrize("chunk_parents", [1, 7, 64])
def test_chunk_boundaries(miller_schupp, chunk_parents):
    from ac_solver_b200 import bfs_batch

    rows = np.array([ms_row(miller_schupp, k) for k in range(0, 170, 9)], np.int8)
    for cyc in (False, True):
        ref = bfs_batch(rows, 3000, cyc, want_visited=True)
        got = bfs_batch(rows, 3000, cyc, want_visited=True, chunk_parents=chunk_parents)
        for a, b in zip(got, ref):
            _same(a, b)
    rows8, budgets = _isolation_rows()
    for a, b in zip(bfs_batch(rows8, budgets, want_visited=True, chunk_parents=chunk_parents),
                    bfs_batch(rows8, budgets, want_visited=True)):
        _same(a, b)


def test_byte_budget_splits_runs(miller_schupp):
    import ctypes as C

    from ac_solver_b200 import _lib, bfs_batch, bfs_groups

    rows = np.array([ms_row(miller_schupp, k) for k in range(0, 170, 5)], np.int8)
    one, three = C.c_int64(0), np.full(3, 20000, np.int64)
    _lib.check(_lib.lib().acs_bfs_batch_bytes(3, rows.shape[1] // 2, three.ctypes.data, 0, C.byref(one)))
    ref = bfs_batch(rows, 20000, want_visited=True)
    got = bfs_batch(rows, 20000, want_visited=True, max_bytes=one.value)  # about three rows per engine run
    for a, b in zip(got, ref):
        _same(a, b)
    # bfs_groups: engines of about three rows, about two engines per wave
    halves = [rows[:17], rows[17:]]
    got_g = bfs_groups(halves, 20000, want_visited=True, max_bytes=one.value, max_total_bytes=2 * one.value)
    for a, b in zip(got_g[0] + got_g[1], ref):
        _same(a, b)


def test_path_buffer_too_small_is_an_error_then_paths_are_fetched():
    """path_cap 0 (no buffer) or too small: the run reports every result and the needed length with an
    error, never a truncated path; acs_bfs_batch_paths then fetches the paths without searching again."""
    import ctypes as C

    from ac_solver_b200 import _lib

    L = _lib.lib()
    rows = np.array([_pad(AK2, 8), _pad(np.array([1, 2, 0, 0, 2, 0, 0, 0]), 8), _pad(AK2, 8)])
    budgets = np.array([10**6, 100, 10], np.int64)
    refs = [_single(r, int(b), False) for r, b in zip(rows, budgets)]
    assert refs[0][0] and refs[1][0] and not refs[2][0]
    h = C.c_void_p()
    _lib.check(L.acs_bfs_batch_create(_lib.default_device(), 3, 8, budgets.ctypes.data, 0, 0, C.byref(h)))
    try:
        for cap in (0, 2):
            res = (_lib.SearchResult * 3)()
            buf = np.zeros((3, max(cap, 1), 2), np.int32)
            rc = L.acs_bfs_batch_run(h, rows.ctypes.data, buf.ctypes.data if cap else None, cap, res)
            assert rc == _lib.ACS_ERR_INVALID
            for r, ref in zip(res, refs):
                assert r.n_visited == ref[2]["n_visited"] and bool(r.solved) == ref[0]
                assert r.path_len == (len(ref[1]) if ref[0] else 0)
        assert L.acs_bfs_batch_paths(h, None, 0) == _lib.ACS_ERR_INVALID
        cap = len(refs[0][1])
        paths = np.zeros((3, cap, 2), np.int32)
        _lib.check(L.acs_bfs_batch_paths(h, paths.ctypes.data, cap))
        for s in (0, 1):
            assert [tuple(int(v) for v in x) for x in paths[s, : len(refs[s][1])]] == refs[s][1]
        # no search can solve: a run without a path buffer succeeds
        one = np.array([10], np.int64)
        h2 = C.c_void_p()
        _lib.check(L.acs_bfs_batch_create(_lib.default_device(), 1, 8, one.ctypes.data, 0, 0, C.byref(h2)))
        try:
            res = (_lib.SearchResult * 1)()
            _lib.check(L.acs_bfs_batch_run(h2, np.ascontiguousarray(rows[2:]).ctypes.data, None, 0, res))
            assert res[0].n_visited == refs[2][2]["n_visited"] and res[0].budget_hit
        finally:
            L.acs_bfs_batch_destroy(h2)
    finally:
        L.acs_bfs_batch_destroy(h)


def test_sweep_known_answers(miller_schupp):
    """All 1190 rows at 1e6, both flags: the shipped BFS-solved lists, and every path replays to length 2."""
    import ac_solver_b200.search.miller_schupp as msp
    from ac_solver_b200 import bfs_groups

    rows = [ms_row(miller_schupp, k) for k in range(1190)]
    by_width = {}
    for k, r in enumerate(rows):
        by_width.setdefault(len(r), []).append(k)
    keys = list(by_width.values())
    groups = [np.array([rows[k] for k in ks], np.int8) for ks in keys]
    data = os.path.join(os.path.dirname(msp.__file__), "data")
    want_plain = {tuple(p) for p in msp.load_presentations_from_text_file(
        os.path.join(data, "bfs_solved_presentations_budget1e6.txt"))}
    assert len(want_plain) == 52
    want_cyc = {int(k) for k in miller_schupp["bfs_solved_index"]}
    for cyc in (True, False):
        solved = set()
        for ks, out in zip(keys, bfs_groups(groups, 1_000_000, cyc)):
            for k, (ok, path, info) in zip(ks, out):
                assert info["status"] == 0
                if not ok:
                    continue
                solved.add(k)
                state, mrl = np.array(rows[k], np.int8), len(rows[k]) // 2
                for action, length in path[1:]:
                    state = np.asarray(O.acmove(int(action), state, mrl, cyclical=cyc)[0], np.int8)
                    assert int(np.count_nonzero(state)) == length
                assert int(np.count_nonzero(state)) == 2, k
        if cyc:
            assert solved == want_cyc
        else:
            assert {tuple(int(v) for v in rows[k]) for k in solved} == want_plain


def test_trivialize_stdout_matches_per_row_bfs(capsys):
    """trivialize_miller_schupp_through_search(bfs) prints what per-row bfs() calls print, in order."""
    from ac_solver_b200 import bfs
    from ac_solver_b200.search.miller_schupp import (generate_miller_schupp_presentations,
                                                     trivialize_miller_schupp_through_search)

    budget = 3000
    got = trivialize_miller_schupp_through_search(1, 3, 1, 3, budget, bfs)
    out_batch = capsys.readouterr().out
    solved, unsolved, paths = [], [], []
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        for n in range(1, 4):
            g = generate_miller_schupp_presentations(n, 3)
            for lenw in range(1, 4):
                print(f"Applying bfs to presentations of n = {n}, lenw = {lenw}")
                for p in g.get(lenw, []):
                    ok, path = bfs(p, budget)
                    (solved if ok else unsolved).append(p)
                    if ok:
                        paths.append(path)
    assert out_batch == buf.getvalue()
    assert got == (solved, unsolved, paths)
