"""Beam search without a GPU: the CPU statement (tests/beam_oracle.py) against the reference BFS where the
two must agree, the oracle's own invariants, argument checks of the C ABI and the Python wrapper before any
device work, the batch splitter, and the sm_100a compile of csrc/beam.cu."""

import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import beam_oracle as B
import goal_oracle as G
from conftest import ROOT, ms_row
from oracle import oracle as O

AK2 = np.array([1, 1, -2, -2, -2, 0, 0, 1, 2, 1, -2, -1, -2, 0], np.int8)
AK3 = np.array([1, 1, 1, -2, -2, -2, -2] + [0] * 17 + [1, 2, 1, -2, -1, -2] + [0] * 18, np.int8)


def _cases(ms):
    return [(AK2, False), (AK2, True), (AK3, False), (AK3, True)] + [(ms_row(ms, k), k % 2 == 1)
                                                                     for k in (0, 171, 345, 520, 700, 1100)]


@pytest.mark.parametrize("budget", [200, 3000])
def test_wide_beam_is_breadth_first_search(miller_schupp, budget):
    """With a width of at least the widest level, every beam is a whole BFS level: the states of every full
    level equal the reference BFS's, and both solve at the same depth."""
    for row, cyc in _cases(miller_schupp):
        bs, bp, bi = B.beam_search(row, budget, budget, cyclically_reduce_after_moves=cyc, want_visited=True,
                                   want_levels=True)
        fs, fp, fi = O.bfs(row, budget, cyclically_reduce_after_moves=cyc, want_visited=True)
        assert bi["status"] == fi["status"] == 0
        V, F = bi["visited"], fi["visited"]
        ends = np.cumsum([len(b) for b in bi["beams"]])
        full = [int(e) for e in ends if e <= min(len(V), len(F))]
        if bi["budget_hit"]:
            full = full[:-1]  # the budget may cut the last beam short of its level
        for n in full:
            assert {r.tobytes() for r in V[:n]} == {r.tobytes() for r in F[:n]}, n
        if bs and fs:
            assert len(bp) == len(fp)
            assert bp[-1][1] == fp[-1][1] == 2
        if fs and not bs:
            assert bi["budget_hit"]
        if bs and not fs:
            assert fi["budget_hit"]


@pytest.mark.parametrize("width,budget,depth", [(1, 50, None), (2, 100, None), (7, 500, None), (64, 2000, None),
                                                (7, 10_000, 4), (1000, 1500, None)])
def test_oracle_invariants(miller_schupp, width, budget, depth):
    """Every node of V is its parent's child by its move (C oracle), beams are at most the width, ordered by
    (total length, candidate id), and |V| never exceeds the budget."""
    for row, cyc in _cases(miller_schupp):
        solved, path, info = B.beam_search(row, width, budget, depth, cyc, want_visited=True, want_levels=True)
        V = info["visited"]
        assert len(V) <= budget and info["n_visited"] == len(V)
        mrl = row.size // 2
        beams = info["beams"]
        assert all(len(b) <= width for b in beams)
        if depth is not None:
            assert info["levels"] <= depth
        node = 1
        for d in range(1, len(beams)):
            prev = beams[d - 1]
            kids, lens, _ = O.moves_batch(np.repeat(V[prev], 12, axis=0), np.tile(np.arange(12, dtype=np.uint8),
                                                                                   len(prev)), cyclical=cyc)
            first = {}  # state -> (total length, smallest candidate id)
            for c in range(len(kids)):
                first.setdefault(kids[c].tobytes(), (int(lens[c].sum()), c))
            keys = []
            for v in beams[d]:
                assert v == node
                node += 1
                keys.append(first[V[v].tobytes()])  # KeyError: no child of the previous beam
            assert keys == sorted(keys)
        if solved:
            s = np.array(row, np.int8)
            for a, length in path[1:]:
                s, lens = O.acmove(a, s, mrl, cyclical=cyc)
                assert int(sum(lens)) == length
            assert path[-1][1] == 2


def test_oracle_goals_root_and_solve_over_goal():
    """A root in the goal set is a hit at depth 0; a child that solves and is a goal counts as a solve."""
    solved, path, info = B.beam_search(AK2, 4, 100, goals=G.goal_dict(AK2[None, :]))
    assert solved and path == [(-1, int(np.count_nonzero(AK2)))] and info["goal"] == 0
    assert info["n_visited"] == 1 and info["n_expanded"] == 0 and info["n_moves"] == 0
    row = np.array([1, 2, 0, 2, 0, 0], np.int8)  # xy, y: move 1 gives x, y
    child, _ = O.acmove(1, row, 3, cyclical=False)
    solved, path, info = B.beam_search(row, 4, 100, goals=G.goal_dict(child[None, :]))
    assert solved and info["goal"] is None and path[-1] == (1, 2)


def test_split_gives_bfs_batch_the_same_ranges():
    """The generalized splitter cuts a bfs_batch batch where the former bisection did."""
    from ac_solver_b200 import _lib
    from ac_solver_b200.build import build
    from ac_solver_b200.search.breadth_first import _engine_bytes, _split

    build()
    L = _lib.lib()

    def former(mrl, budgets, chunk_parents, max_bytes):
        parts, lo = [], 0
        S = len(budgets)
        while lo < S:
            good, bad = lo + 1, S + 1
            if _engine_bytes(L, mrl, budgets[lo:S], chunk_parents) <= max_bytes:
                good = S
            while bad - good > 1 and good < S:
                mid = (good + bad) // 2
                if _engine_bytes(L, mrl, budgets[lo:mid], chunk_parents) <= max_bytes:
                    good = mid
                else:
                    bad = mid
            parts.append((lo, good, _engine_bytes(L, mrl, budgets[lo:good], chunk_parents)))
            lo = good
        return parts

    rng = np.random.default_rng(5)
    for mrl, S in ((18, 37), (36, 200)):
        budgets = rng.integers(1, 200_000, S).astype(np.int64)
        total = _engine_bytes(L, mrl, budgets, 0)
        for max_bytes in (1, total // 7, total // 2, total, 10 * total):
            assert _split(L, mrl, budgets, 0, max_bytes) == former(mrl, budgets, 0, max_bytes)


def test_beam_split_respects_max_bytes():
    from ac_solver_b200 import _lib
    from ac_solver_b200.build import build
    from ac_solver_b200.search.beam import _beam_bytes
    from ac_solver_b200.search.breadth_first import _split_by

    build()
    L = _lib.lib()
    budgets = np.full(50, 10_000, np.int64)
    one = _beam_bytes(L, 18, 100, budgets[:1], 0)
    parts = _split_by(lambda b: _beam_bytes(L, 18, 100, b, 0), budgets, 5 * one)
    assert parts[0][0] == 0 and parts[-1][1] == 50
    assert all(nb <= 5 * one for _, _, nb in parts) and len(parts) > 1


def test_create_rejects_bad_arguments_before_opening_a_device():
    """Bad width, budget, depth and mrl are refused with a message before any device is opened: the calls
    below give the same codes on a host without a GPU."""
    from ac_solver_b200 import _lib
    from ac_solver_b200.build import build

    build()
    L = _lib.lib()
    budgets = np.array([100, 100], np.int64)
    h = C.c_void_p()

    def create(n=2, mrl=7, width=4, b=budgets, depth=0):
        return L.acs_beam_create(0, n, mrl, width, b.ctypes.data, depth, 0, C.byref(h))

    cases = [(dict(width=0), _lib.ACS_ERR_INVALID, "width"), (dict(width=-3), _lib.ACS_ERR_INVALID, "width"),
             (dict(b=np.array([100, 0], np.int64)), _lib.ACS_ERR_INVALID, "budget"),
             (dict(depth=-1), _lib.ACS_ERR_INVALID, "depth"), (dict(n=0), _lib.ACS_ERR_INVALID, "search"),
             (dict(width=(1 << 24) + 1), _lib.ACS_ERR_UNSUPPORTED, "width"),
             (dict(mrl=62), _lib.ACS_ERR_UNSUPPORTED, "max_relator_length"),
             (dict(mrl=0), _lib.ACS_ERR_UNSUPPORTED, "max_relator_length")]
    for kw, code, word in cases:
        assert create(**kw) == code, kw
        assert word in L.acs_last_error().decode(), kw
        assert not h.value
    b = C.c_int64(0)
    assert L.acs_beam_bytes(2, 7, 0, budgets.ctypes.data, 0, C.byref(b)) == _lib.ACS_ERR_INVALID
    assert L.acs_beam_bytes(2, 7, 4, budgets.ctypes.data, 0, C.byref(b)) == _lib.ACS_OK and b.value > 0


def test_python_wrapper_rejects_bad_arguments():
    from ac_solver_b200 import beam_search, beam_search_batch

    rows = np.array([AK2, AK2])
    for kw in (dict(beam_width=0), dict(beam_width=2.5), dict(beam_width=(1 << 24) + 1), dict(max_depth=0),
               dict(max_nodes_to_explore=0), dict(max_nodes_to_explore=[5, 6, 7])):
        args = dict(beam_width=4, max_nodes_to_explore=100)
        args.update(kw)
        with pytest.raises(ValueError):
            beam_search_batch(rows, **args)
    with pytest.raises(ValueError):
        beam_search(rows, 4, 100)
    with pytest.raises(ValueError, match="alphabet"):
        beam_search_batch(np.array([[1, -128, 2, 0]], np.int8), 4, 10)
    with pytest.raises(AssertionError, match="row 1"):
        beam_search_batch(np.array([[1, 0, 2, 0], [1, 2, 0, 0]]), 4, 10)


def test_beam_without_gpu_raises():
    import torch
    from ac_solver_b200 import beam_search_batch
    from ac_solver_b200._lib import AcsError

    if torch.cuda.is_available():
        pytest.skip("GPU present: the loud-failure path is for CPU-only hosts")
    with pytest.raises(AcsError):
        beam_search_batch(np.array([AK2]), 4, 10)


def test_beam_kernels_compile_for_sm100a(tmp_path):
    """Every kernel of csrc/beam.cu compiles for sm_100a without spills."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not installed")
    src = os.path.join(ROOT, "ac_solver_b200", "csrc", "beam.cu")
    out = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                          "-cubin", "-o", str(tmp_path / "beam.cubin"), src], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr[-2000:]
    log = out.stderr
    for name in ("bm_plan_kernel", "bm_prep_kernel", "bm_insert_kernel", "bm_hist_kernel", "bm_decide_kernel",
                 "bm_select_kernel", "mb_expand_kernel", "mb_goal_kernel", "mb_path_kernel"):
        assert name in log, name
    assert "sm_100a" in log
    spills = [int(x) for x in re.findall(r"(\d+) bytes spill stores", log)]
    assert spills and max(spills) == 0
