"""Host-side checks of the batched BFS (no GPU needed): argument validation happens before any
device work, and without a GPU the search fails loudly instead of falling back to the CPU."""

import numpy as np
import pytest


def test_bfs_batch_rejects_bad_shapes_and_alphabet():
    from ac_solver_b200 import bfs_batch

    with pytest.raises(ValueError):
        bfs_batch(np.array([1, 2, 0, 0, 2, 1, 0, 0]), 10)  # one row, not [S, 2*mrl]
    with pytest.raises(ValueError):
        bfs_batch(np.zeros((2, 7), np.int8), 10)  # odd width
    with pytest.raises(ValueError):
        bfs_batch(np.array([[1, 3, 0, 0, 2, 0, 0, 0]]), 10)  # letter outside {+-1, +-2}
    with pytest.raises(ValueError):
        bfs_batch(np.array([[1, -128, 2, 0]], np.int8), 10)  # abs(-128) overflows int8
    with pytest.raises(ValueError):
        bfs_batch(np.array([[1, 0, 2, 0]] * 2), [10, 20, 30])  # one budget per row
    with pytest.raises(ValueError):
        bfs_batch(np.array([[1, 0, 2, 0]]), -1)


def test_every_search_refuses_int8_minus_128_on_the_host():
    """abs() of int8 -128 is -128, so a plain abs test lets it through to the library: every wrapper checks
    the alphabet wide and raises the same ValueError as bfs_batch, before any device work."""
    from ac_solver_b200 import greedy_search, greedy_search_batch
    from ac_solver_b200.search.breadth_first import bfs_device
    from ac_solver_b200.search.greedy import greedy_search_groups
    from ac_solver_b200.search.partitioned import bfs_partitioned

    row = np.array([1, -128, 2, 0], np.int8)
    calls = [lambda: bfs_device(row, 10), lambda: bfs_partitioned(row, 10, sim_world=1),
             lambda: greedy_search(row, 10), lambda: greedy_search_batch(row[None, :], 10),
             lambda: greedy_search_groups([row[None, :]], 10)]
    for call in calls:
        with pytest.raises(ValueError, match="alphabet"):
            call()


def test_bfs_batch_names_the_invalid_row():
    from ac_solver_b200 import bfs_batch, bfs_groups

    rows = np.array([[1, 0, 2, 0], [1, 2, 0, 0], [0, 1, 2, 0]])  # rows 1 and 2: an empty / left-padded half
    with pytest.raises(AssertionError, match="row 1"):
        bfs_batch(rows, 10)
    with pytest.raises(AssertionError, match="row 0"):
        bfs_groups([np.array([[1, 0, 2, 0]]), np.array([[0, 1, 2, 0, 0, 0]])], 10)


def test_bfs_batch_without_gpu_raises():
    import torch
    from ac_solver_b200 import bfs_batch
    from ac_solver_b200._lib import AcsError

    if torch.cuda.is_available():
        pytest.skip("GPU present: the loud-failure path is for CPU-only hosts")
    with pytest.raises(AcsError):
        bfs_batch(np.array([[1, 0, 2, 0], [2, 0, 1, 0]]), 10)


def test_bfs_batch_bytes_plans_without_gpu():
    """The engine size is known on the host, and grows with the budgets."""
    import ctypes as C

    from ac_solver_b200 import _lib

    L = _lib.lib()

    def size(budgets, mrl=18):
        b = np.array(budgets, np.int64)
        out = C.c_int64(0)
        _lib.check(L.acs_bfs_batch_bytes(len(b), mrl, b.ctypes.data, 0, C.byref(out)))
        return out.value

    assert 0 < size([1000]) < size([1000, 1000]) < size([10**6, 10**6])
    assert size([10**6], mrl=36) > size([10**6], mrl=18)  # 48-byte nodes above mrl 29


def test_split_into_engine_runs_is_greedy_and_bounded():
    """Rows are cut into consecutive runs, each as long as the byte budget allows (a single row may exceed it)."""
    from ac_solver_b200 import _lib
    from ac_solver_b200.search.breadth_first import _engine_bytes, _split

    L = _lib.lib()
    budgets = np.array([10**5, 3 * 10**6, 10, 10**6, 10**6, 2 * 10**5, 7, 10**6] * 5, np.int64)
    for max_bytes in (1, 10**8, 3 * 10**8, 10**9, 10**12):
        parts = _split(L, 18, budgets, 0, max_bytes)
        assert parts[0][0] == 0 and parts[-1][1] == len(budgets)
        for (lo, hi, nb), nxt in zip(parts, parts[1:] + [None]):
            assert nb == _engine_bytes(L, 18, budgets[lo:hi], 0)
            assert nb <= max_bytes or hi == lo + 1
            if nxt is not None:  # one more row would not have fitted
                assert nxt[0] == hi and _engine_bytes(L, 18, budgets[lo:hi + 1], 0) > max_bytes
