"""Greedy (best-first) search of the AC graph -- drop-in for the reference's
``ac_solver/search/greedy.py`` (``greedy_search``), executed on the GPU (csrc/greedy.cu), plus
the batched form used for the Miller-Schupp sweep (one CTA per presentation, one launch: a whole
(length, depth) bucket of the frontier is expanded per round, csrc/greedy_bucket.cuh).
"""

from __future__ import annotations

import ctypes as C

import numpy as np

from .. import _lib
from ._common import _raise_for, check_rows, fetch_goal_hits, fetch_visited, search_info
from .breadth_first import _check_goals


def _rows(res, paths, goal_info=None):
    """(solved, path, info) of every search of a run; ``goal_info`` from ``fetch_goal_hits`` for a goal run."""
    out = []
    for s, r in enumerate(res):
        info = search_info(r, "rounds")
        if goal_info is not None:
            info.update(goal_info[s])
        out.append((bool(r.solved), [(int(a), int(l)) for a, l in paths[s, : r.path_len]], info))
    return out


def greedy_search_batch(presentations, max_nodes_to_explore=10000, cyclically_reduce_after_moves=False,
                        want_visited=False, device=None, path_cap=None, goals=None):
    """Run greedy search on every row of ``presentations`` [S, 2*mrl] (same mrl) concurrently.

    Returns a list of ``(solved, path, info)`` per row, each identical to what the reference's
    ``greedy_search`` returns for that row (``path`` is the reference's failure path when not
    solved).  Rows whose first move raises in the reference carry ``info["status"] != 0``.

    ``goals`` (a ``GoalSet`` of the same max_relator_length and ``cyclically_reduce_after_moves``):
    a search also stops at the first generated child that is in the set, tested right after the
    length-2 test (the solve wins on the same child) and before the visited test.  It reports the
    row as solved with ``info["goal"]`` = the entry index (``None`` for rows that did not stop at a
    goal), and the path ends with (action, total length of the goal state).  A root in the set
    stops at depth 0 with the path ``[(-1, L0)]``.  Up to its first goal, a search follows the
    plain search exactly."""
    L = _lib.lib()
    dev = _lib.default_device() if device is None else device
    P8 = check_rows(presentations)
    S, w = P8.shape
    mrl = w // 2
    _check_goals(goals, mrl, cyclically_reduce_after_moves, dev)
    budget = int(max_nodes_to_explore)
    if path_cap is None:
        path_cap = int(min(budget + 4, 1 << 14))
    path_cap = max(path_cap, 4)
    h = C.c_void_p()
    _lib.check(L.acs_greedy_create(dev, S, mrl, budget, int(bool(cyclically_reduce_after_moves)), path_cap,
                                   C.byref(h)))
    try:
        if goals is not None:
            _lib.check(L.acs_greedy_set_goals(h, goals.handle))
        paths = np.zeros((S, path_cap, 2), np.int32)
        res = (_lib.SearchResult * S)()
        _lib.check(L.acs_greedy_run(h, P8.ctypes.data, paths.ctypes.data, res))
        need = max(r.path_len for r in res)
        if need > path_cap:  # deeper than the buffer: the reference has no limit -- run again with room
            L.acs_greedy_destroy(h)
            h = None
            return greedy_search_batch(presentations, max_nodes_to_explore, cyclically_reduce_after_moves, want_visited,
                                       device, path_cap=int(need) + 4, goals=goals)
        goal_info = None
        if goals is not None:
            goal_info = fetch_goal_hits(L.acs_greedy_goal_hits, L.acs_greedy_goal_hit_elements, h, S)
        out = _rows(res, paths, goal_info)
        if want_visited:
            for s, (_, _, info) in enumerate(out):
                if info["status"] == 0:
                    info["visited"] = fetch_visited(L.acs_greedy_visited, info["n_visited"], w, h, s)
    finally:
        if h is not None:
            L.acs_greedy_destroy(h)
    return out


def greedy_search_groups(groups, max_nodes_to_explore=10000, cyclically_reduce_after_moves=False, device=None,
                         path_cap=4096, threads=8):
    """Sweep helper: ``groups`` is a list of presentation arrays [S_k, 2*mrl_k] (one array per max_relator_length).
    All engines are CREATED first, then the groups search concurrently (one stream and one host thread each), then
    the engines are destroyed -- ``cudaMalloc`` stalls behind kernels that are already running (measured: 0.02-1.5 s
    per engine when interleaved with other groups' searches, 5 ms when not), so interleaving allocation and search
    costs a sweep more than the searches themselves.  Returns a list (per group) of ``greedy_search_batch`` results."""
    from concurrent.futures import ThreadPoolExecutor

    L = _lib.lib()
    dev = _lib.default_device() if device is None else device
    budget = int(max_nodes_to_explore)
    arrays, handles = [], []
    try:
        for P in groups:
            P8 = check_rows(P, "every group must be [S, 2*max_relator_length]")
            h = C.c_void_p()
            _lib.check(L.acs_greedy_create(dev, P8.shape[0], P8.shape[1] // 2, budget, int(bool(cyclically_reduce_after_moves)),
                                           int(path_cap), C.byref(h)))
            arrays.append(P8)
            handles.append(h)

        def run(k):
            P8, h = arrays[k], handles[k]
            S = P8.shape[0]
            paths = np.zeros((S, path_cap, 2), np.int32)
            res = (_lib.SearchResult * S)()
            _lib.check(L.acs_greedy_run(h, P8.ctypes.data, paths.ctypes.data, res))
            return paths, res

        with ThreadPoolExecutor(max_workers=max(1, min(threads, len(arrays) or 1))) as pool:
            raw = list(pool.map(run, range(len(arrays))))
    finally:
        for h in handles:
            L.acs_greedy_destroy(h)
    out = []
    for k, (paths, res) in enumerate(raw):
        S = arrays[k].shape[0]
        if any(res[s].path_len > path_cap for s in range(S)):  # deeper than the buffer: redo this group with room
            out.append(greedy_search_batch(arrays[k], budget, cyclically_reduce_after_moves, device=dev,
                                           path_cap=int(max(res[s].path_len for s in range(S))) + 4))
            continue
        out.append(_rows(res, paths))
    return out


def greedy_search(presentation, max_nodes_to_explore=10000, verbose=False, cyclically_reduce_after_moves=False):
    """search/greedy.py:15-121.

    Returns ``(True, path)`` or ``(False, path_of_last_expanded_node + [(11, length)])`` exactly as
    the reference does (its failure value is a path, not ``None``)."""
    p = np.array(presentation, dtype=np.int8)
    mrl = p.size // 2
    solved, path, info = greedy_search_batch(p[None, :], max_nodes_to_explore, cyclically_reduce_after_moves)[0]
    if verbose:
        for m in info["minlen_log"]:
            print(f"New minimal length found: {m}")
    _raise_for(info["status"])
    if solved:
        if verbose:  # greedy.py:92-99: the three lines of the reference, from a replay of the path
            from ..envs.ac_moves import ACMove

            state, lens = p.copy(), [0, 0]
            for action, _ in path[1:]:
                state, lens = ACMove(action, state, mrl, lens, cyclical=cyclically_reduce_after_moves)
            print(f"Found {state[0:1], state[mrl:mrl + 1]} after exploring "
                  f"{info['n_visited'] - info['frontier_left']} nodes")
            print(f"Path to a trivial state: (tuples are of form (action, length of a state)) {path}")
            print(f"Total path length: {len(path)}")
        return True, path
    if info["budget_hit"]:
        print(f"Exiting search as number of explored nodes = {info['n_visited']} has exceeded the limit "
              f"{max_nodes_to_explore}")
    return False, path
