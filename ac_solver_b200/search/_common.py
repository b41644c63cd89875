"""Plumbing shared by the device search wrappers: host-side input checks, the ``info`` dict of a
``SearchResult``, the read-backs of visited states and goal hits, and the run of a batched engine."""

from __future__ import annotations

import ctypes as C

import numpy as np

from .. import _lib


def _raise_for(status):
    if status == _lib.ROW_ASSERT:
        raise AssertionError("a move produced an invalid presentation (empty relator): "
                             "the reference raises AssertionError here (envs/utils.py:261-263)")
    if status == _lib.ROW_INDEX:
        raise IndexError("index 0 is out of bounds for axis 0 with size 0")


def _check_alphabet(P):
    if P.size and np.abs(P.astype(np.int64)).max() > 2:  # wide: abs(int8 -128) is -128
        raise ValueError("the GPU search supports the two-generator alphabet {+-1, +-2} only")


def check_row(presentation):
    """One presentation -> contiguous int8 row, refused on the host before any GPU work."""
    p = np.asarray(presentation)
    if p.ndim != 1 or p.size % 2 or p.size == 0:
        raise AssertionError(f"{presentation} is not a valid presentation")
    _check_alphabet(p)
    return np.ascontiguousarray(p, dtype=np.int8)


def check_rows(presentations, shape_error="presentations must be [S, 2*max_relator_length]"):
    """A batch [S, 2*mrl] -> contiguous int8 rows, refused on the host before any GPU work."""
    P = np.asarray(presentations)
    if P.ndim != 2 or P.shape[1] % 2 or P.shape[1] == 0:
        raise ValueError(shape_error)
    _check_alphabet(P)
    return np.ascontiguousarray(P, dtype=np.int8)


def search_info(r, levels="n_levels"):
    """The ``info`` dict of one ``SearchResult``.  Its ``n_levels`` field goes under ``levels``: BFS levels, or
    for greedy search ``"rounds"`` (bucket rounds; -1 when the one-warp heap kernel served the search)."""
    return {
        "n_visited": int(r.n_visited), "n_expanded": int(r.n_expanded), "n_moves": int(r.n_moves),
        "frontier_left": int(r.frontier_left), "budget_hit": bool(r.budget_hit), levels: int(r.n_levels),
        "status": int(r.status), "minlen_log": [int(r.minlen_log[i]) for i in range(r.n_minlen)],
        "seconds_device": float(r.seconds_device),
    }


def fetch_visited(visited_fn, n_visited, width, *handle):
    """The visited states in insertion order, as int8 rows [n, width], through
    ``visited_fn(*handle, rows, cap_rows, &n_out)`` (acs_bfs_visited, acs_bfs_batch_visited, acs_greedy_visited)."""
    vis = np.zeros((max(int(n_visited), 1), width), np.int8)
    n_out = C.c_int64(0)
    _lib.check(visited_fn(*handle, vis.ctypes.data, vis.shape[0], C.byref(n_out)))
    return vis[: n_out.value]


def fetch_goal_hits(hits_fn, elements_fn, h, S):
    """Per search of a goal run, the ``info`` entries ``goal`` (the entry index) and ``goal_element`` (the
    symmetry u with u.(path end) = the entry's state); both ``None`` for a search that did not stop at a goal."""
    hits = np.full(S, -1, np.int64)
    _lib.check(hits_fn(h, hits.ctypes.data))
    elems = np.full(S, -1, np.int32)
    _lib.check(elements_fn(h, elems.ctypes.data))
    return [{"goal": int(hits[s]) if hits[s] >= 0 else None, "goal_element": int(elems[s]) if hits[s] >= 0 else None}
            for s in range(S)]


class BatchedEngine:
    """Handle of one batched device engine over the validated rows ``self.P8``: ``api`` names its C functions
    (``<api>_run``, ``_paths``, ``_visited``, ``_goal_hits``, ``_goal_hit_elements``, ``_destroy``) and ``levels`` is
    the ``info`` key of its level count.  A subclass creates the engine in ``self.h`` and sets ``self.L``,
    ``self.P8`` and ``self.goals``."""

    api = levels = None

    def run(self, want_visited, path_cap=256):
        """One run over the rows -> a list of ``(solved, path|None, info)``."""
        L, h, P8, api = self.L, self.h, self.P8, self.api
        S = P8.shape[0]
        cap = path_cap
        paths = np.zeros((S, cap, 2), np.int32)
        res = (_lib.SearchResult * S)()
        rc = getattr(L, api + "_run")(h, P8.ctypes.data, paths.ctypes.data, cap, res)
        need = max(int(res[s].path_len) for s in range(S))
        if rc == _lib.ACS_ERR_INVALID and need > cap:  # a deeper solution than the buffer: fetch the paths again
            cap = need
            paths = np.zeros((S, cap, 2), np.int32)
            rc = getattr(L, api + "_paths")(h, paths.ctypes.data, cap)
        _lib.check(rc)
        goal_info = None
        if self.goals is not None:
            goal_info = fetch_goal_hits(getattr(L, api + "_goal_hits"), getattr(L, api + "_goal_hit_elements"), h, S)
        out = []
        for s in range(S):
            r = res[s]
            info = search_info(r, self.levels)
            if goal_info is not None:
                info.update(goal_info[s])
            if want_visited and r.status == 0:
                info["visited"] = fetch_visited(getattr(L, api + "_visited"), r.n_visited, P8.shape[1], h, s)
            plist = [(int(a), int(l)) for a, l in paths[s, : r.path_len]] if r.solved else None
            out.append((bool(r.solved), plist, info))
        return out

    def destroy(self):
        if self.h:
            getattr(self.L, self.api + "_destroy")(self.h)
            self.h = None
