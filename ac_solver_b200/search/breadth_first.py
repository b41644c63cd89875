"""Breadth-first search of the AC graph -- drop-in for the reference's
``ac_solver/search/breadth_first.py`` (``bfs``), executed entirely on the GPU
(csrc/pbfs.cu, the partitioned engine with a world of one): same return value, same visited set in the same order at any node budget,
same console output.
"""

from __future__ import annotations

import ctypes as C

import numpy as np

from .. import _lib
from ..envs.utils import is_array_valid_presentation
from ._common import _raise_for, check_row, check_rows, fetch_goal_hits, fetch_visited, search_info


def bfs_device(presentation, max_nodes_to_explore=10000, cyclically_reduce_after_moves=False,
               want_visited=False, device=None):
    """Run the device search -> (solved, path|None, info).  ``info`` carries the counters the
    reference keeps implicitly (visited, expanded, moves, successive minimal lengths) and,
    on request, the visited states in insertion order as int8 rows."""
    L = _lib.lib()
    dev = _lib.default_device() if device is None else device
    p8 = check_row(presentation)
    mrl = p8.size // 2
    h = C.c_void_p()
    _lib.check(L.acs_bfs_create(None, dev, mrl, int(max_nodes_to_explore), int(bool(cyclically_reduce_after_moves)),
                                C.byref(h)))
    try:
        cap = 1 << 16
        path = np.zeros((cap, 2), np.int32)
        res = _lib.SearchResult()
        _lib.check(L.acs_bfs_run(h, p8.ctypes.data, path.ctypes.data, cap, C.byref(res)))
        info = search_info(res)
        if want_visited and res.status == 0:
            info["visited"] = fetch_visited(L.acs_bfs_visited, res.n_visited, 2 * mrl, h)
    finally:
        L.acs_bfs_destroy(h)
    _raise_for(res.status)
    plist = [(int(a), int(l)) for a, l in path[: res.path_len]] if res.solved else None
    return bool(res.solved), plist, info


DEFAULT_MAX_BYTES = 32 << 30  # device bytes of one batched engine; larger batches are split into several runs
# device bytes of the engines bfs_groups keeps alive at once (a B200 has 180 GB); more runs in several waves
DEFAULT_MAX_TOTAL_BYTES = 128 << 30


def _batch_inputs(presentations, max_nodes_to_explore):
    """Validate a batch on the host, before any GPU work -> (int8 rows, int64 budgets)."""
    P = check_rows(presentations)
    budgets = np.broadcast_to(np.asarray(max_nodes_to_explore, dtype=np.int64), (P.shape[0],))
    if np.ndim(max_nodes_to_explore) > 1 or (budgets < 0).any():
        raise ValueError("max_nodes_to_explore must be one non-negative int or one per row")
    for k in range(P.shape[0]):  # breadth_first.py:36-38
        assert is_array_valid_presentation(P[k]), f"row {k}: {P[k].tolist()} is not a valid presentation"
    return P, np.ascontiguousarray(budgets)


def _engine_bytes(L, mrl, budgets, chunk_parents):
    b, arr = C.c_int64(0), np.ascontiguousarray(budgets, dtype=np.int64)
    _lib.check(L.acs_bfs_batch_bytes(len(arr), mrl, arr.ctypes.data, int(chunk_parents), C.byref(b)))
    return b.value


def _split_by(engine_bytes, budgets, max_bytes):
    """Consecutive row ranges whose engines each need at most max_bytes (a single row may need more)
    -> list of (lo, hi, bytes), where ``engine_bytes(budgets[lo:hi])`` is the size of the engine of rows
    [lo, hi).  An engine's size grows with its rows, so each range end is found by bisection."""
    parts, lo = [], 0
    S = len(budgets)
    while lo < S:
        good, bad = lo + 1, S + 1  # rows [lo, good) fit (or are a single row); [lo, bad) do not
        if engine_bytes(budgets[lo:S]) <= max_bytes:
            good = S
        while bad - good > 1 and good < S:
            mid = (good + bad) // 2
            if engine_bytes(budgets[lo:mid]) <= max_bytes:
                good = mid
            else:
                bad = mid
        parts.append((lo, good, engine_bytes(budgets[lo:good])))
        lo = good
    return parts


def _split(L, mrl, budgets, chunk_parents, max_bytes):
    """``_split_by`` for ``bfs_batch`` engines."""
    return _split_by(lambda b: _engine_bytes(L, mrl, b, chunk_parents), budgets, max_bytes)


class _BatchEngine:
    """One acs_bfs_batch engine over rows [lo, hi) of a validated batch."""

    def __init__(self, L, dev, P8, budgets, cyclical, chunk_parents, goals=None, stop_at_trivial=True, symmetric=False):
        self.L, self.P8 = L, np.ascontiguousarray(P8)
        self.S, w = P8.shape
        self.h = C.c_void_p()
        self.goals = goals
        b = np.ascontiguousarray(budgets, dtype=np.int64)  # referenced until the call returns
        _lib.check(L.acs_bfs_batch_create(dev, self.S, w // 2, b.ctypes.data, int(bool(cyclical)), int(chunk_parents),
                                          C.byref(self.h)))
        try:
            if goals is not None or not stop_at_trivial:
                _lib.check(L.acs_bfs_batch_set_goals(self.h, goals.handle if goals is not None else None,
                                                     int(bool(stop_at_trivial))))
            if symmetric:
                _lib.check(L.acs_bfs_batch_set_symmetric(self.h, 1))
        except BaseException:
            self.destroy()
            raise

    def run(self, want_visited):
        L, S = self.L, self.S
        cap = 256
        paths = np.zeros((S, cap, 2), np.int32)
        res = (_lib.SearchResult * S)()
        rc = L.acs_bfs_batch_run(self.h, self.P8.ctypes.data, paths.ctypes.data, cap, res)
        need = max(int(res[s].path_len) for s in range(S))
        if rc == _lib.ACS_ERR_INVALID and need > cap:  # a deeper solution than the buffer: fetch the paths again
            cap = need
            paths = np.zeros((S, cap, 2), np.int32)
            rc = L.acs_bfs_batch_paths(self.h, paths.ctypes.data, cap)
        _lib.check(rc)
        goal_info = None
        if self.goals is not None:
            goal_info = fetch_goal_hits(L.acs_bfs_batch_goal_hits, L.acs_bfs_batch_goal_hit_elements, self.h, S)
        out = []
        for s in range(S):
            r = res[s]
            info = search_info(r)
            if goal_info is not None:
                info.update(goal_info[s])
            if want_visited and r.status == 0:
                info["visited"] = fetch_visited(L.acs_bfs_batch_visited, r.n_visited, self.P8.shape[1], self.h, s)
            plist = [(int(a), int(l)) for a, l in paths[s, : r.path_len]] if r.solved else None
            out.append((bool(r.solved), plist, info))
        return out

    def destroy(self):
        if self.h:
            self.L.acs_bfs_batch_destroy(self.h)
            self.h = None


def _check_goals(goals, mrl, cyclical, dev):
    if goals is None:
        return
    if goals.closed:
        raise ValueError("the goal set is closed")
    if goals.max_relator_length != mrl:
        raise ValueError(f"the goal set has max_relator_length {goals.max_relator_length}, the presentations {mrl}")
    if goals.cyclical != bool(cyclical):
        raise ValueError(f"the goal set was built with cyclically_reduce_after_moves={goals.cyclical}, "
                         f"the search uses {bool(cyclical)}")
    if goals.device != dev:
        raise ValueError(f"the goal set lives on device {goals.device}, the search runs on device {dev}")


def bfs_batch(presentations, max_nodes_to_explore=10000, cyclically_reduce_after_moves=False, want_visited=False,
              device=None, chunk_parents=0, max_bytes=DEFAULT_MAX_BYTES, goals=None, stop_at_trivial=True,
              symmetric=False):
    """Breadth-first search of every row of ``presentations`` [S, 2*mrl] in one device run
    (csrc/mbfs.cu).  ``max_nodes_to_explore`` is one budget or one per row.

    Returns a list of ``(solved, path|None, info)``, element s equal to ``bfs_device(row s, ...)``.
    A row on which the reference raises carries ``info["status"] != 0`` instead of raising.  Rows
    are split into several engine runs when one engine would need more than ``max_bytes`` of device
    memory; ``chunk_parents`` > 0 caps the parents expanded per chunk (the results do not depend on it).

    ``goals`` (a ``GoalSet`` of the same max_relator_length and ``cyclically_reduce_after_moves``):
    a search also stops at the first generated child that is in the set, tested right after the
    length-2 test, and reports it as solved with ``info["goal"]`` = the entry index (``None`` for
    rows that did not stop at a goal); the path then ends with (action, total length of the goal
    state).  ``info["goal_element"]`` is the element u of the presentation symmetries with u.(the state the
    path ends at) = the entry's stored state: 0 for an exact set, any element for a symmetric set
    (``GoalSet.from_rows(..., symmetric=True)``), which matches a state when any of its images is in the set.  A root in the set stops at depth 0 with the path ``[(-1, L0)]``.  ``stop_at_trivial=False``
    turns the length-2 rule off: searches run until a goal, their budget or exhaustion.

    ``symmetric=True`` runs orbit searches: breadth-first search over the orbits of the 16 presentation
    symmetries (``canonical_form``).  The root and every new state are stored as canonical forms, and a
    child is new when its canonical form is unseen, so each stored state stands for its whole orbit and the
    path lengths stay shortest.  Paths are moves of the input row in the format above; ``info["visited"]``
    holds the canonical states.  The node budget then counts orbits, so at a budget cut the solved rows can
    differ from exact search in both directions.  With ``goals`` the set must be symmetric: an orbit search
    knows the orbit of a child, not which of its states is in the set."""
    P8, budgets = _batch_inputs(presentations, max_nodes_to_explore)
    dev = _lib.default_device() if device is None else device
    _check_goals(goals, P8.shape[1] // 2, cyclically_reduce_after_moves, dev)
    if symmetric and goals is not None and not goals.symmetric:
        raise ValueError("an orbit search (symmetric=True) needs a symmetric goal set: it knows only the orbit "
                         "of a child, not which of its states is in the set")
    if P8.shape[0] == 0:
        return []
    L = _lib.lib()
    out = []
    for lo, hi, _ in _split(L, P8.shape[1] // 2, budgets, chunk_parents, max_bytes):
        e = _BatchEngine(L, dev, P8[lo:hi], budgets[lo:hi], cyclically_reduce_after_moves, chunk_parents, goals,
                         stop_at_trivial, symmetric)
        try:
            out += e.run(want_visited)
        finally:
            e.destroy()
    return out


def canonical_form(rows, device=None):
    """Canonical forms under the presentation symmetries, in one device call (csrc/sym.cu).

    The group has order 16: the 8 signed permutations of the generators (swap x and y, invert x, invert y)
    and the swap of the two relators; it maps AC' moves to AC' moves.  ``rows`` [n, 2*mrl] right-padded int8
    -> ``(canon, elements)``: ``canon[i]`` is the smallest image of row i in the order (length of relator 0,
    relator 0 read from its last letter, length of relator 1, relator 1 likewise; letters y < x < y^-1 <
    x^-1), ``elements[i]`` the smallest element g = 8r + 4s + 2a + b mapping the row there (s: swap x and y,
    then a: invert x, then b: invert y, then r: swap the relators)."""
    P = np.asarray(rows)
    if P.ndim != 2 or P.shape[1] % 2 or P.shape[1] == 0:
        raise ValueError("rows must be [n, 2*max_relator_length]")
    P8 = np.ascontiguousarray(P, dtype=np.int8)
    if not np.array_equal(P8, P):
        raise ValueError("rows must hold letters in {+-1, +-2} and 0 padding")
    L = _lib.lib()
    dev = _lib.default_device() if device is None else device
    out = np.empty_like(P8)
    elem = np.zeros(P8.shape[0], np.uint8)
    _lib.check(L.acs_canonical_form(dev, P8.shape[1] // 2, P8.ctypes.data, P8.shape[0], out.ctypes.data,
                                    elem.ctypes.data))
    return out, elem


def bfs_groups(groups, max_nodes_to_explore=10000, cyclically_reduce_after_moves=False, want_visited=False, device=None,
               chunk_parents=0, max_bytes=DEFAULT_MAX_BYTES, max_total_bytes=DEFAULT_MAX_TOTAL_BYTES, threads=8):
    """Sweep helper: ``groups`` is a list of presentation arrays [S_k, 2*mrl_k] (one per max_relator_length).
    Rows are split into engines of at most ``max_bytes`` each, and the engines into waves of at most
    ``max_total_bytes`` together.  Every engine of a wave is created before any of its searches runs
    (``cudaMalloc`` stalls behind running kernels, see ``greedy_search_groups``), then they run
    concurrently (one stream and one host thread each).  Returns one ``bfs_batch`` result list per group."""
    from concurrent.futures import ThreadPoolExecutor

    inputs = [_batch_inputs(P, max_nodes_to_explore) for P in groups]
    L = _lib.lib()
    dev = _lib.default_device() if device is None else device
    plan = []  # (group, lo, hi, bytes) in group and row order
    for g, (P8, budgets) in enumerate(inputs):
        if P8.shape[0]:
            plan += [(g, lo, hi, nb) for lo, hi, nb in _split(L, P8.shape[1] // 2, budgets, chunk_parents, max_bytes)]
    waves, total = [], 0
    for item in plan:
        if not waves or total + item[3] > max_total_bytes:
            waves.append([])
            total = 0
        waves[-1].append(item)
        total += item[3]
    out = [[] for _ in groups]
    for wave in waves:
        engines = []
        try:
            for g, lo, hi, _ in wave:
                P8, budgets = inputs[g]
                engines.append(_BatchEngine(L, dev, P8[lo:hi], budgets[lo:hi], cyclically_reduce_after_moves, chunk_parents))
            with ThreadPoolExecutor(max_workers=max(1, min(threads, len(engines)))) as pool:
                raw = list(pool.map(lambda e: e.run(want_visited), engines))
        finally:
            for e in engines:
                e.destroy()
        for (g, _, _, _), rows in zip(wave, raw):
            out[g] += rows
    return out


def bfs(presentation, max_nodes_to_explore=10000, verbose=False, cyclically_reduce_after_moves=False):
    """search/breadth_first.py:15-97.

    Returns ``(True, path)`` with ``path = [(-1, L0), (action, total_length), ...]`` ending in a
    state of total length 2, or ``(False, None)`` when the node budget is exhausted."""
    assert is_array_valid_presentation(presentation), f"{presentation} is not a valid presentation"
    solved, path, info = bfs_device(presentation, max_nodes_to_explore, cyclically_reduce_after_moves)
    if verbose:
        for m in info["minlen_log"]:
            print(f"New minimal length found: {m}")
    if solved:
        return True, path
    if info["budget_hit"]:
        print(f"Exiting search as number of explored nodes = {info['n_visited']} has exceeded the limit "
              f"{max_nodes_to_explore}")
    return False, None
