"""Batched beam search on the GPU (csrc/beam.cu): at every level each search keeps the ``beam_width``
shortest new states.  Between breadth-first search, which spends its budget on every state near the row,
and greedy search, which follows one state at a time, a beam reaches depth about budget / width with
12 * width candidates per search per level to spread over the GPU.
"""

from __future__ import annotations

import ctypes as C

import numpy as np

from .. import _lib
from ._common import BatchedEngine
from .breadth_first import DEFAULT_MAX_BYTES, _batch_inputs, _check_goals, _split_by

MAX_BEAM_WIDTH = 1 << 24


def _beam_bytes(L, mrl, beam_width, budgets, max_depth):
    b, arr = C.c_int64(0), np.ascontiguousarray(budgets, dtype=np.int64)
    _lib.check(L.acs_beam_bytes(len(arr), mrl, int(beam_width), arr.ctypes.data, int(max_depth), C.byref(b)))
    return b.value


class _BeamEngine(BatchedEngine):
    """One acs_beam engine over rows of a validated batch."""

    api, levels = "acs_beam", "levels"

    def __init__(self, L, dev, P8, budgets, beam_width, max_depth, cyclical, goals=None):
        self.L, self.P8 = L, np.ascontiguousarray(P8)
        self.S, w = P8.shape
        self.h = C.c_void_p()
        self.goals = goals
        b = np.ascontiguousarray(budgets, dtype=np.int64)
        _lib.check(L.acs_beam_create(dev, self.S, w // 2, int(beam_width), b.ctypes.data, int(max_depth),
                                     int(bool(cyclical)), C.byref(self.h)))
        try:
            if goals is not None:
                _lib.check(L.acs_beam_set_goals(self.h, goals.handle))
        except BaseException:
            self.destroy()
            raise


def _check_args(beam_width, max_depth):
    if isinstance(beam_width, bool) or int(beam_width) != beam_width or not 1 <= beam_width <= MAX_BEAM_WIDTH:
        raise ValueError(f"beam_width must be an int in [1, 2^24], got {beam_width!r}")
    if max_depth is not None and (isinstance(max_depth, bool) or int(max_depth) != max_depth or max_depth < 1):
        raise ValueError(f"max_depth must be None or an int >= 1, got {max_depth!r}")
    return int(beam_width), 0 if max_depth is None else int(max_depth)


def beam_search_batch(presentations, beam_width, max_nodes_to_explore, max_depth=None,
                      cyclically_reduce_after_moves=False, want_visited=False, device=None, goals=None,
                      max_bytes=DEFAULT_MAX_BYTES, _path_cap=256):
    """Beam search of every row of ``presentations`` [S, 2*mrl] in one device run (csrc/beam.cu).
    ``max_nodes_to_explore`` is one node budget (>= 1) or one per row.

    A search keeps a visited list V = [root] and a beam = [root].  At each level the candidates
    c = 12*i + m (move m applied to beam node i) are walked in increasing c; the first that has total length 2,
    or is in ``goals``, solves the search (a solve wins over a goal on the same child), and one on which the
    reference's ``ACMove`` raises ends it with ``info["status"] != 0``.  Otherwise the children whose state is
    not in V, each at its smallest c, are ordered by (total length, c); the first
    ``min(beam_width, budget - |V|)`` of them become the next beam and are appended to V.  A search stops
    after a level with no new child, that brought |V| to the budget (``info["budget_hit"]``), or the
    ``max_depth``-th level.

    Returns a list of ``(solved, path|None, info)``: the path in the reference's format
    ``[(-1, L_root), (action, total_length), ...]`` ends at the solving (or goal) child; ``info`` holds
    ``n_visited``, ``n_expanded``, ``n_moves``, ``frontier_left``, ``levels`` (levels kept), ``budget_hit``,
    ``status``, ``minlen_log`` (every new minimal total length in (level, c) order), ``seconds_device``;
    with ``goals`` also ``goal`` and ``goal_element`` as in ``bfs_batch``; with ``want_visited`` the rows of
    V in order.  A root in ``goals`` is a hit at depth 0 with the path ``[(-1, L0)]``.  Goal sets may be
    exact or symmetric; orbit search is not offered.  Rows are split into several engine runs when one
    engine would need more than ``max_bytes`` of device memory; the results do not depend on the split."""
    beam_width, depth = _check_args(beam_width, max_depth)
    P8, budgets = _batch_inputs(presentations, max_nodes_to_explore)
    if (budgets < 1).any():
        raise ValueError("max_nodes_to_explore must be at least 1")
    dev = _lib.default_device() if device is None else device
    mrl = P8.shape[1] // 2
    _check_goals(goals, mrl, cyclically_reduce_after_moves, dev)
    if P8.shape[0] == 0:
        return []
    L = _lib.lib()
    out = []
    for lo, hi, _ in _split_by(lambda b: _beam_bytes(L, mrl, beam_width, b, depth), budgets, max_bytes):
        e = _BeamEngine(L, dev, P8[lo:hi], budgets[lo:hi], beam_width, depth, cyclically_reduce_after_moves, goals)
        try:
            out += e.run(want_visited, _path_cap)
        finally:
            e.destroy()
    return out


def beam_search(presentation, beam_width, max_nodes_to_explore, max_depth=None, cyclically_reduce_after_moves=False,
                want_visited=False, device=None, goals=None):
    """``beam_search_batch`` of one row -> ``(solved, path|None, info)``."""
    row = np.asarray(presentation)
    if row.ndim != 1:
        raise ValueError("presentation must be one row of 2*max_relator_length letters")
    return beam_search_batch(row[None, :], beam_width, max_nodes_to_explore, max_depth, cyclically_reduce_after_moves,
                             want_visited, device, goals)[0]


def beam_meet_in_the_middle(presentations, beam_width, max_nodes_to_explore, ball, max_depth=None, device=None,
                            max_bytes=DEFAULT_MAX_BYTES):
    """Meet-in-the-middle beam search, without cyclic reduction: ``beam_search_batch`` of every row with
    ``ball`` (usually ``trivial_ball(...)``, exact or symmetric) as its goal set, stitched as in
    ``bfs_meet_in_the_middle``: a row solved directly keeps its beam path; a row that reached the ball gets
    its forward path followed by the ball path walked backwards -> ``(trivialized, path|None, info)``."""
    from .goals import _check_ball, _stitch_through_ball

    _check_ball(ball, "beam_meet_in_the_middle", "beam_search_batch")
    res = beam_search_batch(presentations, beam_width, max_nodes_to_explore, max_depth, False, device=device,
                            goals=ball, max_bytes=max_bytes)
    return _stitch_through_ball(res, ball)
