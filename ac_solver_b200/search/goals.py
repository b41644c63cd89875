"""Goal sets for the batched breadth-first and greedy searches (csrc/goalset.cu, csrc/mbfs.cu, csrc/greedy.cu).

A goal set is a device-resident set of states.  ``bfs_batch(..., goals=g)`` stops a search at the
first generated child that is in ``g``.  Meet-in-the-middle uses it with a large ball of states
around the trivial presentations (``trivial_ball``): a forward search that reaches the ball is
trivialized by the forward path followed by the ball path walked backwards
(``bfs_meet_in_the_middle``, ``greedy_meet_in_the_middle``).  ``greedy_search_batch(..., goals=g)``
runs the same goal test in the greedy engine (csrc/greedy.cu).
"""

from __future__ import annotations

import ctypes as C

import numpy as np

from .. import _lib
from ..envs.utils import generate_trivial_states, is_array_valid_presentation
from ._common import check_rows
from .breadth_first import DEFAULT_MAX_BYTES, _BatchEngine, _batch_inputs, bfs_batch

# the move that undoes each of the 12 moves when relators are only freely reduced (bfs_common.cuh, skip_moves):
# r1 <- r1 r0^{+-1} (0, 2), r0 <- r0 r1^{-+1} (1, 3), and conjugation by g / g^-1 (4..7 <-> 8..11)
INVERSE_MOVE = (2, 3, 0, 1, 8, 9, 10, 11, 4, 5, 6, 7)

# The presentation symmetries of csrc/ac_sym.cuh: element g = 8r + 4s + 2a + b (swap x <-> y, then invert x,
# then invert y, then swap the relators).  sym_mul(g, h) is "h, then g"; move m on a state is move PI[g][m]
# on g.state.


def sym_mul(g, h):
    sg, ah, bh = g >> 2 & 1, h >> 1 & 1, h & 1
    a, b = (g >> 1 & 1) ^ (bh if sg else ah), (g & 1) ^ (ah if sg else bh)
    return ((g ^ h) & 12) | a << 1 | b


def sym_inv(g):
    return (g & 12) | (g & 1) << 1 | (g >> 1 & 1) if g & 4 else g


PI = [[int(T >> (4 * m) & 15) for m in range(12)] for T in (
    0xBA9876543210, 0xB6587A943210, 0x7A94B6583210, 0x7654BA983210,
    0x587A94B63210, 0x987654BA3210, 0x54BA98763210, 0x94B6587A3210,
    0x49A7856B0123, 0x456789AB0123, 0x89AB45670123, 0x856B49A70123,
    0x6789AB450123, 0xA7856B490123, 0x6B49A7850123, 0xAB4567890123)]


def _goal_rows(rows, cyclical):
    """Validate goal rows on the host -> int8 rows.  A row must be a state a search can generate."""
    R8 = check_rows(rows, "goal rows must be [n, 2*max_relator_length]")
    mrl = R8.shape[1] // 2
    for k in range(R8.shape[0]):
        if not is_array_valid_presentation(R8[k]):
            raise ValueError(f"goal row {k}: {R8[k].tolist()} is not a valid presentation "
                             "(an empty relator, or zeros before letters)")
        for h in range(2):
            r = R8[k, h * mrl:(h + 1) * mrl]
            r = r[: np.count_nonzero(r)].astype(np.int64)
            if (r[:-1] == -r[1:]).any():
                raise ValueError(f"goal row {k}: relator {h} is not freely reduced, so no search generates it")
            if cyclical and r.size > 1 and r[0] == -r[-1]:
                raise ValueError(f"goal row {k}: relator {h} is not cyclically reduced, so no search with "
                                 "cyclically_reduce_after_moves=True generates it")
    return R8


class GoalSet:
    """A set of states on one GPU, built with ``from_rows`` or ``explore``.  Entry ``i`` holds a state,
    its parent entry and the move from it, and its root; a state held by several entries is represented
    by the smallest entry index.  Free it with ``close()`` or a ``with`` block."""

    def __init__(self, handle, max_relator_length, cyclical, device, results=None):
        self.handle = handle
        flag = C.c_int(0)
        _lib.check(_lib.lib().acs_goalset_is_symmetric(handle, C.byref(flag)))
        self.symmetric = bool(flag.value)  # entries are canonical forms; a state matches when any image is held
        self.max_relator_length = int(max_relator_length)
        self.cyclical = bool(cyclical)
        self.device = int(device)
        self.results = results  # explore: the (solved, path, info) of every root's search

    @classmethod
    def from_rows(cls, rows, cyclically_reduce_after_moves=False, device=None, symmetric=False):
        """Entries are the rows [n, 2*mrl], each its own root.  Rows must be freely reduced (and
        cyclically reduced with ``cyclically_reduce_after_moves``): no search generates other rows.
        ``symmetric=True`` stores each row's canonical form (``canonical_form``): the set then holds every
        image of its rows under the 16 presentation symmetries."""
        R8 = _goal_rows(rows, cyclically_reduce_after_moves)
        L = _lib.lib()
        dev = _lib.default_device() if device is None else device
        h = C.c_void_p()
        fn = L.acs_goalset_from_rows_symmetric if symmetric else L.acs_goalset_from_rows
        _lib.check(fn(dev, R8.shape[1] // 2, int(bool(cyclically_reduce_after_moves)),
                                           R8.ctypes.data, R8.shape[0], C.byref(h)))
        return cls(h, R8.shape[1] // 2, cyclically_reduce_after_moves, dev)

    @classmethod
    def explore(cls, roots, max_nodes_to_explore, cyclically_reduce_after_moves=False, device=None, chunk_parents=0,
                symmetric=False):
        """Breadth-first search from every root with the length-2 rule off (each search runs until its
        budget or exhaustion), in one engine; every visited state becomes an entry, in (root, visit order)
        order.  ``results`` keeps each root's ``(solved, path, info)``.  ``symmetric=True`` explores with
        orbit search (``bfs_batch(symmetric=True)``) and makes a symmetric set of canonical forms."""
        P8, budgets = _batch_inputs(roots, max_nodes_to_explore)
        if P8.shape[0] == 0:
            raise ValueError("explore needs at least one root")
        L = _lib.lib()
        dev = _lib.default_device() if device is None else device
        e = _BatchEngine(L, dev, P8, budgets, cyclically_reduce_after_moves, chunk_parents, None, False, symmetric)
        try:
            results = e.run(False)
            h = C.c_void_p()
            _lib.check(L.acs_goalset_from_bfs_batch(e.h, C.byref(h)))
        finally:
            e.destroy()
        return cls(h, P8.shape[1] // 2, cyclically_reduce_after_moves, dev, results)

    @property
    def closed(self):
        return not self.handle

    def _size(self):
        if self.closed:
            raise ValueError("the goal set is closed")
        n, s, b = C.c_int64(0), C.c_int64(0), C.c_int64(0)
        _lib.check(_lib.lib().acs_goalset_size(self.handle, C.byref(n), C.byref(s), C.byref(b)))
        return n.value, s.value, b.value

    @property
    def n_entries(self):
        return self._size()[0]

    @property
    def n_states(self):
        """Distinct states among the entries."""
        return self._size()[1]

    @property
    def nbytes(self):
        """Device bytes the set holds."""
        return self._size()[2]

    def path(self, entry):
        """-> (root, path): the entry's root index and ``[(-1, L_root), (action, total_length), ...]`` from the
        root's state to the entry's state -- in a symmetric set, moves of the root row to the state
        ``frame(entry)``.(stored state)."""
        return self._path(entry)[:2]

    def frame(self, entry):
        """The element H with (end state of ``path(entry)``) = H.(the entry's stored state); 0 in an exact set."""
        return self._path(entry)[2]

    def _path(self, entry):
        if self.closed:
            raise ValueError("the goal set is closed")
        L = _lib.lib()
        root, n, fr = C.c_int(0), C.c_int(0), C.c_int(0)
        cap = 256
        buf = np.zeros((cap, 2), np.int32)
        rc = L.acs_goalset_path_frame(self.handle, int(entry), C.byref(root), buf.ctypes.data, cap, C.byref(n),
                                      C.byref(fr))
        if rc == _lib.ACS_ERR_INVALID and n.value > cap:
            cap = n.value
            buf = np.zeros((cap, 2), np.int32)
            rc = L.acs_goalset_path_frame(self.handle, int(entry), C.byref(root), buf.ctypes.data, cap, C.byref(n),
                                          C.byref(fr))
        _lib.check(rc)
        return int(root.value), [(int(a), int(l)) for a, l in buf[: n.value]], int(fr.value)

    def close(self):
        if self.handle:
            _lib.lib().acs_goalset_destroy(self.handle)
            self.handle = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def trivial_ball(max_relator_length, max_nodes_to_explore, cyclically_reduce_after_moves=False, device=None,
                 chunk_parents=0, symmetric=False):
    """``GoalSet.explore`` from the eight trivial presentations (<x^+-1, y^+-1> and <y^+-1, x^+-1>), each with
    ``max_nodes_to_explore`` nodes: a ball of states from which a path to a trivial presentation is known.
    ``symmetric=True``: one orbit search from <x, y> (the eight form one orbit) with ``max_nodes_to_explore``
    nodes, each entry standing for every image of its state."""
    roots = generate_trivial_states(max_relator_length)
    if symmetric:
        mrl = max_relator_length
        roots = np.zeros((1, 2 * mrl), np.int8)
        roots[0, 0], roots[0, mrl] = 1, 2
    return GoalSet.explore(roots, max_nodes_to_explore, cyclically_reduce_after_moves, device, chunk_parents,
                           symmetric)


def _stitch_through_ball(results, ball):
    """Meet-in-the-middle paths: every row that stopped at a ball entry gets its forward path followed by
    the entry's ball path walked backwards, each move replaced by its inverse -> ``(trivialized, path,
    info)`` with ``info["ball_root"]`` and ``info["ball_path"]``.  Other rows are kept as they are."""
    out = []
    for solved, path, info in results:
        if not solved or info["goal"] is None:
            out.append((solved, path, info))
            continue
        root, bpath, frame = ball._path(info["goal"])
        # forward end s_f = u^-1.c_e, ball path end b_e = H_e.c_e: k = u^-1.H_e^-1 maps b_e to s_f and the ball
        # path from its root t onto a path from the trivial k.t to s_f, move m becoming PI[k][m]
        k = sym_mul(sym_inv(info["goal_element"]), sym_inv(frame))
        back = [(INVERSE_MOVE[PI[k][bpath[j][0]]], bpath[j - 1][1]) for j in range(len(bpath) - 1, 0, -1)]
        info["ball_root"], info["ball_path"] = root, bpath
        full = path + back
        out.append((full[-1][1] == 2, full, info))
    return out


def _check_ball(ball, name, search):
    if ball.cyclical:
        raise ValueError(f"{name} needs a ball built with cyclically_reduce_after_moves=False: with "
                         f"cyclic reduction the ball path cannot be walked backwards; use {search}(goals=...) and "
                         "GoalSet.path")


def bfs_meet_in_the_middle(presentations, max_nodes_to_explore, ball, device=None, chunk_parents=0,
                           max_bytes=DEFAULT_MAX_BYTES, symmetric=False):
    """Meet-in-the-middle breadth-first search, without cyclic reduction: ``bfs_batch`` of every row with
    ``ball`` (usually ``trivial_ball(...)``) as its goal set.

    Returns a list of ``(trivialized, path|None, info)``.  ``path`` is in the reference's format and ends at
    total length 2: a row solved directly keeps its ``bfs`` path; a row that reached the ball gets its
    forward path followed by the ball path from the ball's root to the meeting state, walked backwards
    with every move replaced by its inverse (``INVERSE_MOVE``).  Then ``info["goal"]`` is the entry met,
    ``info["ball_root"]`` and ``info["ball_path"]`` its root and path in the ball.

    Only for ``cyclically_reduce_after_moves=False``: with cyclic reduction a move is not undone by a
    single move, so no such path exists.  There, ``bfs_batch(..., goals=ball)`` gives the forward path and
    ``ball.path(info["goal"])`` the ball path, which together certify the meeting.

    ``ball`` may be symmetric (``trivial_ball(..., symmetric=True)``): the ball path is then mapped onto the
    forward end state by the symmetry ``goal_element^-1 . ball.frame(entry)^-1`` before it is walked back.
    ``symmetric=True`` runs the forward search as an orbit search (needs a symmetric ball)."""
    _check_ball(ball, "bfs_meet_in_the_middle", "bfs_batch")
    res = bfs_batch(presentations, max_nodes_to_explore, False, device=device, chunk_parents=chunk_parents,
                    max_bytes=max_bytes, goals=ball, symmetric=symmetric)
    return _stitch_through_ball(res, ball)


def greedy_meet_in_the_middle(presentations, max_nodes_to_explore, ball, device=None):
    """Meet-in-the-middle greedy search, without cyclic reduction: ``greedy_search_batch`` of every row
    with ``ball`` (usually ``trivial_ball(...)``) as its goal set.

    Returns a list of ``(trivialized, path, info)``, stitched as in ``bfs_meet_in_the_middle``: a row
    solved directly keeps its greedy path, a row that reached the ball gets its forward path followed by
    the reversed ball path, and a row that did neither keeps greedy's failure path.  Every row plain
    greedy search solves is trivialized: a search with goals follows the plain search until its first
    goal, and every ball state has a path to a trivial presentation."""
    from .greedy import greedy_search_batch

    _check_ball(ball, "greedy_meet_in_the_middle", "greedy_search_batch")
    res = greedy_search_batch(presentations, max_nodes_to_explore, False, device=device, goals=ball)
    return _stitch_through_ball(res, ball)
