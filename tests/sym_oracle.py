"""The presentation symmetry group G on int8 rows, and breadth-first search over its orbits (test
infrastructure).  Written plainly from the definitions, independently of the bit tricks of
``csrc/ac_sym.cuh``.

G has order 16.  An element g = (r, s, a, b) has index 8r + 4s + 2a + b and acts on a state by
  s: swap x <-> y,  then  a: invert x,  then  b: invert y  (on every letter),  then  r: swap the relators.
It maps the 12 AC' moves to themselves: acmove(PI[g][m], g.state) = g.acmove(m, state).

``canonical`` picks the smallest image under the order of ``order_key``: (len r0, r0 read from its last
letter to its first, len r1, r1 likewise), letters compared by their 2-bit codes y=0, x=1, y^-1=2, x^-1=3.
Among elements giving that image the smallest index is returned.

``orbit_bfs`` is ``goal_oracle.bfs_goals`` (no goals) run on canonical states: the root is stored as its
canonical form, a child is new when its canonical form is unseen and is stored canonical.  Its path is in
actual moves from the input row (``actual_path``).
"""

from __future__ import annotations

import numpy as np

from oracle import oracle as O

ELEMENTS = [(g >> 3 & 1, g >> 2 & 1, g >> 1 & 1, g & 1) for g in range(16)]  # (r, s, a, b)

# move m on a state <-> move PI[g][m] on g.state (the table of the issue that introduced the group,
# checked against the C oracle by tests/test_symmetry_cpu.py)
PI = [
    [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11],
    [0, 1, 2, 3, 4, 9, 10, 7, 8, 5, 6, 11],
    [0, 1, 2, 3, 8, 5, 6, 11, 4, 9, 10, 7],
    [0, 1, 2, 3, 8, 9, 10, 11, 4, 5, 6, 7],
    [0, 1, 2, 3, 6, 11, 4, 9, 10, 7, 8, 5],
    [0, 1, 2, 3, 10, 11, 4, 5, 6, 7, 8, 9],
    [0, 1, 2, 3, 6, 7, 8, 9, 10, 11, 4, 5],
    [0, 1, 2, 3, 10, 7, 8, 5, 6, 11, 4, 9],
    [3, 2, 1, 0, 11, 6, 5, 8, 7, 10, 9, 4],
    [3, 2, 1, 0, 11, 10, 9, 8, 7, 6, 5, 4],
    [3, 2, 1, 0, 7, 6, 5, 4, 11, 10, 9, 8],
    [3, 2, 1, 0, 7, 10, 9, 4, 11, 6, 5, 8],
    [3, 2, 1, 0, 5, 4, 11, 10, 9, 8, 7, 6],
    [3, 2, 1, 0, 9, 4, 11, 6, 5, 8, 7, 10],
    [3, 2, 1, 0, 5, 8, 7, 10, 9, 4, 11, 6],
    [3, 2, 1, 0, 9, 8, 7, 6, 5, 4, 11, 10],
]


def letter_map(g, v):
    """Image of one letter (in {+-1, +-2}) under g."""
    _, s, a, b = ELEMENTS[g]
    if s:
        v = (3 - abs(v)) * (1 if v > 0 else -1)
    if a and abs(v) == 1:
        v = -v
    if b and abs(v) == 2:
        v = -v
    return v


def act(g, rows):
    """g.rows for int8 rows [..., 2*mrl] of letters (0 = padding)."""
    rows = np.asarray(rows)
    mrl = rows.shape[-1] // 2
    lut = np.array([letter_map(g, v) if v else 0 for v in range(-2, 3)], np.int8)
    out = lut[rows.astype(np.int64) + 2]
    if ELEMENTS[g][0]:
        out = np.concatenate([out[..., mrl:], out[..., :mrl]], axis=-1)
    return out


def _letter_images(g):
    return tuple(letter_map(g, v) for v in (1, -1, 2, -2))


def compose(g, h):
    """The element k with k.state = g.(h.state)."""
    want = tuple(letter_map(g, letter_map(h, v)) for v in (1, -1, 2, -2))
    r = ELEMENTS[g][0] ^ ELEMENTS[h][0]
    (k,) = [k for k in range(16) if ELEMENTS[k][0] == r and _letter_images(k) == want]
    return k


MUL = [[compose(g, h) for h in range(16)] for g in range(16)]
INV = [next(h for h in range(16) if MUL[g][h] == 0) for g in range(16)]


def code(v):
    return {2: 0, 1: 1, -2: 2, -1: 3}[int(v)]


def order_key(row):
    row = np.asarray(row)
    mrl = row.size // 2
    key = []
    for half in (row[:mrl], row[mrl:]):
        w = [int(v) for v in half if v]
        key.append(len(w))
        key.extend(code(v) for v in reversed(w))
    return tuple(key)


def canonical(row):
    """-> (the smallest image of row, the smallest g producing it)."""
    best, best_g = None, None
    for g in range(16):
        im = act(g, row)
        k = order_key(im)
        if best is None or k < best[0]:
            best, best_g = (k, im), g
    return best[1], best_g


_CODE = np.array([2, 3, 0, 1, 0], np.uint8)  # code of letter v at index v + 2 (-2, -1, 0, 1, 2); padding 0


def canonical_batch(rows):
    """``canonical`` of every row of int8 rows [n, 2*mrl] -> (rows, elements), by comparing the byte
    strings of ``order_key`` (faster for the search oracle; tests/test_symmetry_cpu.py checks it equals
    ``canonical``)."""
    X = np.ascontiguousarray(rows, dtype=np.int8)
    n, w = X.shape
    mrl = w // 2
    keys = []
    for g in range(16):
        im = act(g, X)
        parts = []
        for half in (im[:, :mrl], im[:, mrl:]):
            length = np.count_nonzero(half, axis=1)
            idx = length[:, None] - 1 - np.arange(mrl)[None, :]  # last letter first; padding after
            rev = np.take_along_axis(half, np.clip(idx, 0, mrl - 1), axis=1)
            codes = np.where(idx >= 0, _CODE[rev.astype(np.int64) + 2], 0).astype(np.uint8)
            parts += [length.astype(np.uint8)[:, None], codes]
        keys.append((np.concatenate(parts, axis=1), im))
    out = np.empty_like(X)
    elem = np.zeros(n, np.int64)
    for i in range(n):
        g = min(range(16), key=lambda g: (keys[g][0][i].tobytes(), g))
        out[i], elem[i] = keys[g][1][i], g
    return out, elem


def actual_path(frames):
    """Canonical-frame path -> actual moves from the input row.  ``frames`` is the root's
    (g0, L0) followed by one (m_k, g_{k+1}, L_{k+1}) per edge: move m_k applied to the stored state c_k
    produced a child whose canonical form c_{k+1} = g_{k+1}.child.  The last edge may have g = None (a
    child that was not stored, such as the solving one).  Returns [(-1, L0), (action, total length), ...]."""
    g0, l0 = frames[0]
    h = INV[g0]  # actual state a_k = h_k . c_k
    path = [(-1, l0)]
    for m, g, length in frames[1:]:
        path.append((PI[h][m], length))
        if g is not None:
            h = MUL[h][INV[g]]
    return path


class SymGoals:
    """A symmetric goal set for the search oracles: ``key in goals`` and ``goals[key]`` look up the canonical
    form of the state whose bytes are ``key`` in ``{canonical state bytes: entry}``."""

    def __init__(self, entries):
        self.d = entries

    def _c(self, key):
        return canonical(np.frombuffer(key, np.int8))[0].tobytes()

    def __contains__(self, key):
        return self._c(key) in self.d

    def __getitem__(self, key):
        return self.d[self._c(key)]


def orbit_bfs(presentation, max_nodes_to_explore, cyclically_reduce_after_moves=False, want_visited=False,
              goals=None, stop_at_trivial=True):
    """-> (solved, path|None, info) like ``goal_oracle.bfs_goals``; ``info["visited"]`` holds the canonical
    states in insertion order.  ``goals`` (a ``SymGoals``) is tested on every child after the length-2 test,
    and on the root first; ``info["goal"]`` is the entry hit."""
    p = np.ascontiguousarray(presentation, dtype=np.int8)
    mrl = p.size // 2
    cyc = bool(cyclically_reduce_after_moves)
    info = {"n_visited": 0, "n_expanded": 0, "n_moves": 0, "frontier_left": 0, "budget_hit": False,
            "minlen_log": [], "status": 0, "goal": None}
    l0, l1 = int(np.count_nonzero(p[:mrl])), int(np.count_nonzero(p[mrl:]))
    if l0 == 0 or l1 == 0 or p[l0:mrl].any() or p[mrl + l1:].any():
        info["status"] = O.ACO_ASSERT
        return False, None, info
    c0, g0 = canonical(p)
    states = [c0]
    index = {c0.tobytes(): 0}
    parent, action, length, elem = [-1], [-1], [l0 + l1], [g0]
    min_length = l0 + l1
    head = 0
    solved, hit_from = False, None

    def finish():
        info["n_visited"] = len(states)
        info["frontier_left"] = len(states) - head
        if want_visited:
            info["visited"] = np.array(states, np.int8).reshape(len(states), 2 * mrl)
        if not solved:
            return False, None, info
        chain = []
        node = hit_from[0]
        while node >= 0:
            chain.append(node)
            node = parent[node]
        chain = chain[::-1]
        frames = [(elem[0], length[0])] + [(action[n], elem[n], length[n]) for n in chain[1:]]
        if hit_from[1] is not None:
            frames.append((hit_from[1], None, hit_from[2]))
        return True, actual_path(frames), info

    if goals is not None and c0.tobytes() in goals:
        solved, hit_from = True, (0, None, None)
        info["goal"] = goals[c0.tobytes()]
        return finish()

    while head < len(states):
        lo, hi = head, len(states)
        parents = np.repeat(np.array(states[lo:hi], np.int8), 12, axis=0)
        acts = np.tile(np.arange(12, dtype=np.uint8), hi - lo)
        out, lens, status = O.moves_batch(parents, acts, cyclical=cyc)
        tot = lens.astype(np.int64).sum(axis=1)
        canon, elems = canonical_batch(np.where(status[:, None] == 0, out, parents))
        for cur in range(lo, hi):
            head = cur + 1
            info["n_expanded"] += 1
            for a in range(12):
                r = (cur - lo) * 12 + a
                info["n_moves"] += 1
                if status[r]:
                    info["status"] = int(status[r])
                    return finish()
                nl = int(tot[r])
                if nl < min_length:
                    min_length = nl
                    info["minlen_log"].append(nl)
                if nl == 2 and stop_at_trivial:
                    solved, hit_from = True, (cur, a, nl)
                    return finish()
                c, g = canon[r], int(elems[r])
                key = c.tobytes()
                if goals is not None and key in goals:
                    solved, hit_from = True, (cur, a, nl)
                    info["goal"] = goals[key]
                    return finish()
                if key not in index:
                    index[key] = len(states)
                    states.append(c)
                    parent.append(cur)
                    action.append(a)
                    length.append(nl)
                    elem.append(g)
            if len(states) >= max_nodes_to_explore:
                info["budget_hit"] = True
                return finish()
    return finish()


def replay(row, path, cyclical):
    """Total length after applying the path's actions (all but the first pair) to row with the C oracle;
    asserts every step's total length matches the path."""
    s = np.ascontiguousarray(row, dtype=np.int8)
    mrl = s.size // 2
    assert path[0] == (-1, int(np.count_nonzero(s)))
    for a, length in path[1:]:
        s, lens = O.acmove(a, s, mrl, cyclical=cyclical)
        assert int(np.sum(lens)) == length, (a, length, lens)
    return int(np.count_nonzero(s))
