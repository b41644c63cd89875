"""CPU restatement of breadth-first search with a goal set (test infrastructure).

``bfs_goals`` is the reference's ``bfs`` (ac_solver/search/breadth_first.py:15-97, restated in C as
``oracle/ac_oracle.c:aco_bfs``) with two changes:
  * the goal test: a generated child that is in ``goals`` ends the search with a hit.  It runs after
    the minimal-length update and the length-2 test, before the visited test, on every child,
    visited or not.  A root in ``goals`` is a hit before anything is expanded;
  * ``stop_at_trivial=False`` turns the length-2 test off.
Moves come from the pinned C oracle (``oracle.moves_batch``, one call per batch of parents); the
search order is the reference's.  With ``goals=None`` and ``stop_at_trivial=True`` it returns what
``oracle.bfs`` returns, which tests/test_goal_search_cpu.py checks on the reference fixtures.
"""

from __future__ import annotations

import numpy as np

from oracle import oracle as O


def bfs_goals(presentation, max_nodes_to_explore, cyclically_reduce_after_moves=False, goals=None,
              stop_at_trivial=True, want_visited=False):
    """-> (solved, path|None, info).  ``goals``: a dict {state bytes: entry index} (int8 rows of
    2*mrl letters), or None.  ``info["goal"]`` is the entry hit, or None."""
    p = np.ascontiguousarray(presentation, dtype=np.int8)
    mrl = p.size // 2
    cyc = bool(cyclically_reduce_after_moves)
    info = {"n_visited": 0, "n_expanded": 0, "n_moves": 0, "frontier_left": 0, "budget_hit": False,
            "minlen_log": [], "status": 0, "goal": None}
    l0, l1 = int(np.count_nonzero(p[:mrl])), int(np.count_nonzero(p[mrl:]))
    if l0 == 0 or l1 == 0 or p[l0:mrl].any() or p[mrl + l1:].any():  # breadth_first.py:36-38
        info["status"] = O.ACO_ASSERT
        return False, None, info
    states = [p.copy()]
    index = {p.tobytes(): 0}
    parent, action, length = [-1], [-1], [l0 + l1]
    min_length = l0 + l1
    head = 0
    solved, hit_from = False, None  # hit_from: (node, action, total length) of the ending child

    def finish():
        info["n_visited"] = len(states)
        info["frontier_left"] = len(states) - head
        if want_visited:
            info["visited"] = np.array(states, np.int8).reshape(len(states), 2 * mrl)
        if not solved:
            return False, None, info
        chain = []
        node = hit_from[0] if hit_from else 0
        while node >= 0:
            chain.append((action[node], length[node]))
            node = parent[node]
        path = chain[::-1]
        if hit_from:
            path.append((hit_from[1], hit_from[2]))
        return True, path, info

    if goals is not None and p.tobytes() in goals:  # the root is a goal: a hit at depth 0
        solved = True
        info["goal"] = goals[p.tobytes()]
        return finish()
    while head < len(states):
        lo, hi = head, len(states)
        parents = np.repeat(np.array(states[lo:hi], np.int8), 12, axis=0)
        acts = np.tile(np.arange(12, dtype=np.uint8), hi - lo)
        out, lens, status = O.moves_batch(parents, acts, cyclical=cyc)
        tot = lens.astype(np.int64).sum(axis=1)
        for cur in range(lo, hi):
            head = cur + 1  # popleft
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
                key = out[r].tobytes()
                if goals is not None and key in goals:
                    solved, hit_from = True, (cur, a, nl)
                    info["goal"] = goals[key]
                    return finish()
                if key not in index:
                    index[key] = len(states)
                    states.append(out[r].copy())
                    parent.append(cur)
                    action.append(a)
                    length.append(nl)
            if len(states) >= max_nodes_to_explore:  # only after all 12 children
                info["budget_hit"] = True
                return finish()
    return finish()


def goal_dict(rows):
    """{state bytes: smallest row index} of int8 rows."""
    d = {}
    for i, r in enumerate(np.ascontiguousarray(rows, dtype=np.int8)):
        d.setdefault(r.tobytes(), i)
    return d
