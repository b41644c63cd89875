"""CPU restatement of greedy search with a goal set (test infrastructure).

``greedy_goals`` is the reference's ``greedy_search`` (ac_solver/search/greedy.py:15-121, restated in C as
``oracle/ac_oracle.c:aco_greedy``) with the goal test of ``goal_oracle.bfs_goals`` applied literally to
every child.  Moves come from the pinned C oracle.  With ``goals=None`` it returns what
``oracle.greedy_search`` returns, which tests/test_greedy_goals_cpu.py checks on the reference fixtures.
Goal sets are the dicts of ``goal_oracle.goal_dict``.
"""

from __future__ import annotations

import numpy as np

from oracle import oracle as O


def greedy_goals(presentation, max_nodes_to_explore, cyclically_reduce_after_moves=False, goals=None,
                 want_visited=False):
    """The reference's greedy loop (ac_solver/search/greedy.py:15-121, restated in C as
    ``oracle/ac_oracle.c:aco_greedy``) on a ``heapq`` of (total length, depth, state tuple), with the goal
    test applied literally to every child: after the minimal-length update and the length-2 test, before
    the visited test.  A root in ``goals`` is a hit before anything is expanded.

    -> (solved, path, info) like ``oracle.greedy_search`` (the failure path is the last expanded node's
    path + [(11, length of its 12th child)]); a raising move ends the search with ``info["status"]`` set
    and an empty path.  ``goals``: a dict {state bytes: entry index}, or None.  ``info["goal"]`` is the
    entry hit, or None."""
    import heapq

    p = np.ascontiguousarray(presentation, dtype=np.int8)
    mrl = p.size // 2
    cyc = bool(cyclically_reduce_after_moves)
    L0 = int(np.count_nonzero(p))
    states, parent, action, length, depth = [p.copy()], [-1], [-1], [L0], [0]
    index = {p.tobytes(): 0}
    heap = [(L0, 0, tuple(int(x) for x in p), 0)]
    info = {"n_visited": 0, "n_expanded": 0, "n_moves": 0, "frontier_left": 0, "budget_hit": False,
            "minlen_log": [], "status": 0, "goal": None}
    min_length = L0
    cur, last = 0, (11, L0)  # the final pair of the path: (action, length)

    def finish(solved, node, final):
        info["n_visited"] = len(states)
        info["frontier_left"] = len(heap)
        if want_visited:
            info["visited"] = np.array(states, np.int8).reshape(len(states), 2 * mrl)
        if info["status"]:
            return False, [], info
        chain = []
        while node >= 0:
            chain.append((action[node], length[node]))
            node = parent[node]
        return solved, chain[::-1] + ([final] if final else []), info

    if goals is not None and p.tobytes() in goals:  # the root is a goal: a hit at depth 0
        info["goal"] = goals[p.tobytes()]
        return finish(True, 0, None)
    while heap:
        cur = heapq.heappop(heap)[3]
        info["n_expanded"] += 1
        out, lens, status = O.moves_batch(np.repeat(states[cur][None, :], 12, axis=0), np.arange(12, dtype=np.uint8),
                                          cyclical=cyc)
        for a in range(12):
            info["n_moves"] += 1
            if status[a]:
                info["status"] = int(status[a])
                return finish(False, cur, None)
            nl = int(lens[a].astype(np.int64).sum())
            last = (a, nl)
            if nl < min_length:
                min_length = nl
                info["minlen_log"].append(nl)
            if nl == 2:
                return finish(True, cur, (a, nl))
            key = out[a].tobytes()
            if goals is not None and key in goals:
                info["goal"] = goals[key]
                return finish(True, cur, (a, nl))
            if key not in index:
                k = len(states)
                index[key] = k
                states.append(out[a].copy())
                parent.append(cur)
                action.append(a)
                length.append(nl)
                depth.append(depth[cur] + 1)
                heapq.heappush(heap, (nl, depth[k], tuple(int(x) for x in out[a]), k))
        if len(states) >= max_nodes_to_explore:  # only after all 12 children
            info["budget_hit"] = True
            break
    return finish(False, cur, last)
