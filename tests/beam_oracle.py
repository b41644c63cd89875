"""CPU statement of batched beam search (test infrastructure): the contract of csrc/beam.cu written
literally on int8 rows, with moves from the pinned C oracle (``oracle.moves_batch``, one call per level).

One search from a row with beam width W, node budget N, optional depth limit D, cyclic flag and optional
goal set (a dict {state bytes: entry} from ``goal_oracle.goal_dict``, or ``sym_oracle.SymGoals``):
  * V = [root], the level-0 beam is [root]; a root in the goal set is a hit at depth 0;
  * level d: candidate c = 12*i + m is move m applied to beam node i.  Walking c upwards, the first
    candidate that raises, has total length 2 or is in the goal set ends the search (a solve wins over a
    goal on the same child) and nothing of the level is committed;
  * otherwise the candidates whose state is not in V, each at its smallest c, are ordered by
    (total length, c); the first min(W, N - |V|) become the next beam and are appended to V in that order;
  * the search stops after a level whose next beam is empty, when |V| >= N (budget_hit), or at d + 1 = D.
"""

from __future__ import annotations

import numpy as np

from oracle import oracle as O


def beam_search(presentation, beam_width, max_nodes_to_explore, max_depth=None, cyclically_reduce_after_moves=False,
                goals=None, want_visited=False, want_levels=False):
    """-> (solved, path|None, info), ``info`` as ``beam_search_batch`` reports it.  ``want_levels`` adds
    ``info["beams"]``: the beams of every level, as lists of indices into V."""
    p = np.ascontiguousarray(presentation, dtype=np.int8)
    mrl = p.size // 2
    cyc = bool(cyclically_reduce_after_moves)
    W, N = int(beam_width), int(max_nodes_to_explore)
    info = {"n_visited": 0, "n_expanded": 0, "n_moves": 0, "frontier_left": 0, "budget_hit": False, "levels": 0,
            "status": 0, "minlen_log": []}
    if goals is not None:
        info["goal"] = None
    l0, l1 = int(np.count_nonzero(p[:mrl])), int(np.count_nonzero(p[mrl:]))
    if l0 == 0 or l1 == 0 or p[l0:mrl].any() or p[mrl + l1:].any():  # is_array_valid_presentation
        info["status"] = O.ACO_ASSERT
        return False, None, info
    states, parent, action, length = [p.copy()], [-1], [-1], [l0 + l1]
    index = {p.tobytes(): 0}
    beam = [0]
    beams = [beam]
    min_length = l0 + l1
    hit = None  # (parent node, action, total length) of the child that ended the search

    def finish(solved):
        info["n_visited"] = len(states)
        info["frontier_left"] = len(states) - info["n_expanded"]
        if want_visited:
            info["visited"] = np.array(states, np.int8).reshape(len(states), 2 * mrl)
        if want_levels:
            info["beams"] = beams
        if not solved:
            return False, None, info
        chain = []
        node = hit[0] if hit else 0
        while node >= 0:
            chain.append((action[node], length[node]))
            node = parent[node]
        path = chain[::-1]
        if hit:
            path.append((hit[1], hit[2]))
        return True, path, info

    if goals is not None and p.tobytes() in goals:
        info["goal"] = goals[p.tobytes()]
        return finish(True)
    while True:
        parents = np.repeat(np.array([states[i] for i in beam], np.int8), 12, axis=0)
        acts = np.tile(np.arange(12, dtype=np.uint8), len(beam))
        out, lens, status = O.moves_batch(parents, acts, cyclical=cyc)
        tot = lens.astype(np.int64).sum(axis=1)
        new = {}  # state bytes -> smallest c
        for c in range(12 * len(beam)):
            info["n_moves"] += 1
            if status[c]:
                info["status"] = int(status[c])
                info["n_expanded"] += c // 12 + 1
                return finish(False)
            nl = int(tot[c])
            if nl < min_length:
                min_length = nl
                info["minlen_log"].append(nl)
            key = out[c].tobytes()
            if nl == 2 or (goals is not None and key in goals):
                if nl != 2:
                    info["goal"] = goals[key]
                info["n_expanded"] += c // 12 + 1
                hit = (beam[c // 12], c % 12, nl)
                return finish(True)
            if key not in index and key not in new:
                new[key] = c
        info["n_expanded"] += len(beam)
        order = sorted(new.values(), key=lambda c: (int(tot[c]), c))
        take = order[: max(0, min(W, N - len(states)))]
        beam = []
        for c in take:
            index[out[c].tobytes()] = len(states)
            beam.append(len(states))
            states.append(out[c].copy())
            parent.append(beams[-1][c // 12])
            action.append(c % 12)
            length.append(int(tot[c]))
        beams.append(beam)
        info["levels"] += 1
        if len(states) >= N:
            info["budget_hit"] = True
        if not beam or info["budget_hit"] or (max_depth is not None and info["levels"] >= max_depth):
            return finish(False)
