"""CPU model of the bucket kernel's capacity bookkeeping (test infrastructure).

``greedy_bucket_kernel`` (ac_solver_b200/csrc/greedy_bucket.cuh) is bit-exact with the reference's greedy
loop, so which nodes it expands, and in which rounds and tiles, follows from the reference's pop order.
What the reference does not have are the kernel's fixed capacities: the bucket directory, the segment pool,
the segments per bucket, the sort buffer and the frontier array.  ``bucket_pass`` replays the reference's
search (the loop of ``greedy_goal_oracle.greedy_goals``, moves from the pinned C oracle) grouped the way the
kernel groups it, and does the kernel's bookkeeping literally:

- a round pops the minimal (length, depth) bucket: more than ``max_seg`` segments is reason 1, more than
  ``sort_cap`` nodes reason 2 (tested second, so it wins when both hold);
- the bucket's nodes, in state order, are expanded in tiles of ``tile`` nodes; a tile stops at a solving,
  raising or goal child, at the node after which the budget is reached, and after the first node that
  produced a new child shorter than the bucket (the run is interrupted);
- after each tile, the committed children of each length L (ascending) make one segment of bucket
  (L, depth + 1): a full segment pool is reason 3, a full frontier (2 * (budget + 16) entries) reason 4, a
  depth of 2^24 reason 6, and a new bucket in a full directory reason 5;
- the unexpanded rest of an interrupted bucket goes back as one segment under the same key, with the
  checks of reasons 3, 4 and 5 in that order.

A hand-back at a pop reports the nodes committed before it; one in a directory update reports the nodes
committed before that tile.  ``tiers`` chains the passes the way ``greedy_run_impl`` does.
"""

from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from oracle import oracle as O


@dataclass(frozen=True)
class Caps:
    tile: int = 1024
    small: int = 256
    buckets1: int = 2048
    buckets2: int = 12288
    max_seg: int = 512
    seg_pool: int = 1 << 16
    sort_cap: int = 1 << 16


def bucket_pass(presentation, budget, cyclical=False, goals=None, caps=Caps(), max_buckets=None, stats=None):
    """One launch of the bucket kernel with a directory of ``max_buckets`` entries.

    -> ("done", rounds, n_visited) when the search finishes in this pass, or ("handback", reason, n_nodes).
    ``stats`` (a dict) receives the largest bucket popped, the number of rests put back and every node's depth."""
    p = np.ascontiguousarray(presentation, dtype=np.int8)
    max_buckets = caps.buckets1 if max_buckets is None else max_buckets
    L0 = int(np.count_nonzero(p))
    if goals is not None and p.tobytes() in goals:
        return ("done", 0, 1)
    states, tuples = [p], [tuple(int(x) for x in p)]
    index = {p.tobytes()}
    fcap = 2 * (int(budget) + 16)
    # directory: (length, depth) -> [segments, node ids]
    dirs = {(L0, 0): [1, [0]]}
    seg_used, f_end, rounds = 1, 1, 0
    depth = [0]
    if stats is not None:
        stats.update(max_bucket=1, rests=0, depth=depth)
    while dirs:
        key = min(dirs)
        nseg, nodes = dirs.pop(key)
        if nseg > caps.max_seg or len(nodes) > caps.sort_cap:
            return ("handback", 2 if len(nodes) > caps.sort_cap else 1, len(states))
        rounds += 1
        Lcur, dcur = key
        if stats is not None:
            stats["max_bucket"] = max(stats["max_bucket"], len(nodes))
        nodes = sorted(nodes, key=lambda i: tuples[i])
        done, stop = 0, None
        for tile0 in range(0, len(nodes), caps.tile):
            n_before = len(states)
            by_len = {}
            for i in nodes[tile0 : tile0 + caps.tile]:
                done += 1
                out, lens, status = O.moves_batch(np.repeat(states[i][None, :], 12, axis=0),
                                                  np.arange(12, dtype=np.uint8), cyclical=cyclical)
                shorter = False
                for a in range(12):
                    if status[a]:
                        stop = "error"
                        break
                    nl = int(lens[a].astype(np.int64).sum())
                    if nl == 2:
                        stop = "solved"
                        break
                    k = out[a].tobytes()
                    if goals is not None and k in goals:
                        stop = "goal"
                        break
                    if k not in index:
                        index.add(k)
                        states.append(out[a].copy())
                        tuples.append(tuple(int(x) for x in out[a]))
                        depth.append(dcur + 1)
                        by_len.setdefault(nl, []).append(len(states) - 1)
                        shorter |= nl < Lcur
                if stop is None and len(states) >= budget:
                    stop = "budget"
                elif stop is None and shorter:
                    stop = "interrupt"
                if stop is not None:
                    break
            for L in sorted(by_len):
                cnt = len(by_len[L])
                if seg_used >= caps.seg_pool or f_end + cnt > fcap or dcur + 1 >= 1 << 24:
                    return ("handback", 3 if seg_used >= caps.seg_pool else (4 if f_end + cnt > fcap else 6), n_before)
                seg_used += 1
                f_end += cnt
                nk = (L, dcur + 1)
                if nk in dirs:
                    dirs[nk][0] += 1
                    dirs[nk][1].extend(by_len[L])
                else:
                    if len(dirs) >= max_buckets:
                        return ("handback", 5, n_before)
                    dirs[nk] = [1, list(by_len[L])]
            if stop is not None:
                break
        if stop in ("solved", "error", "goal", "budget"):
            return ("done", rounds, len(states))
        rest = len(nodes) - done
        if rest:
            if seg_used >= caps.seg_pool or f_end + rest > fcap or len(dirs) >= max_buckets:
                return ("handback", 3 if seg_used >= caps.seg_pool else (4 if f_end + rest > fcap else 5), len(states))
            seg_used += 1
            f_end += rest
            dirs[key] = [1, nodes[done:]]
            if stats is not None:
                stats["rests"] += 1
    return ("done", rounds, len(states))


def tiers(presentation, budget, cyclical=False, goals=None, caps=Caps()):
    """The two bucket passes of ``greedy_run_impl``.

    -> (hand-backs, rounds): hand-backs is the list of (pass, reason, n_nodes) the engine reports, and rounds
    the bucket rounds of the pass that finished the search, or None when the heap kernel re-runs it."""
    handbacks = []
    for pass_, mb in enumerate((caps.buckets1, caps.buckets2)):
        r = bucket_pass(presentation, budget, cyclical, goals, caps, mb)
        if r[0] == "done":
            return handbacks, r[1]
        handbacks.append((pass_, r[1], r[2]))
    return handbacks, None
