"""Miller-Schupp presentations MS(n, w) = <x, y | x^-1 y^n x = y^(n+1), x = w> and the search
sweep over them -- the caller of BASELINE config 3, mirroring the reference's
``ac_solver/search/miller_schupp/miller_schupp.py`` (same function names, arguments, return
values and output-file formats).

What differs is where the work runs: the free + cyclic reduction of all 4^len candidate words of
one length is ONE batched call of the GPU reduction kernel (``simplify_relator`` semantics,
envs/utils.py:175-240) instead of a Python loop, and a greedy sweep runs all presentations of a
group concurrently (one warp per presentation, ``greedy_search_batch``; a BFS sweep likewise
through one batched engine, ``bfs_batch``) instead of one after the other.  The enumeration order,
the cyclic-permutation de-duplication and the file layout are the reference's, so the generated
lists are identical.
"""

from __future__ import annotations

import os
from itertools import product

import numpy as np

from ... import _lib
from ..._host import generic_call


def generate_miller_schupp_presentations(n, max_w_len):
    """miller_schupp.py:20-83.  Returns {len(w): [presentation as a list of ints, ...]}."""
    assert n >= 1 and max_w_len >= 1, f"expect n >= 1 and max_w_len >=1 ; got n = {n}, max_w_len = {max_w_len}"
    max_relator_length = 2 * max(2 * n + 3, max_w_len + 1) + 2
    relator1 = [-1] + [2] * n + [1] + [-2] * (n + 1) + [0] * (max_relator_length - 2 * n - 3)
    seen = set()
    out = {}
    for search_len in range(1, max_w_len + 1):
        words = np.array([w for w in product([1, 2, -1, -2], repeat=search_len)
                          if sum(x for x in w if abs(x) == 1) == 0], dtype=np.int8)  # zero exponent sum on x
        if len(words) == 0:
            continue
        rows = np.concatenate([np.full((len(words), 1), -1, np.int8), words], axis=1)  # x^-1 w
        reduced, lens, status = generic_call(_lib.OP_SIMPLIFY_RELATOR, rows, cyclical=True)
        assert not status.any()
        for k in range(len(words)):
            relator2 = [int(v) for v in reduced[k, : lens[k]]]
            if relator2 == [-1]:  # x^-1 w = x^-1: len(w) must be > 0
                continue
            lenw = len(relator2) - 1
            if tuple(relator2) not in seen:  # keep one representative per cyclic permutation class
                for i in range(len(relator2)):
                    seen.add(tuple(relator2[i:] + relator2[:i]))
                out.setdefault(lenw, []).append(relator1 + relator2 + [0] * (max_relator_length - len(relator2)))
    return out


def write_list_to_text_file(list, filepath):  # noqa: A002 - the reference's argument name
    """miller_schupp.py:86-92: one Python literal per line."""
    if not filepath.endswith(".txt"):
        filepath = filepath + ".txt"
    with open(filepath, "w") as f:
        for element in list:
            f.write(f"{element}\n")


def trivialize_miller_schupp_through_search(min_n, max_n, min_w_len, max_w_len, max_nodes_to_explore, search_fn,
                                            write_output_to_file=False, output_dir=None):
    """miller_schupp.py:95-177.  ``search_fn`` is this package's ``greedy_search`` or ``bfs``.
    Returns (solved_rels, unsolved_rels, solved_paths) in the reference's order."""
    assert search_fn.__name__ in ["greedy_search", "bfs"], f"expect search_fn to be greedy or bfs; got {search_fn.__name__}"
    from .._common import _raise_for
    from ..breadth_first import bfs_batch
    from ..greedy import greedy_search_batch

    rels = {n: generate_miller_schupp_presentations(n, max_w_len) for n in range(min_n, max_n + 1)}
    solved_rels, unsolved_rels, solved_paths = [], [], []
    for n in range(min_n, max_n + 1):
        for lenw in range(min_w_len, max_w_len + 1):
            print(f"Applying {search_fn.__name__} to presentations of n = {n}, lenw = {lenw}")
            group = rels[n].get(lenw, [])
            if not group:
                continue
            # all presentations of the group in one device run; output and errors in row order, as the reference's loop
            batch = greedy_search_batch if search_fn.__name__ == "greedy_search" else bfs_batch
            results = []
            for s_, p_, info in batch(np.array(group, dtype=np.int8), max_nodes_to_explore, False):
                _raise_for(info["status"])  # the reference raises where a move empties a relator
                if not s_ and info["budget_hit"]:  # greedy.py:116-118 / breadth_first.py print this per presentation
                    print(f"Exiting search as number of explored nodes = {info['n_visited']} has exceeded the limit "
                          f"{max_nodes_to_explore}")
                results.append((s_, p_))
            for pres, (solved, path) in zip(group, results):
                if solved:
                    solved_rels.append(pres)
                    solved_paths.append(path)
                else:
                    unsolved_rels.append(pres)
    if write_output_to_file:
        dirname = output_dir or os.path.join(os.path.dirname(os.path.realpath(__file__)), "data")
        os.makedirs(dirname, exist_ok=True)
        base = f"n-{min_n}-to-{max_n}_lenw-{min_w_len}-to-{max_w_len}-max-nodes-{max_nodes_to_explore}-{search_fn.__name__}"
        fb = os.path.join(dirname, base)
        write_list_to_text_file(list=solved_rels, filepath=fb + "_solved")
        write_list_to_text_file(list=unsolved_rels, filepath=fb + "_unsolved")
        write_list_to_text_file(list=solved_paths, filepath=fb + "_paths")
        print(f"saved output in {dirname} with filenames:\n  {base}_solved\n  {base}_unsolved\n  {base}_paths")
    return solved_rels, unsolved_rels, solved_paths


def load_presentations_from_text_file(path):
    """One Python list literal per line (the format of the reference's data/*.txt files,
    agents/utils.py:10-34) -> list of lists."""
    from ast import literal_eval

    with open(path) as f:
        return [literal_eval(line.strip()) for line in f if line.strip()]


def load_initial_states_from_text_file(states_type):
    """Mirror of the reference's ``ac_solver/agents/utils.py:10-34``: the shipped presentations,
    sorted by hardness (greedy-solved first).  states_type: "solved" or "all"."""
    assert states_type in ["solved", "all"], "states_type must be 'solved' or 'all'"
    name = ("greedy_solved" if states_type == "solved" else "all") + "_presentations.txt"
    states = load_presentations_from_text_file(os.path.join(os.path.dirname(os.path.realpath(__file__)), "data", name))
    print(f"Loaded {len(states)} presentations from {name}.")
    return states
