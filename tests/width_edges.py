"""Roots at the edges of the packed key layout (csrc/ac_keys.cuh), shared by the width-edge tests.

Every device search packs a state into ``Key<W>``: W = 1 (16-byte keys) up to max_relator_length 29,
W = 2 (32 bytes) up to 61, 2-bit letter codes with each relator's length in the top 6 bits of its last
64-bit word.  ``WIDTHS`` puts a search where a full relator meets that layout: letter 28 right under the
length field (29), a length of 61 setting bit 63, relators crossing the 32-bit halves and 64-bit words
(15-17, 31-33), both sides of the key-width switch (28-30) and of the last two-word width (60-61), and the
widths 1-4 where most concatenations are rejected and roots raise or solve at once.
"""

from __future__ import annotations

import numpy as np

from ac_solver_b200 import _lib
from ac_solver_b200.synthetic import random_presentations

WIDTHS = (1, 2, 3, 4, 15, 16, 17, 28, 29, 30, 31, 32, 33, 60, 61)
BUDGET = 20_000

# mrl -> a row that raises (r1 == r0^-1 or r1 == r0: a concatenation empties a relator before any child
# has total length 2) and a row that solves at the first level (total length 2 already, or xy, y -> x, y);
# outcomes read off the oracle, checked by tests/test_width_edges_cpu.py
HAND_PICKED = {
    1: [[1, -1], [2, 1]],
    2: [[1, 2, 1, 2], [1, 2, 2, 0]],
    3: [[1, 2, 2, 1, 2, 2], [1, 2, 0, 2, 0, 0]],
    4: [[1, 2, -1, -2, 2, 1, -2, -1], [1, 2, 0, 0, 2, 0, 0, 0]],
}


def roots(mrl):
    """-> int8 [k, 2*mrl], the same on every call:
    rows 0-3: relator 0 of 2 to mrl letters (at least mrl - 2), relator 1 of 1 to 3 letters;
    row 4: both relators at full length;
    row 5 (mrl >= 2): both relators of mrl - 1 letters, so a conjugation that cancels nothing is
    rejected by one letter;
    then, at mrl 1-4, the rows of ``HAND_PICKED``."""
    base = random_presentations(4, mrl, seed=mrl, min_len=max(1, mrl - 2))
    base[:, mrl:] = random_presentations(4, mrl, seed=mrl + 7, max_len=min(3, mrl))[:, mrl:]
    rows = [base, random_presentations(1, mrl, seed=100 + mrl, min_len=mrl)]
    if mrl >= 2:
        rows.append(random_presentations(1, mrl, seed=200 + mrl, min_len=mrl - 1, max_len=mrl - 1))
    if mrl in HAND_PICKED:
        rows.append(np.array(HAND_PICKED[mrl], np.int8))
    return np.ascontiguousarray(np.concatenate(rows), dtype=np.int8)


def relator_lengths(states, mrl):
    """-> (lengths of relator 0, lengths of relator 1) of int8 rows [n, 2*mrl]."""
    s = np.asarray(states)
    return np.count_nonzero(s[:, :mrl], axis=1), np.count_nonzero(s[:, mrl:], axis=1)


def full_length_count(visited, mrl):
    """Visited states with at least one relator of exactly mrl letters."""
    l0, l1 = relator_lengths(visited, mrl)
    return int(((l0 == mrl) | (l1 == mrl)).sum())


def oracle_or_status(fn, *args, **kwargs):
    """``fn(*args, **kwargs)``, or the row status the batched engines report where it raises like the
    reference: ``_lib.ROW_ASSERT`` for AssertionError, ``_lib.ROW_INDEX`` for IndexError."""
    try:
        return fn(*args, **kwargs)
    except AssertionError:
        return _lib.ROW_ASSERT
    except IndexError:
        return _lib.ROW_INDEX
