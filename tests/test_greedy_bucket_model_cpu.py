"""The CPU model of the bucket kernel's bookkeeping (tests/greedy_bucket_model.py) replays the oracle's search:
when no capacity is reached it ends with the oracle's node count, whatever the tile size."""

import numpy as np
import pytest

import greedy_bucket_model as M
from conftest import ms_row
from oracle import oracle as O


@pytest.mark.parametrize("cyc", [False, True])
@pytest.mark.parametrize("tile", [1024, 64, 8])
def test_model_replays_the_oracle_search(miller_schupp, cyc, tile):
    for k in (0, 40, 200, 700, 1000):
        r = ms_row(miller_schupp, k)
        st = {}
        res = M.bucket_pass(r, 2000, cyc, caps=M.Caps(tile=tile), stats=st)
        _, _, ei = O.greedy_search(r, 2000, cyc)
        assert res[0] == "done" and res[2] == ei["n_visited"] == len(st["depth"]), k
        assert res[1] >= 1


def test_model_hands_back_at_the_first_capacity_reached(miller_schupp):
    """A directory of one bucket overflows at the root's first children, before any node is committed."""
    r = ms_row(miller_schupp, 0)
    assert M.bucket_pass(r, 2000, caps=M.Caps(buckets1=1)) == ("handback", 5, 1)
    assert M.tiers(r, 2000, caps=M.Caps(buckets1=1, buckets2=1))[0] == [(0, 5, 1), (1, 5, 1)]
