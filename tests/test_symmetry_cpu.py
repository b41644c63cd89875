"""The presentation symmetry group G (tests/sym_oracle.py, csrc/ac_sym.cuh) on the CPU: group laws, the
move permutation pi_g against the C oracle, the header's canonical form against the plain one, and the
conversion of canonical-frame paths into actual moves."""

import numpy as np
import pytest

import sym_oracle as S
from ac_solver_b200.synthetic import random_presentations
from hostsim import sym as H
from oracle import oracle as O
from width_edges import HAND_PICKED, WIDTHS


def _states(mrl, n=24, seed=0):
    """Random reduced states, plus rows on which concatenations raise (r1 = r0 and r1 = r0^-1)."""
    P = random_presentations(n, mrl, seed=seed)
    extra = []
    for r in P[:4]:
        w = r[:mrl]
        inv = -w[: np.count_nonzero(w)][::-1]
        extra.append(np.concatenate([w, w]))
        extra.append(np.concatenate([w, np.pad(inv, (0, mrl - inv.size))]))
    rows = [P, np.array(extra, np.int8)]
    if mrl in HAND_PICKED:
        rows.append(np.array(HAND_PICKED[mrl], np.int8))
    return np.ascontiguousarray(np.concatenate(rows), dtype=np.int8)


def test_group_laws():
    mul, inv = np.array(S.MUL), np.array(S.INV)
    assert (mul[0] == np.arange(16)).all() and (mul[:, 0] == np.arange(16)).all()
    assert all(mul[g, inv[g]] == 0 and mul[inv[g], g] == 0 for g in range(16))
    for g in range(16):
        assert sorted(mul[g]) == list(range(16))  # a Latin square: every product once
        for h in range(16):
            for k in range(16):
                assert mul[mul[g, h], k] == mul[g, mul[h, k]]
    for g in range(16):
        assert sorted(S.PI[g]) == list(range(12))
        for h in range(16):
            assert [S.PI[mul[g, h]][m] for m in range(12)] == [S.PI[g][S.PI[h][m]] for m in range(12)]
    # the product is the action's composition
    row = np.array([1, -2, 1, 2, 0, 2, 2, -1, 0, 0], np.int8)
    for g in range(16):
        for h in range(16):
            assert np.array_equal(S.act(mul[g, h], row), S.act(g, S.act(h, row)))
    # the 8 trivial presentations are one orbit
    triv = np.array([[1, 0, 2, 0]], np.int8)
    assert len({S.act(g, triv[0]).tobytes() for g in range(16)}) == 8


def test_header_tables_match_oracle():
    mul, inv, pi = H.tables()
    assert np.array_equal(mul, np.array(S.MUL)) and np.array_equal(inv, np.array(S.INV))
    assert np.array_equal(pi, np.array(S.PI))


@pytest.mark.parametrize("cyclical", [False, True])
def test_pi_is_equivariant(cyclical):
    """acmove(PI[g][m], g.s) = g.acmove(m, s) and the same status, for every g and m, at every width edge,
    on states that include raising ones."""
    raised = 0
    for mrl in WIDTHS:
        P = _states(mrl, seed=mrl)
        n = len(P)
        for m in range(12):
            out, _, st = O.moves_batch(P, np.full(n, m, np.uint8), cyclical=cyclical)
            raised += int((st != 0).sum())
            for g in range(16):
                out2, _, st2 = O.moves_batch(S.act(g, P), np.full(n, S.PI[g][m], np.uint8), cyclical=cyclical)
                assert np.array_equal(st, st2), (mrl, g, m)
                ok = st == 0
                assert np.array_equal(S.act(g, out[ok]), out2[ok]), (mrl, g, m)
    assert raised > 0


def test_header_canonical_matches_oracle():
    rng = np.random.default_rng(5)
    for mrl in (1, 2, 3, 4, 28, 29, 30, 31, 32, 33, 60, 61):
        P = _states(mrl, n=60, seed=100 + mrl)
        c, g = H.canonical(P)
        cb, gb = S.canonical_batch(P)
        assert np.array_equal(cb, c) and np.array_equal(gb, g)
        for k in range(len(P)):
            ck, gk = S.canonical(P[k])
            assert np.array_equal(c[k], ck) and g[k] == gk, (mrl, P[k])
            assert np.array_equal(S.act(int(g[k]), P[k]), c[k])
        el = rng.integers(0, 16, size=len(P)).astype(np.uint8)
        img, _ = H.canonical(P, apply=el)
        for k in range(len(P)):
            assert np.array_equal(img[k], S.act(int(el[k]), P[k]))
        # every image of a row has the same canonical form
        for k in range(0, len(P), 7):
            imgs = np.stack([S.act(h, P[k]) for h in range(16)])
            ci, _ = H.canonical(imgs)
            assert (ci == c[k]).all()


def test_canonical_order_is_length_then_reversed_codes():
    # the shorter relator goes first
    c, g = S.canonical(np.array([1, 2, 0, 1, 0, 0], np.int8))
    assert c.tolist() == [2, 0, 0, 2, 1, 0] and g == 12  # swap x <-> y and the relators
    # then relator 0 from its last letter: xy (y=0 last) before yx (x=1 last)
    assert S.order_key([1, 2, 2, 0]) < S.order_key([2, 1, 2, 0])
    # codes y=0 < x=1 < y^-1=2 < x^-1=3
    assert [S.order_key([v, 2])[1] for v in (2, 1, -2, -1)] == [0, 1, 2, 3]


@pytest.mark.parametrize("cyclical", [False, True])
def test_orbit_paths_replay(cyclical):
    """Canonical-frame paths converted to actual moves replay from the row to total length 2 under the
    oracle, and have the length exact search finds."""
    P = random_presentations(40, 4, seed=11, max_len=4)
    n_solved = 0
    for row in P:
        ok, path, info = S.orbit_bfs(row, 3000, cyclical)
        if not ok:
            continue
        n_solved += 1
        assert S.replay(row, path, cyclical) == 2
        ok2, path2, _ = O.bfs(row, 200_000, cyclical)
        if ok2:
            assert len(path2) == len(path)
    assert n_solved >= 10


def test_actual_path_frames():
    # root not canonical: the first actual move is PI[g0^-1][m]
    row = np.array([2, 2, 1, 0, 1, 0, 0, 0], np.int8)
    c0, g0 = S.canonical(row)
    assert g0 != 0
    for m in range(12):
        child, lens = O.acmove(m, c0, 4, cyclical=False)
        path = S.actual_path([(g0, 4), (m, None, int(sum(lens)))])
        actual, lens2 = O.acmove(path[1][0], row, 4, cyclical=False)
        assert np.array_equal(S.act(S.INV[g0], child), actual) and sum(lens2) == sum(lens)


def test_package_tables_match_oracle():
    from ac_solver_b200.search.goals import PI, sym_inv, sym_mul

    assert [[sym_mul(g, h) for h in range(16)] for g in range(16)] == S.MUL
    assert [sym_inv(g) for g in range(16)] == S.INV
    assert PI == S.PI
