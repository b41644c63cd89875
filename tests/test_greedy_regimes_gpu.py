"""Every tier of the batched greedy engine against the oracle (csrc/greedy.cu, csrc/greedy_bucket.cuh).

``greedy_run_impl`` serves a search in one of three tiers: bucket pass 0 (a directory of kGbBuckets1
buckets), bucket pass 1 (the searches pass 0 handed back, re-run from scratch with kGbBuckets2 buckets),
and the one-warp heap kernel (whatever pass 1 handed back).  At the production capacities almost nothing
leaves pass 0 below budget 1e6, so the tests build the library twice more with lowered capacities
(greedy_bucket.cuh's GB_* macros):

- "tiles": 64-node tiles and all-pairs ranking up to 16 nodes, so buckets span several tiles, go through
  the bitonic sort and are interrupted, at budgets the oracle finishes in milliseconds; nothing is handed back.
- "tiny": directories of 64 and 256 buckets, 3 segments per bucket, 32 sortable nodes and 200 segment
  records, so searches are handed back for reasons 1 (segments per bucket), 2 (sort buffer), 3 (segment pool)
  and 5 (directory), in pass 0 and in pass 1, and finish in pass 0, in pass 1 or in the heap kernel.

Reasons 4 and 6 cannot be reached.  Reason 6 needs a node of depth 2^24 - 1, so a chain of 2^24 committed
nodes, but a search stops once it holds ``budget`` nodes and acs_greedy_create refuses budgets above
2^24 - 32.  Reason 4 needs a frontier array of 2 * (budget + 16) entries to overflow: every committed node
enters it once, and every rest of an interrupted bucket once more; the rests alone would have to exceed
``budget`` entries before the search holds ``budget`` nodes.  The CPU model (tests/greedy_bucket_model.py)
checks the frontier exactly as the kernel does, so a reason-4 hand-back would show up in its predictions, and
none of the cases here predicts one.

Each row is checked three ways: the tier (the ACS_GREEDY_DEBUG hand-back lines and ``info["rounds"]``) equals
the CPU model's prediction, hand-back node count and bucket rounds included; the answer, the counters, the
minimal-length log and the visited array equal the oracle's; and goal runs equal ``greedy_goals``.
"""

import os
import re
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import goal_oracle as G
import greedy_bucket_model as M
from conftest import ms_row
from greedy_goal_oracle import greedy_goals
from oracle import oracle as O

pytestmark = pytest.mark.gpu

KEYS = ("n_visited", "n_expanded", "n_moves", "frontier_left", "budget_hit", "status", "minlen_log")
VARIANTS = {
    "tiles": ({"GB_TILE": 64, "GB_SMALL": 16}, M.Caps(tile=64, small=16)),
    "tiny": ({"GB_BUCKETS1": 64, "GB_BUCKETS2": 256, "GB_MAX_SEG": 3, "GB_SORT_CAP": 32, "GB_SEG_POOL": 200},
             M.Caps(buckets1=64, buckets2=256, max_seg=3, sort_cap=32, seg_pool=200)),
}
# Miller-Schupp rows by key width: W=1 (mrl 18, 24), W=2 (mrl 32, 36); row 119 is listed twice
ROWS = {1: [0, 35, 49, 105, 119, 238, 273, 119, 742], 2: [497, 504, 896, 903, 924, 1060, 1106, 1106]}
BUDGET = 3000
HANDBACK = re.compile(r"greedy: pass (\d), search (\d+) handed back \(reason (\d+), (\d+) nodes\)")


@pytest.fixture(scope="session")
def variant_libs(tmp_path_factory):
    """libacsolver_b200.so built with each variant's capacities, all sources (the loader binds every entry
    point), both variants compiling at once."""
    from ac_solver_b200 import build as B

    root = tmp_path_factory.mktemp("greedy_variants")
    env = {k: v for k, v in os.environ.items() if k not in ("CC", "CXX")}
    procs, out = [], {}
    for name, (defs, _) in VARIANTS.items():
        out[name] = str(root / f"libacsolver_b200_{name}.so")
        cmd = [B._nvcc(), *B.NVCC_FLAGS, *[f"-D{k}={v}" for k, v in defs.items()], "-o", out[name],
               *[os.path.join(B.CSRC, s) for s in B.SOURCES]]
        procs.append(subprocess.Popen(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    for p in procs:
        log = p.communicate()[0]
        assert p.returncode == 0, log.decode(errors="replace")
    return out


@pytest.fixture
def use_variant(variant_libs, monkeypatch):
    """Point the loader at a variant's library for one test; ACS_GREEDY_DEBUG makes the engine print its
    hand-backs."""
    from ac_solver_b200 import _lib

    monkeypatch.delenv("ACS_GREEDY_KERNEL", raising=False)
    monkeypatch.setenv("ACS_GREEDY_DEBUG", "1")

    def use(name):
        monkeypatch.setattr(_lib, "LIB_PATH", variant_libs[name])
        monkeypatch.setattr(_lib, "_lib", None)
        return VARIANTS[name][1]

    return use


def _handbacks(err):
    hb = {}
    for m in HANDBACK.finditer(err):
        hb.setdefault(int(m.group(2)), []).append((int(m.group(1)), int(m.group(3)), int(m.group(4))))
    return hb


def _run(capfd, rows, budget, cyc, **kw):
    from ac_solver_b200 import greedy_search_batch

    capfd.readouterr()
    got = greedy_search_batch(np.array(rows, np.int8), budget, cyc, want_visited=True, **kw)
    return got, _handbacks(capfd.readouterr().err)


def _same(a, ref):
    assert (a[0], a[1]) == (ref[0], ref[1])
    for k in KEYS:
        assert a[2][k] == ref[2][k], k
    assert np.array_equal(a[2]["visited"], ref[2]["visited"])


def _check(rows, got, hb, budget, cyc, caps, goals=None):
    """Tier = the model's, answer = the oracle's; -> the tiers seen, as (hand-backs, finished by)."""
    seen = []
    gd = None if goals is None else G.goal_dict(goals)
    for s, (r, a) in enumerate(zip(rows, got)):
        want_hb, rounds = M.tiers(r, budget, cyc, gd, caps)
        assert hb.get(s, []) == want_hb, s
        assert a[2]["rounds"] == (-1 if rounds is None else rounds), s
        if goals is None:
            es, ep, ei = O.greedy_search(r, budget, cyc, want_visited=True)
            _same(a, (es, ep, ei))
        else:
            ref = greedy_goals(r, budget, cyc, goals=gd, want_visited=True)
            _same(a, ref)
            assert a[2]["goal"] == ref[2]["goal"]
        seen.append((tuple((p, q) for p, q, _ in want_hb), "heap" if rounds is None else f"pass {len(want_hb)}"))
    return seen


def _groups(ms, ks):
    by = {}
    for k in ks:
        r = ms_row(ms, k)
        by.setdefault(len(r), []).append(r)
    return by.values()


@pytest.mark.parametrize("cyc", [False, True])
@pytest.mark.parametrize("W", [1, 2])
def test_small_tiles_multi_tile_buckets_match_the_oracle(miller_schupp, use_variant, capfd, W, cyc):
    """64-node tiles: buckets of several tiles, sorted by the bitonic network, interrupted and put back."""
    caps = use_variant("tiles")
    big = rests = 0
    for rows in _groups(miller_schupp, ROWS[W]):
        got, hb = _run(capfd, rows, BUDGET, cyc)
        assert not hb
        _check(rows, got, hb, BUDGET, cyc, caps)
        for r in rows:
            st = {}
            M.bucket_pass(r, BUDGET, cyc, caps=caps, stats=st)
            big, rests = max(big, st["max_bucket"]), rests + st["rests"]
    print(f"W={W} cyc={cyc}: largest bucket {big} nodes, {rests} interrupted rests put back")
    # the bitonic sort everywhere; buckets of several tiles except in the plain W=1 searches (38 nodes at most)
    assert big > (caps.small if (W, cyc) == (1, False) else caps.tile) and rests > 0


# (pass, reason) hand-backs the "tiny" cases reach, and how their searches finish, per (W, cyclical)
TINY_COVERAGE = {
    (1, False): {(0, 2), (0, 5), (1, 2), (1, 3)},
    (1, True): {(0, 1), (0, 2), (0, 5), (1, 1), (1, 2)},
    (2, False): {(0, 2), (0, 5), (1, 2), (1, 3)},
    (2, True): {(0, 2), (0, 5), (1, 2), (1, 3)},
}


@pytest.mark.parametrize("cyc", [False, True])
@pytest.mark.parametrize("W", [1, 2])
def test_tiny_capacities_every_tier_matches_the_oracle(miller_schupp, use_variant, capfd, W, cyc):
    """Rows served by pass 0, pass 1 and the heap kernel in one launch (a row listed twice included): each
    one's hand-backs and rounds are the model's, and its answer, counters and visited array the oracle's."""
    caps = use_variant("tiny")
    seen = []
    for rows in _groups(miller_schupp, ROWS[W]):
        got, hb = _run(capfd, rows, BUDGET, cyc)
        seen += _check(rows, got, hb, BUDGET, cyc, caps)
        for i, j in [(i, j) for i in range(len(rows)) for j in range(i) if np.array_equal(rows[i], rows[j])]:
            _same(got[i], got[j])
    print(f"W={W} cyc={cyc}: " + "; ".join(f"{h} -> {f}" for h, f in sorted(set(seen))))
    assert {x for h, _ in seen for x in h} == TINY_COVERAGE[(W, cyc)]
    assert {f for _, f in seen} >= {"pass 0", "heap"}
    if not (W == 2 and cyc):
        assert "pass 1" in {f for _, f in seen}


# (row, cyclical, tier at which the goal must be met, whether the search is handed back deeper than the goal)
GOAL_CASES = [(35, False, "pass 1", False), (49, True, "pass 1", False), (119, False, "heap", True),
              (896, False, "heap", False), (1106, True, "heap", True)]


def _goal_for(r, cyc, caps, tier):
    """Two states of the plain search's visited array generated well after the hand-back the goal must
    outlast: one halfway to the end, and the shallowest one.  -> (visited indices, deepest node committed
    before that hand-back, depth of the shallow goal)."""
    hb, _ = M.tiers(r, BUDGET, cyc, None, caps)
    st = {}
    M.bucket_pass(r, BUDGET, cyc, stats=st)  # the plain search, at the production capacities
    after = hb[-1][2] if tier == "heap" else hb[0][2]
    depth = st["depth"]
    cand = list(range(after + max(1, (len(depth) - after) // 4), len(depth)))
    deep = max(depth[:after])
    shallow = min(cand, key=lambda j: (depth[j], j))
    return [cand[len(cand) // 2], shallow], deep, depth[shallow]


@pytest.mark.parametrize("k,cyc,tier,past", GOAL_CASES)
def test_goals_across_a_handback(miller_schupp, use_variant, capfd, k, cyc, tier, past):
    """Goal hits resolved in pass 1 (the goal slot follows the larger directory) and in the heap re-run; one
    goal of each search is shallower than where the search was handed back.  The path-overflow re-run
    (path_cap=4) keeps the hits."""
    from ac_solver_b200 import GoalSet

    caps = use_variant("tiny")
    r = ms_row(miller_schupp, k)
    _, _, plain = O.greedy_search(r, BUDGET, cyc, want_visited=True)
    picks, deep, shallow_depth = _goal_for(r, cyc, caps, tier)
    for pick in picks:
        goals = plain["visited"][[pick]]
        with GoalSet.from_rows(goals, cyc) as g:
            got, hb = _run(capfd, [r], BUDGET, cyc, goals=g)
            seen = _check([r], got, hb, BUDGET, cyc, caps, goals)
            assert got[0][2]["goal"] == 0
            assert seen[0][1] == tier and seen[0][0], seen
            small, _ = _run(capfd, [r], BUDGET, cyc, goals=g, path_cap=4)
        assert len(got[0][1]) > 4
        _same(small[0], got[0])
        assert small[0][2]["goal"] == 0
    assert (shallow_depth < deep) == past


def test_production_capacities_at_the_sweep_budget(miller_schupp, capfd, monkeypatch):
    """The 1190 Miller-Schupp rows at budget 1e6 with the default library: every row pass 0 hands back equals
    the oracle in full (the visited array included), and greedy_search_groups returns what
    greedy_search_batch does."""
    from ac_solver_b200 import greedy_search_batch
    from ac_solver_b200.search.greedy import greedy_search_groups

    monkeypatch.delenv("ACS_GREEDY_KERNEL", raising=False)
    monkeypatch.setenv("ACS_GREEDY_DEBUG", "1")
    budget = 1_000_000
    ks = {}
    for k in range(1190):
        ks.setdefault(len(ms_row(miller_schupp, k)), []).append(k)
    groups = [np.array([ms_row(miller_schupp, k) for k in v], np.int8) for v in ks.values()]
    batch, hb = [], []
    for gi, P in enumerate(groups):
        capfd.readouterr()
        batch.append(greedy_search_batch(P, budget))
        hb += [(gi, s, h) for s, h in _handbacks(capfd.readouterr().err).items()]
    assert hb, "no search left pass 0"
    assert all(h[0][0] == 0 for _, _, h in hb)
    print(f"{len(hb)} searches handed back by pass 0: " + ", ".join(
        f"mrl {groups[gi].shape[1] // 2} #{s} {h}" for gi, s, h in hb))
    for gi, P in enumerate(groups):
        idx = [s for g, s, _ in hb if g == gi]
        if not idx:
            continue
        again = greedy_search_batch(P[idx], budget, want_visited=True)
        with ThreadPoolExecutor(8) as pool:
            refs = list(pool.map(lambda s: O.greedy_search(P[s], budget, want_visited=True), idx))
        for s, a, ref in zip(idx, again, refs):
            _same(a, ref)
            assert (a[0], a[1], a[2]["rounds"]) == (batch[gi][s][0], batch[gi][s][1], batch[gi][s][2]["rounds"])
    for P, a, b in zip(groups, greedy_search_groups(groups, budget, path_cap=4096), batch):
        for x, y in zip(a, b):
            assert (x[0], x[1]) == (y[0], y[1])
            for k in KEYS + ("rounds",):
                assert x[2][k] == y[2][k], k
