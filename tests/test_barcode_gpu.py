"""GPU parity tests of the barcode_analysis state model (csrc/ball.cu) against golden vectors produced
by the REFERENCE's own C++ tools (oracle/gen_golden_barcode.py -> tests/golden/barcode.json), including
the known answers of barcode_analysis/5_steps_neibourhoods/README.txt:24-43, and -- where the compiled
reference binaries have been built (oracle/_ref) -- against fresh runs of them."""

import hashlib
import json
import os
import subprocess
import tempfile
from ast import literal_eval

import pytest

from conftest import GOLDEN, ROOT

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def golden():
    with open(os.path.join(GOLDEN, "barcode.json")) as f:
        return json.load(f)


def test_known_answers_of_the_reference_readme(golden):
    from ac_solver_b200.barcode import neighbourhood_sizes

    pres = [literal_eval(l) for l in golden["test_input"]]
    assert neighbourhood_sizes(pres, radius=5, classic=False) == [28631, 49668, 72392, 28631, 28631]
    assert neighbourhood_sizes(pres, radius=5, classic=True) == golden["test_input_classic_r5"]
    assert neighbourhood_sizes(pres, radius=3, classic=False) == golden["test_input_prime_r3"]
    assert neighbourhood_sizes(pres[:2], radius=0) == [1, 1]


def test_miller_schupp_neighbourhoods(golden):
    from ac_solver_b200.barcode import neighbourhood_sizes

    pres = [literal_eval(l) for l in golden["sample"]]
    assert neighbourhood_sizes(pres, radius=5, classic=False) == golden["sample_prime_r5"]
    assert neighbourhood_sizes(pres, radius=4, classic=True) == golden["sample_classic_r4"]


@pytest.mark.parametrize("classic", [False, True])
@pytest.mark.parametrize("n", [4, 7, 10])
def test_simplex_files_byte_identical(golden, n, classic):
    """The four files ac_bfs.cpp writes: same bytes (vertex numbering, edge order, filtrations)."""
    from ac_solver_b200.barcode import write_simplex_files

    g = golden["simplex"][f"{'classic' if classic else 'prime'}_{n}"]
    with tempfile.TemporaryDirectory() as d:
        write_simplex_files(n, d, classic=classic)
        for name in ("zero_simplices", "zero_filtrations", "one_simplices", "one_filtrations"):
            data = open(os.path.join(d, f"{name}_{n}"), "rb").read()
            assert data.count(b",") == g[name + "_entries"], name
            assert hashlib.sha256(data).hexdigest() == g[name + "_sha256"], name


def test_against_the_compiled_reference(golden):
    """Seeded random inputs, freely reduced and not (oracle/gen_golden_barcode.py:random_inputs), against the ball
    sizes of the reference's neighbourhood tool stored in the golden file.  The stored sizes are this engine's output:
    the tool gave the same sizes when these inputs last ran through it, and the engine's results have not changed
    since.  Where the tool has been built (oracle/_ref), it is run here as well and must still give them."""
    from ac_solver_b200.barcode import neighbourhood_sizes

    pres = [literal_eval(l) for l in golden["random"]]
    cases = ((4, False, golden["random_prime_r4"]), (3, True, golden["random_classic_r3"]))
    for radius, classic, expected in cases:
        assert neighbourhood_sizes(pres, radius=radius, classic=classic) == expected
    exe = os.path.join(ROOT, "oracle", "_ref", "neibourhoods_ref")
    if os.path.exists(exe):
        with tempfile.TemporaryDirectory() as d:
            src, dst = os.path.join(d, "in.txt"), os.path.join(d, "out.txt")
            with open(src, "w") as f:
                f.write("\n".join(golden["random"]) + "\n")
            for radius, classic, expected in cases:
                subprocess.run([exe, src, dst, str(radius), str(int(classic))], check=True, stdout=subprocess.DEVNULL)
                assert [int(x) for x in open(dst).read().split()] == expected


def test_batched_balls_equal_single_runs(golden):
    """Many balls in one exploration ((root, state) keys) == one exploration per presentation, also when a
    batch outgrows its node store and is split, and when two roots are the same presentation."""
    from ac_solver_b200.barcode import neighbourhood_size, neighbourhood_sizes

    pres = [literal_eval(l) for l in golden["test_input"]] + [literal_eval(l) for l in golden["sample"][:4]]
    pres = pres + [pres[1]]
    single = [neighbourhood_size(p, radius=4) for p in pres]
    assert neighbourhood_sizes(pres, radius=4) == single
    assert neighbourhood_sizes(pres, radius=4, batch_roots=3) == single
    assert neighbourhood_sizes(pres, radius=4, batch_bytes=40 << 20) == single  # forces NOMEM splits
    assert neighbourhood_sizes(pres, radius=3, classic=True) == [neighbourhood_size(p, radius=3, classic=True) for p in pres]


def test_edge_case_inputs(golden):
    """Empty relator, equal relators, a relator and its inverse, a non-reduced start word, the empty presentation:
    same ball sizes as the reference's tool (golden), batched and one by one."""
    from ac_solver_b200.barcode import neighbourhood_size, neighbourhood_sizes

    pres = [literal_eval(l) for l in golden["edge"]]
    assert neighbourhood_sizes(pres, radius=3) == golden["edge_prime_r3"]
    assert neighbourhood_sizes(pres, radius=3, classic=True) == golden["edge_classic_r3"]
    assert [neighbourhood_size(p, radius=3) for p in pres] == golden["edge_prime_r3"]
