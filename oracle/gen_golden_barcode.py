#!/usr/bin/env python
"""TEST INFRASTRUCTURE.  Generates tests/golden/barcode.json by running the REFERENCE's own
barcode_analysis tools (compiled from /root/reference into oracle/_ref by `make -C oracle _ref`):
radius-5 ball sizes for the reference's test_input.txt (known answers of its README.txt:24-43) and
for sampled Miller-Schupp presentations, prime and classic moves; for seeded random presentations,
reduced and not; and, for small n, the sha256 of the four simplex files ac_bfs writes plus their
vertex / edge counts."""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = "/root/reference/barcode_analysis"
sys.path.insert(0, ROOT)


def ball_sizes(lines, radius, classic):
    with tempfile.TemporaryDirectory() as d:
        src, dst = os.path.join(d, "in.txt"), os.path.join(d, "out.txt")
        with open(src, "w") as f:
            f.write("\n".join(lines) + "\n")
        subprocess.run([os.path.join(HERE, "_ref", "neibourhoods_ref"), src, dst, str(radius), str(int(classic))],
                       check=True, stdout=subprocess.DEVNULL)
        return [int(x) for x in open(dst).read().split()]


def simplex(n, classic):
    exe = os.path.join(HERE, "_ref", "ac_bfs_classic" if classic else "ac_bfs_prime")
    with tempfile.TemporaryDirectory() as d:
        subprocess.run([exe, str(n)], cwd=d, check=True, stdout=subprocess.DEVNULL)
        out = {}
        for name in ("zero_simplices", "zero_filtrations", "one_simplices", "one_filtrations"):
            data = open(os.path.join(d, f"{name}_{n}"), "rb").read()
            out[name + "_sha256"] = hashlib.sha256(data).hexdigest()
            out[name + "_entries"] = data.count(b",")
        return out


def random_inputs():
    """Six seeded random presentations of freely reduced words, then six of words that are NOT freely reduced: the
    reference's reduce_ is not plain free reduction on them (AC_UTILS_no_hash.cpp:58-88), and inv0_ does not reduce
    at all -- the engine restates both literally."""
    import numpy as np

    rng = np.random.default_rng(4)
    pres = []
    for _ in range(6):
        rows = []
        for _h in range(2):
            w = []
            while len(w) < int(rng.integers(1, 7)):
                c = int(rng.choice([-2, -1, 1, 2]))
                if not w or w[-1] != -c:
                    w.append(c)
            rows.append(w + [0] * (8 - len(w)))
        pres.append(rows[0] + rows[1])
    for _ in range(6):
        rows = []
        for _h in range(2):
            w = [int(rng.choice([-2, -1, 1, 2])) for _ in range(int(rng.integers(0, 7)))]
            rows.append(w + [0] * (8 - len(w)))
        pres.append(rows[0] + rows[1])
    return [str(p) for p in pres]


def main():
    subprocess.check_call(["make", "-C", HERE, "_ref"])
    test_input = [l.strip() for l in open(os.path.join(REF, "5_steps_neibourhoods", "test_input.txt")) if l.strip()]
    solved = [l.strip() for l in open(os.path.join(REF, "5_steps_neibourhoods", "solved_miller_schupp_presentations.txt")) if l.strip()]
    unsolved = [l.strip() for l in open(os.path.join(REF, "5_steps_neibourhoods", "unsolved_miller_schupp_presentations.txt")) if l.strip()]
    sample = solved[:: max(1, len(solved) // 10)][:10] + unsolved[:: max(1, len(unsolved) // 10)][:10]
    # edge cases of the input format (neibourhoods.cpp:80-90 drops the zeros of each half): an empty relator, two equal
    # relators, a relator and its inverse, a NON-reduced start word, the empty presentation
    edge = ["[0, 0, 0, 0, 2, 0, 0, 0]", "[1, 2, 0, 0, 1, 2, 0, 0]", "[1, 2, 0, 0, -2, -1, 0, 0]", "[1, -1, 0, 0, 2, 0, 0, 0]",
            "[0, 0, 0, 0]"]
    random = random_inputs()
    g = {"edge": edge, "edge_prime_r3": ball_sizes(edge, 3, False), "edge_classic_r3": ball_sizes(edge, 3, True),
         "test_input": test_input, "test_input_prime_r5": ball_sizes(test_input, 5, False),
         "test_input_classic_r5": ball_sizes(test_input, 5, True), "test_input_prime_r3": ball_sizes(test_input, 3, False),
         "sample": sample, "sample_prime_r5": ball_sizes(sample, 5, False), "sample_classic_r4": ball_sizes(sample, 4, True),
         "simplex": {f"{'classic' if c else 'prime'}_{n}": simplex(n, c) for c in (False, True) for n in (4, 7, 10)},
         "random": random, "random_prime_r4": ball_sizes(random, 4, False), "random_classic_r3": ball_sizes(random, 3, True)}
    assert g["test_input_prime_r5"] == [28631, 49668, 72392, 28631, 28631]  # README.txt:24-43
    with open(os.path.join(ROOT, "tests", "golden", "barcode.json"), "w") as f:
        json.dump(g, f, indent=1)
    print("wrote tests/golden/barcode.json:", {k: (v if "r" in k and isinstance(v, list) and len(v) < 8 else "...") for k, v in g.items()})


if __name__ == "__main__":
    main()
