"""Compare the device code of the search kernels between a git revision and the working tree.

    python scripts/compare_kernel_sass.py [BASE_REV] [--keep DIR]

Both trees' ``ac_solver_b200/csrc`` sources are compiled with the library's nvcc flags plus
``-Xptxas -v``, one object per translation unit.  ``cuobjdump -sass`` of each object is split per
function, the address and encoding comments are stripped, and every function whose demangled
name starts with one of the watched kernel names (every template instantiation) is compared.
Register, stack and spill lines from ptxas are compared for the same functions.  Prints one line
per function and exits non-zero when a kernel listed in ``MUST_MATCH`` differs.  Needs no GPU.
"""

from __future__ import annotations

import argparse
import concurrent.futures as cf
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ac_solver_b200.build import NVCC_FLAGS, SOURCES, _nvcc  # noqa: E402

# kernels whose code a refactor of the host plumbing must not touch
MUST_MATCH = [
    "pb_expand_kernel", "pb_expand_cta_kernel", "pb_insert_kernel", "pb_commit_kernel",
    "mb_expand_kernel", "mb_insert_kernel", "mb_commit_kernel", "mb_goal_kernel",
    "greedy_kernel", "greedy_bucket_kernel", "gs_insert_kernel",
    "sb_expand_kernel", "sb_insert_kernel", "canonical_form_kernel",
]
# kernels reported for information (unpack, lookup, path and decide kernels)
WATCH = MUST_MATCH + [
    "records_unpack_kernel", "keys_unpack_kernel", "pb_unpack_kernel", "mb_unpack_kernel",
    "mb_decide_kernel", "pb_path_kernel", "pb_lookup_kernel", "mb_path_kernel", "greedy_path_kernel",
    "gs_path_kernel", "sb_lookup_kernel", "sb_path_kernel",
]


def _compile(csrc: str, src: str, out_dir: str) -> tuple[str, str]:
    obj = os.path.join(out_dir, src.replace(".cu", ".o"))
    flags = [f for f in NVCC_FLAGS if f not in ("-shared",)]
    cmd = [_nvcc(), *flags, "-Xptxas", "-v", "-c", "-o", obj, os.path.join(csrc, src)]
    env = {k: v for k, v in os.environ.items() if k not in ("CC", "CXX")}
    p = subprocess.run(cmd, capture_output=True, text=True, env=env)
    if p.returncode:
        raise RuntimeError(f"{src}: nvcc failed\n{p.stderr}")
    return obj, p.stderr


def _demangle(names: list[str]) -> dict[str, str]:
    p = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True)
    return dict(zip(names, p.stdout.splitlines()))


def _sass(obj: str) -> dict[str, str]:
    text = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    funcs: dict[str, list[str]] = {}
    cur = None
    for line in text.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
            continue
        if cur is None:
            continue
        line = re.sub(r"/\*[0-9a-f]{4,}\*/", "", line)      # instruction address
        line = re.sub(r"/\* 0x[0-9a-f]+ \*/", "", line)     # encoding
        line = line.strip()
        if line:
            funcs[cur].append(line)
    return {k: "\n".join(v) for k, v in funcs.items()}


def _ptxas(log: str) -> dict[str, str]:
    out: dict[str, str] = {}
    cur = None
    for line in log.splitlines():
        m = re.search(r"Compiling entry function '(\S+)'", line) or re.search(r"Function properties for (\S+)", line)
        if m:
            cur = m.group(1)
            continue
        if cur and ("registers" in line or "stack frame" in line):
            out[cur] = (out.get(cur, "") + " " + re.sub(r"^ptxas info\s*:\s*", "", line.strip())).strip()
    return out


def _tree(csrc: str, work: str) -> tuple[dict[str, str], dict[str, str]]:
    os.makedirs(work, exist_ok=True)
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(csrc, s))]
    sass: dict[str, str] = {}
    regs: dict[str, str] = {}
    with cf.ThreadPoolExecutor(max_workers=min(len(srcs), os.cpu_count() or 1)) as ex:
        for obj, log in ex.map(lambda s: _compile(csrc, s, work), srcs):
            sass.update(_sass(obj))
            regs.update(_ptxas(log))
    return sass, regs


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("base", nargs="?", default="HEAD")
    ap.add_argument("--keep", help="directory for the objects (default: a temporary one)")
    a = ap.parse_args()
    with tempfile.TemporaryDirectory() as tmp:
        work = a.keep or tmp
        base_src = os.path.join(work, "base")
        os.makedirs(base_src, exist_ok=True)
        archive = subprocess.run(["git", "-C", ROOT, "archive", a.base, "ac_solver_b200/csrc", "include"], capture_output=True,
                                 check=True).stdout
        subprocess.run(["tar", "-x", "-C", base_src], input=archive, check=True)
        base_csrc = os.path.join(base_src, "ac_solver_b200", "csrc")
        with cf.ThreadPoolExecutor(max_workers=2) as ex:
            fb = ex.submit(_tree, base_csrc, os.path.join(work, "base_obj"))
            fh = ex.submit(_tree, os.path.join(ROOT, "ac_solver_b200", "csrc"), os.path.join(work, "head_obj"))
            (sb, rb), (sh, rh) = fb.result(), fh.result()
    names = sorted(set(sb) | set(sh))
    pretty = _demangle(names)
    bad = 0
    for n in sorted(names, key=lambda k: pretty[k]):
        p = pretty[n]
        base = p.split("(")[0].split("<")[0].split("::")[-1]
        if base.startswith("void "):
            base = base[5:]
        if base not in WATCH:
            continue
        if n not in sb:
            state = "new"
        elif n not in sh:
            state = "removed"
        else:
            same = sb[n] == sh[n] and rb.get(n) == rh.get(n)
            state = "identical" if same else "DIFFERS"
            if not same and base in MUST_MATCH:
                bad += 1
        print(f"{state:9s} {p}\n          base: {rb.get(n, '-')}\n          head: {rh.get(n, '-')}")
    print(f"{bad} watched kernel(s) that must match differ")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
