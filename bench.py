#!/usr/bin/env python
"""bench.py -- headline benchmark of the AC-move hot path (BASELINE.json config 2).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the batched ``ACEnv.step`` kernel over one batch of 1 Mi synthetic
presentations (max_relator_length 36, uniform random AC' moves) per GPU.  Rows are independent,
so N GPUs run N shards with no data-path collective (weak scaling).  One JSON line is printed
by rank 0; see the task contract for the keys.  ``--impl reference`` times the CPU oracle (the
C restatement of the reference's pure-Python path, oracle/) on all host threads instead.
"""

from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HORIZON = 200
# The synthetic states are freely and cyclically reduced, and ACEnv.step keeps them so: the
# steady-state (ACS_FLAG_NORMALIZED) variant of the kernel is the one an environment runs on
# every step but the first after a reset with caller-supplied states.  Like ACEnv.lengths, the
# relator lengths travel with the state (ACS_FLAG_LENS_VALID).  BENCH_FLAGS=0 times the general variant.
FLAGS = int(os.environ.get("BENCH_FLAGS", "6"))
L2_BYTES = 126 * 1024 * 1024
DUMP_BYTES = 48 << 20  # --dump-outputs: 161 319 of the 1 Mi rows at mrl 36


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=1 << 20, help="presentations per GPU per step")
    ap.add_argument("--mrl", type=int, default=36)
    ap.add_argument("--cpu-sample-rows", type=int, default=1 << 17)
    ap.add_argument("--skip-bfs", action="store_true")
    ap.add_argument("--bfs-budget", type=int, default=1_000_000_000, help="BASELINE.json configs[4]: 1e9 nodes")
    ap.add_argument("--bfs-timeout", type=float, default=420.0)
    ap.add_argument("--skip-python-baseline", action="store_true")
    ap.add_argument("--skip-greedy", action="store_true")
    ap.add_argument("--skip-vecenv", action="store_true")
    ap.add_argument("--skip-barcode", action="store_true")
    ap.add_argument("--skip-ppo", action="store_true")
    ap.add_argument("--greedy-budget", type=int, default=1_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (rank 0's rows; a fixed sample of them "
                         "when they exceed DUMP_BYTES) to DIR/<name>.npy as float32")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.steps < 1):
        ap.error("--dump-outputs needs --impl b200 and --steps >= 1")
    return args


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the benchmark runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []  # (phase, sm_mhz, reasons)
        self.phase = "warmup"
        self.stop_flag = False
        self.sm_max = None
        self.ok = False

    def run(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            self.ok = True
            while not self.stop_flag:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append((self.phase, sm, r))
                time.sleep(0.002)
        except Exception:
            self.ok = False

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": ["unavailable"]}
        timed = [s for s in self.samples if s[0] == "timed"] or [s for s in self.samples if s[0] != "idle"]
        names = {
            0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x10: "sync_boost",
            0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown",
            0x100: "display_clock_setting",
        }
        mask = 0
        for s in timed:
            mask |= s[2]
        return {
            "sm_mhz": statistics.median(s[1] for s in timed),
            "sm_max_mhz": self.sm_max,
            "reasons": sorted(n for b, n in names.items() if mask & b),
            "samples": len(timed),
        }


def cpu_baseline(rows, mrl, seconds_target=12.0):
    """The CPU oracle (C restatement of the reference path) on all host threads, bounded sample."""
    from ac_solver_b200.synthetic import random_actions, random_presentations
    from oracle import oracle as O

    S = random_presentations(rows, mrl, seed=0)
    sc = np.zeros(rows, np.int32)
    A = random_actions(rows, seed=1)
    threads = host_threads()  # torchrun pins OMP_NUM_THREADS=1: ask for every core explicitly
    O.env_step_batch(S, A, sc, HORIZON, nthreads=threads)  # warm
    t0 = time.perf_counter()
    reps = 0
    while True:
        O.env_step_batch(S, A, sc, HORIZON, nthreads=threads)
        reps += 1
        if time.perf_counter() - t0 > seconds_target or reps >= 2000:
            break
    dt = time.perf_counter() - t0
    return {
        "value": rows * reps / dt,
        "unit": "moves/s",
        "cores": threads,
        "kind": "port",
        "sample": f"{reps} passes of ACEnv.step over {rows} synthetic rows (mrl {mrl}), C oracle, {threads} OpenMP threads",
    }


def _py_worker(job):
    """One process of the pure-Python baseline: ACMove(cyclical=True) of the STAGED reference
    (baseline/_ref, the reference's own modules) over a slice of rows for a fixed time."""
    rows, actions, mrl, seconds = job
    sys.path.insert(0, os.path.join(ROOT, "baseline", "_ref"))
    from ac_solver.envs.ac_moves import ACMove  # the reference's function, unmodified

    n, t0, i = 0, time.perf_counter(), 0
    while time.perf_counter() - t0 < seconds:
        r = rows[i % len(rows)]
        lens = [int(np.count_nonzero(r[:mrl])), int(np.count_nonzero(r[mrl:]))]
        try:
            ACMove(int(actions[i % len(rows)]), r, mrl, lens, cyclical=True)
        except AssertionError:
            pass  # the reference raises when a move empties a relator
        n += 1
        i += 1
    return n, time.perf_counter() - t0


def _py_greedy_worker(job):
    """The reference's own greedy_search (baseline/_ref) on one presentation at a small budget."""
    import contextlib
    import io

    pres, budget = job
    sys.path.insert(0, os.path.join(ROOT, "baseline", "_ref"))
    from ac_solver.search.greedy import greedy_search as ref_greedy

    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        ref_greedy(np.array(pres), max_nodes_to_explore=budget)
    return time.perf_counter() - t0


def _py_bfs_worker(job):
    """The reference's own bfs (baseline/_ref) on one presentation; returns seconds (one core)."""
    import contextlib
    import io

    pres, budget = job
    sys.path.insert(0, os.path.join(ROOT, "baseline", "_ref"))
    from ac_solver.search.breadth_first import bfs as ref_bfs

    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        ref_bfs(np.array(pres), max_nodes_to_explore=budget)
    return time.perf_counter() - t0


def python_pool_map(fn, jobs, procs, timeout=180.0):
    """Run fn over jobs in fresh interpreters (spawn); None if the staged reference is missing or anything fails."""
    if not os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "ac_solver")):
        return None
    import multiprocessing as mp

    try:
        with mp.get_context("spawn").Pool(max(1, min(procs, len(jobs)))) as pool:
            return pool.map_async(fn, jobs).get(timeout=timeout)  # bounded: an auxiliary baseline must never hang the bench
    except Exception:
        return None


def cpu_baseline_python(rows, mrl, seconds=8.0):
    """The reference's own pure-Python ACMove on every host core (BASELINE.md section 3), bounded sample."""
    if not os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "ac_solver")):
        return {"unavailable": "baseline/_ref not staged (run __graft_entry__.build() where /root/reference exists)"}
    import multiprocessing as mp

    from ac_solver_b200.synthetic import random_actions, random_presentations

    cores = host_threads()
    S = random_presentations(rows, mrl, seed=0)
    A = random_actions(rows, seed=1)
    per = max(1, rows // cores)
    jobs = [(S[k * per:(k + 1) * per], A[k * per:(k + 1) * per], mrl, seconds) for k in range(cores) if len(S[k * per:(k + 1) * per])]
    try:
        with mp.get_context("spawn").Pool(len(jobs)) as pool:
            out = pool.map(_py_worker, jobs)
    except Exception as e:  # the baseline is auxiliary: never lose the headline line
        return {"unavailable": repr(e)}
    total = sum(n for n, _ in out)
    dt = max(t for _, t in out)
    return {"value": total / dt, "unit": "moves/s", "cores": len(jobs), "kind": "reference",
            "per_core": total / dt / len(jobs),
            "sample": f"the reference's own ACMove(cyclical=True) (baseline/_ref, pure Python) over the first {rows} "
                      f"synthetic rows (mrl {mrl}), {len(jobs)} processes x {seconds:.0f} s"}


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    from ac_solver_b200.synthetic import random_actions, random_presentations
    from oracle import oracle as O

    rows, mrl = args.cpu_sample_rows, args.mrl
    S = random_presentations(rows, mrl, seed=0)
    A = random_actions(rows, seed=1)
    sc = np.zeros(rows, np.int32)
    threads = host_threads()  # torchrun pins OMP_NUM_THREADS=1: ask for every core explicitly
    w0 = time.perf_counter()  # warm for >= 1.5 s: thread pool, page tables and caches in steady state
    for _ in range(max(args.warmup, 1)):
        O.env_step_batch(S, A, sc, HORIZON, nthreads=threads)
    while time.perf_counter() - w0 < 1.5:
        O.env_step_batch(S, A, sc, HORIZON, nthreads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        O.env_step_batch(S, A, sc, HORIZON, nthreads=threads)
    dt = time.perf_counter() - t0
    v = rows * args.steps / dt
    sample = f"each step = ACEnv.step over a {rows}-row sample of the 1 Mi-row workload, C oracle on {threads} host threads"
    line = {
        "impl": "reference", "metric": "AC moves/sec (batched env steps)", "value": v, "unit": "moves/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int8", "data": "synthetic",
        "config": {"workload": f"batched ACEnv.step, {rows}-row sample of 1Mi rows, mrl {mrl}, uniform 12 moves, CPU"},
        "cpu_baseline": {"value": v, "unit": "moves/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "moves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def bind_to_gpu_numa_node(local_rank):
    """One process per GPU: run on (and first-touch the pinned buffers from) the host cores of the NUMA node the
    GPU hangs off, so that the e2e copies of N ranks do not all land in one socket's memory.  Best effort: returns
    what was done (or why not) for the JSON line."""
    try:
        import torch

        p = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            # sysfs knows nothing (containers often hide it): ask NVML for the GPU's ideal CPU set
            import pynvml

            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByPciBusId(bdf.encode() if hasattr(bdf, "encode") else bdf)
            ncpu = os.cpu_count() or 1
            words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
            cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
            allowed = os.sched_getaffinity(0)
            use = cpus & allowed
            if not use or use == allowed:
                return {"node": None, "why": "neither sysfs nor NVML reports a CPU affinity narrower than this process's mask"}
            os.sched_setaffinity(0, use)
            return {"node": "nvml", "cores": len(use), "gpu": bdf}
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        if not use:
            return {"node": node, "why": "none of the node's cores are in this process's affinity mask"}
        os.sched_setaffinity(0, use)
        return {"node": node, "cores": len(use), "gpu": bdf}
    except Exception as e:  # sysfs layout, permissions: keep going unbound
        return {"node": None, "why": repr(e)}


def run_b200(args):
    import torch

    rank, local_rank, world = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the AC-move kernels have no CPU fallback")
    # stdout carries exactly ONE JSON line: libraries that chat on fd 1 (NCCL prints its version
    # banner there) are sent to stderr until the line is printed.
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("cpu:gloo,cuda:nccl", device_id=torch.device("cuda", local_rank))

    from ac_solver_b200 import _lib
    from ac_solver_b200.synthetic import random_actions, random_presentations

    L = _lib.lib()
    ctx = _lib.ctx(local_rank)
    rows, mrl = args.rows, args.mrl
    rowb = 2 * mrl
    nbuf = max(4, -(-3 * L2_BYTES // (rows * rowb)) + 1)  # rotated state buffers: working set > L2
    base = random_presentations(min(rows, 1 << 18), mrl, seed=rank)
    reps = -(-rows // len(base))
    host_states = np.tile(base, (reps, 1))[:rows]
    states = [torch.from_numpy(np.roll(host_states, 7919 * b, axis=0).copy()).cuda() for b in range(nbuf)]
    actions = [torch.from_numpy(random_actions(rows, seed=1 + 17 * b + rank)).cuda() for b in range(nbuf)]
    reward = torch.zeros(rows, dtype=torch.int32, device="cuda")
    done = torch.zeros(rows, dtype=torch.uint8, device="cuda")
    trunc = torch.zeros(rows, dtype=torch.uint8, device="cuda")
    stepc = [torch.zeros(rows, dtype=torch.int32, device="cuda") for _ in range(nbuf)]
    # ACEnv keeps `lengths` beside `state` (ac_env.py:84-92): so does the batched env (2 B per row)
    lens = [torch.stack([(s[:, :mrl] != 0).sum(1), (s[:, mrl:] != 0).sum(1)], dim=1).to(torch.uint8).contiguous()
            for s in states]
    err = torch.tensor([0, -1], dtype=torch.int64, device="cuda")
    stream = torch.cuda.current_stream()
    sptr = stream.cuda_stream

    def step(i, flags=FLAGS):
        b = i % nbuf
        rc = L.acs_env_step_batch(states[b].data_ptr(), actions[(i // nbuf + b) % nbuf].data_ptr(), reward.data_ptr(),
                                  done.data_ptr(), trunc.data_ptr(), stepc[b].data_ptr(), lens[b].data_ptr(), None,
                                  err.data_ptr(), rows, mrl, HORIZON, flags, sptr)
        if rc != 0:
            _lib.check(rc)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    for i in range(args.warmup):
        step(i)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.phase = "timed"
    ev0.record(stream)
    for i in range(args.steps):
        step(args.warmup + i)
    ev1.record(stream)
    torch.cuda.synchronize()
    sampler.phase = "post"
    if args.dump_outputs and rank == 0:
        b = (args.warmup + args.steps - 1) % nbuf  # the buffers the last timed step updated in place
        dump_outputs(args.dump_outputs, state=states[b], reward=reward, done=done, truncated=trunc, step_count=stepc[b],
                     lengths=lens[b])
    ms = ev0.elapsed_time(ev1)
    if dist is not None:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    barrier()
    n_bad = int(err[0].item())

    # ---- the general variant (flags = 0: full validate + simplify of both relators, lengths recounted),
    # what a caller gets from ac_moves_batch / a first step on caller-supplied states ----
    gen_steps = max(20, min(args.steps // 4, 400))
    for i in range(10):
        step(i, 0)
    barrier()
    gv0, gv1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    gv0.record(stream)
    for i in range(gen_steps):
        step(10 + i, 0)
    gv1.record(stream)
    torch.cuda.synchronize()
    ms_general = gv0.elapsed_time(gv1) / gen_steps
    if dist is not None:
        t = torch.tensor([ms_general], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_general = float(t.item())
    barrier()

    # ---- in-run parity (BASELINE.md section 3): the first 131 072 rows of the batch, one step with each
    # kernel variant, every output against the CPU oracle ----
    parity = None
    if rank == 0:
        from oracle import oracle as O

        pn = min(rows, 1 << 17)
        ps = np.ascontiguousarray(host_states[:pn])
        pa = random_actions(pn, seed=1)
        exp_state = ps.copy()
        exp_sc = np.full(pn, HORIZON - 1, np.int32)  # the step reaches the horizon: truncated is exercised too
        er, ed, et, el, es = O.env_step_batch(exp_state, pa, exp_sc, HORIZON, nthreads=host_threads())
        mism = 0
        for flags in sorted({FLAGS, 0}):
            d_s = torch.from_numpy(ps.copy()).cuda()
            d_a = torch.from_numpy(pa).cuda()
            d_r = torch.zeros(pn, dtype=torch.int32, device="cuda")
            d_d = torch.zeros(pn, dtype=torch.uint8, device="cuda")
            d_t = torch.zeros(pn, dtype=torch.uint8, device="cuda")
            d_c = torch.full((pn,), HORIZON - 1, dtype=torch.int32, device="cuda")
            d_l = torch.stack([(d_s[:, :mrl] != 0).sum(1), (d_s[:, mrl:] != 0).sum(1)], dim=1).to(torch.uint8).contiguous()
            d_st = torch.zeros(pn, dtype=torch.uint8, device="cuda")
            _lib.check(L.acs_env_step_batch(d_s.data_ptr(), d_a.data_ptr(), d_r.data_ptr(), d_d.data_ptr(), d_t.data_ptr(),
                                            d_c.data_ptr(), d_l.data_ptr(), d_st.data_ptr(), None, pn, mrl, HORIZON, flags, sptr))
            torch.cuda.synchronize()
            ok = es == 0
            bad = (d_s.cpu().numpy() != exp_state).any(axis=1) | (d_st.cpu().numpy() != es)
            bad |= ok & ((d_r.cpu().numpy() != er) | (d_d.cpu().numpy() != ed) | (d_t.cpu().numpy() != et)
                         | (d_c.cpu().numpy() != exp_sc) | (d_l.cpu().numpy() != el).any(axis=1))
            mism += int(bad.sum())
        parity = {"rows": pn, "variants_checked": sorted({FLAGS, 0}), "mismatches": mism, "rows_raising": int((es != 0).sum()),
                  "checked": "next state, reward, done, truncated, step counter, lengths, per-row status vs the CPU oracle"}

    # ---- e2e: the vector-env call with HOST buffers (actions in; obs, reward, flags out) ----
    e2e_steps = max(3, min(args.steps, 30))
    h_act = [torch.from_numpy(random_actions(rows, seed=100 + b + rank)).pin_memory() for b in range(2)]
    h_obs = torch.empty((rows, rowb), dtype=torch.int8).pin_memory()
    h_rew = torch.empty(rows, dtype=torch.int32).pin_memory()
    h_done = torch.empty(rows, dtype=torch.uint8).pin_memory()
    h_tr = torch.empty(rows, dtype=torch.uint8).pin_memory()
    nbad = C.c_int64(0)

    def e2e_step(i):
        b = i % nbuf
        _lib.check(L.acs_env_step_host(ctx, states[b].data_ptr(), stepc[b].data_ptr(), h_act[i % 2].data_ptr(),
                                       h_obs.data_ptr(), h_rew.data_ptr(), h_done.data_ptr(), h_tr.data_ptr(),
                                       rows, mrl, HORIZON, FLAGS, C.byref(nbad)))

    for i in range(3):
        e2e_step(i)
    barrier()
    sampler.phase = "e2e"
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        e2e_step(i)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    sampler.phase = "post"
    if dist is not None:
        t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    # what the PCIe link gives a plain pinned device->host copy of the same observation buffer on this box:
    # the e2e call moves 78 B per move to the host, so this bandwidth bounds it
    torch.cuda.synchronize()
    d2h_t = []
    for _ in range(5):
        c0 = time.perf_counter()
        h_obs.copy_(states[0], non_blocking=True)
        torch.cuda.synchronize()
        d2h_t.append(time.perf_counter() - c0)
    d2h_gbps = rows * rowb / min(d2h_t) / 1e9
    sampler.stop_flag = True
    sampler.join(timeout=2)

    single = None
    if rank == 0 and world == 1:
        # the reference's one-presentation-at-a-time API through the GPU (latency, not throughput: H2D + kernel + D2H +
        # stream sync per call); reported so that nobody mistakes the drop-in single calls for the fast path
        from ac_solver_b200.envs.ac_moves import ACMove

        p0 = host_states[0].copy()
        ln = [int((p0[:mrl] != 0).sum()), int((p0[mrl:] != 0).sum())]
        for k in range(50):
            ACMove(k % 12, p0, mrl, ln)
        t0 = time.perf_counter()
        ncall = 2000
        for k in range(ncall):
            ACMove(k % 12, p0, mrl, ln)
        single = {"ACMove_us_per_call": 1e6 * (time.perf_counter() - t0) / ncall, "calls": ncall,
                  "note": "single-presentation ACMove(cyclical=True) through acs_generic_host; compare 1e6 / cpu_baseline_python.per_core"}

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        ms_per_step = ms / args.steps
        moves_per_s = world * rows * args.steps / (ms * 1e-3)
        algo_bytes = 4 * mrl + 6  # 2*mrl in + 2*mrl out + action 1 + reward 4 + done 1 (150 at mrl 36)
        achieved = algo_bytes * rows / (ms_per_step * 1e-3) / 1e9
        # the CPU baseline is timed on rank 0 at N=1 only (it would stall the other ranks)
        cpu = cpu_baseline(args.cpu_sample_rows, mrl) if world == 1 else None
        cpu_py = cpu_baseline_python(args.cpu_sample_rows, mrl) if (world == 1 and not args.skip_python_baseline) else None
        traffic, traffic_src = ncu_traffic()
        achieved_general = algo_bytes * rows / (ms_general * 1e-3) / 1e9
        line = {
            "metric": "AC moves/sec (batched env steps)",
            "value": moves_per_s,
            "unit": "moves/s",
            "n_gpus": world,
            "steps": args.steps,
            "warmup": args.warmup,
            "ms_per_step": ms_per_step,
            "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": None,
            "dtype": "int8",
            "data": "synthetic",
            "config": {
                "workload": f"batched ACEnv.step microbench: {rows} synthetic random presentations per GPU, "
                            f"max_relator_length {mrl}, uniform random over the 12 AC' moves, horizon {HORIZON} "
                            "(BASELINE.json configs[1])",
                "rows_per_gpu": rows,
                "l2": f"rotating {nbuf} distinct in-place state buffers ({nbuf * rows * rowb >> 20} MiB > 126 MiB L2)",
                "parallelism": f"{world} independent shards, no collective",
                "rows_raising": n_bad,
            },
            "roofline": {
                "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_move": 4 * mrl + 6,
                "kernel": ("acs::ac_step_words_kernel<NW=9, TRUSTED=%s, LENS=%s, TR=128>"
                           % (bool(FLAGS & 2), bool(FLAGS & 4))) if mrl == 36 else "acs::ac_step_*_kernel",
                "kernel_flags": FLAGS,
                "frac_of_nominal_8TBs": achieved / 8000.0,
                # what the kernel really moves per move with the lengths carried (FLAGS & 4): the algorithmic 4*mrl+6 plus the
                # step counter in and out (8), the two lengths in and out (4) and `truncated` (1)
                "real_bytes_per_move": (4 * mrl + 6 + 13) if (FLAGS & 4) else (4 * mrl + 6 + 11),
                "frac_real_traffic": achieved / peak * ((4 * mrl + 6 + 13) if (FLAGS & 4) else (4 * mrl + 6 + 11)) / (4 * mrl + 6),
            },
            "roofline_general": {
                "bound": "hbm", "achieved": achieved_general, "peak": peak, "unit": "GB/s", "frac": achieved_general / peak,
                "ms_per_step": ms_general, "steps": gen_steps, "kernel_flags": 0,
                "kernel": "the general variant: reference's full validate + simplify of both relators, lengths recounted",
            },
            "parity": parity,
            "cpu_baseline": cpu,
            "cpu_baseline_python": cpu_py,
            "e2e": {
                "value": world * rows * e2e_steps / e2e_s,
                "unit": "moves/s",
                "h2d_bytes_per_step": rows * 1,
                "d2h_bytes_per_step": rows * (rowb + 4 + 1 + 1),
                "steps": e2e_steps,
                "api": "acs_env_step_host: pinned host actions in; host observations, rewards, done, truncated out",
                "numa_binding_rank0": numa,
                "d2h_GBps_achieved": rows * (rowb + 6) * e2e_steps / e2e_s / 1e9,
                "pinned_d2h_GBps_measured": d2h_gbps,
                "frac_of_pinned_d2h": rows * (rowb + 6) * e2e_steps / e2e_s / 1e9 / d2h_gbps,
            },
            "single_call": single,
            "gpu_launches": args.steps,  # kernels of the timed region (one ac_step kernel per step)
            "clocks": sampler.summary(),
        }
    else:
        line = None

    def emit(extra=None, greedy=None):
        if rank == 0:
            if extra is not None:
                line["bfs"] = extra
            if greedy is not None:
                line["greedy"] = greedy
            sys.stdout.flush()
            os.dup2(real_stdout, 1)
            print(json.dumps(line), flush=True)

    # Secondary metrics (greedy sweep seconds, BFS nodes expanded/s).  At N > 1 the BFS is a multi-rank
    # program: a watchdog guarantees that the headline line is printed and every rank exits even if it stalls.
    bfs_line = greedy_line = None

    def bail():
        emit(bfs_line if bfs_line is not None else {"error": f"the search benches did not finish within {args.bfs_timeout} s"},
             greedy_line)
        os._exit(0)

    dog = threading.Timer(args.bfs_timeout, bail)
    dog.daemon = True
    dog.start()
    # the search legs first: they are the ones that are sensitive to the state earlier legs leave the device in
    # (measured: the greedy sweep takes 2.0-2.4 s right after the K1 legs, 3.8-4.8 s after the PPO / barcode legs)
    if not args.skip_greedy:
        try:
            greedy_line = bench_greedy(args, world, dist)
        except Exception as e:  # auxiliary: never lose the headline line
            greedy_line = {"error": repr(e)}
    if not args.skip_bfs:
        try:
            bfs_line = bench_bfs(args, world, dist)
        except Exception as e:
            bfs_line = {"error": repr(e)}
            if world > 1:  # ranks may be out of step now: no further collectives
                dog.cancel()
                emit(bfs_line, greedy_line)
                os._exit(0)
    if world == 1 and not args.skip_vecenv:
        try:
            line["vecenv"] = bench_vecenv(args)
        except Exception as e:
            line["vecenv"] = {"error": repr(e)}
    if world == 1:
        try:
            line["config1"] = bench_config1()
        except Exception as e:
            line["config1"] = {"error": repr(e)}
    if world == 1 and not args.skip_ppo:
        try:
            line["ppo"] = bench_ppo(args)
        except Exception as e:
            line["ppo"] = {"error": repr(e)}
    if world == 1 and not args.skip_barcode:
        try:
            line["barcode"] = bench_barcode(args)
        except Exception as e:
            line["barcode"] = {"error": repr(e)}
    dog.cancel()
    emit(bfs_line, greedy_line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def dump_outputs(out_dir, **outputs):
    """Each [rows, ...] device output to out_dir/<name>.npy as float32: every row, or the same seeded sample of rows
    for all outputs when every row would take more than DUMP_BYTES."""
    import torch

    rows = len(next(iter(outputs.values())))
    n = min(rows, DUMP_BYTES // (4 * sum(t[0].numel() for t in outputs.values())))
    idx = np.arange(rows) if n == rows else np.sort(np.random.default_rng(0).choice(rows, n, replace=False))
    idx = torch.from_numpy(idx)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.index_select(0, idx.to(t.device)).cpu().numpy().astype(np.float32))


def ncu_traffic():
    """DRAM bytes per launch of the step kernel from the latest committed ncu capture under
    profiles/ (dram__bytes_read.sum + dram__bytes_write.sum), with its provenance.  A single
    profiled launch under-counts writes still resident in L2 when the capture ends, so the
    round-2 summary averages >= 8 back-to-back launches (profiles/k1_step_r2_ncu_summary.json)."""
    for name in ("k1_step_r2_ncu_summary.json", "k1_step_r1_ncu_summary.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                d = json.load(f)
            if "traffic_bytes_per_launch" in d:
                return float(d["traffic_bytes_per_launch"]), d.get("source", name)
            m = d[sorted(d)[-1]]
            return ((float(m["dram__bytes_read.sum"]) + float(m["dram__bytes_write.sum"])) * 1e6,
                    f"profiles/{name} (single cold-cache launch; last tiles' write-back still in L2)")
        except Exception:
            continue
    return None, None


AK3 = np.array([1, 1, 1, -2, -2, -2, -2] + [0] * 17 + [1, 2, 1, -2, -1, -2] + [0] * 18, np.int8)
RANDOM_REQUEST_PEAK = 37.0e9  # measured on B200: scripts/microbench/random_access.cu (profiles/random_access_r2.jsonl)


def bench_bfs(args, world=1, dist=None):
    """Secondary metric: BFS nodes expanded / s on AK(3), mrl 24, budget 1e9 (BASELINE.json
    configs[4]) with the native hash-partitioned search (csrc/pbfs.cu): one GPU = a world of one;
    N GPUs = one process per GPU, newly generated states stored straight into the owner's inbox
    over NVLink (cudaIpc peer memory), same total budget (strong scaling).  Also, in the same run:
    bit-exact parity of a 1e6-budget search on the same ranks against the CPU oracle, and the
    roofline of the search (algorithmic bytes of SURVEY 8d with the measured u)."""
    import torch

    from ac_solver_b200.search.partitioned import PartitionedBfs

    rank = dist.get_rank() if dist is not None else 0

    def sync():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    # ---- parity on the same ranks: visited ARRAY in insertion order, path, counters ----
    parity_budget = 1_000_000
    with PartitionedBfs(24, parity_budget) as eng:
        solved, path, info = eng.run(AK3, want_visited=True)
    parity = None
    if rank == 0:
        from oracle import oracle as O

        es, ep, ei = O.bfs(AK3, parity_budget, want_visited=True)
        same = (solved, path) == (es, ep) and all(info[k] == ei[k] for k in
                                                    ("n_visited", "n_expanded", "n_moves", "budget_hit", "minlen_log"))
        vis_ok = info["visited"].shape == ei["visited"].shape and bool(np.array_equal(info["visited"], ei["visited"]))
        parity = {"budget": parity_budget, "world": world, "visited_rows_compared": int(ei["n_visited"]),
                  "mismatches": 0 if (same and vis_ok) else int((info["visited"][: len(ei["visited"])] != ei["visited"][: len(info["visited"])]).any(axis=1).sum()) + (0 if same else 1),
                  "checked": "result, path, counters, minimal-length log and the visited array in insertion order vs the CPU oracle"}
    # ---- timed search ----
    with PartitionedBfs(24, args.bfs_budget) as eng:
        eng.run(AK3)  # warm-up: first touch of the buffers, peer mappings
        sync()
        t0 = time.perf_counter()
        solved, path, info = eng.run(AK3)
        sync()
        wall = time.perf_counter() - t0
    t = torch.tensor([wall, info["seconds_device"]], device="cuda", dtype=torch.float64)
    recs = torch.tensor([float(info["records_sent"][0]), float(info["records_recv"][0])], device="cuda", dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(recs, op=dist.ReduceOp.SUM)
    wall, dev_s = float(t[0]), float(t[1])
    if rank != 0:
        return None
    expanded, visited = info["n_expanded"], info["n_visited"]
    records = float(recs[0])
    u = visited / max(expanded, 1)
    peak, peak_src = measured_peak_gbs()
    # SURVEY 8d: parent read 2*mrl + 12 probes x 16 B key + u x (key insert 16 + frontier append 2*mrl + parent record 8)
    bytes_per_exp = 2 * 24 + 12 * 16 + u * (16 + 2 * 24 + 8)
    achieved = bytes_per_exp * expanded / dev_s / 1e9
    # the insert kernel is bound by random memory REQUESTS, not bytes: one bucket load per record, one log-key
    # load per duplicate, one CAS per new state (an atomic costs ~1.85 loads at the measured 20 G atomics/s)
    dup = max(records - visited, 0.0)
    req_per_exp = (records + dup + 1.85 * visited) / max(expanded, 1)
    out = {
        "metric": "BFS nodes expanded/sec",
        "workload": f"bfs AK(3) mrl 24 budget {args.bfs_budget} (BASELINE.json configs[4]), {world} GPU(s), hash-partitioned, "
                    "native driver (csrc/pbfs.cu): expansion fused with the NVLink exchange (peer stores), no host syncs per chunk",
        "n_gpus": world, "nodes_expanded": expanded, "visited": visited, "levels": info["n_levels"], "chunks": info["chunks"],
        "expanded_per_s_device": expanded / dev_s, "visited_per_s_device": visited / dev_s, "seconds_device": dev_s,
        "expanded_per_s_wall": expanded / wall, "seconds_wall": wall, "scaling": "strong",
        "new_states_per_expansion_u": u, "records_per_expansion": records / max(expanded, 1),
        "parity": parity,
        "roofline": {"bound": "hbm", "bytes_per_expansion": bytes_per_exp, "achieved": achieved, "peak": peak * world,
                     "unit": "GB/s", "frac": achieved / (peak * world), "traffic": bfs_traffic(world), "peak_source": peak_src,
                     "note": "algorithmic bytes of SURVEY 8d with the measured u; the search is bound by random-access "
                             "REQUESTS (request_roofline), not by bytes"},
        "request_roofline": {"bound": "random 32-byte memory requests", "requests_per_expansion": req_per_exp,
                             "achieved": req_per_exp * expanded / dev_s / 1e9, "peak": RANDOM_REQUEST_PEAK * world / 1e9,
                             "unit": "G requests/s", "frac": req_per_exp * expanded / dev_s / (RANDOM_REQUEST_PEAK * world),
                             "peak_source": "measured, scripts/microbench/random_access.cu on B200 (profiles/random_access_r2.jsonl)"},
        "nvlink": None if world == 1 else {
            "bytes_sent_per_expansion": records * (world - 1) / world * 20 / max(expanded, 1),
            "GBps_per_gpu": records * (world - 1) / world * 20 / world / dev_s / 1e9, "peak_GBps_per_gpu_per_direction": 900.0},
    }
    if world == 1:
        from oracle import oracle as O

        c0 = time.perf_counter()
        _, _, cinfo = O.bfs(AK3, 2_000_000)
        cpu_s = time.perf_counter() - c0
        out["cpu_baseline"] = {"value": cinfo["n_expanded"] / cpu_s, "unit": "nodes expanded/s", "cores": 1, "kind": "port",
                               "sample": "C oracle bfs, same presentation, budget 2e6 (sequential algorithm, one core)"}
        if not getattr(args, "skip_python_baseline", False):
            # BASELINE.md section 3, config 5: the reference's own bfs on AK(3) at budget 1e5, one core
            pyb = 100_000
            secs = python_pool_map(_py_bfs_worker, [(AK3.tolist(), pyb)], 1)
            if secs:
                _, _, pinfo = O.bfs(AK3, pyb)  # the same run through the oracle: how many nodes that budget expands
                out["cpu_baseline_python"] = {"value": pinfo["n_expanded"] / secs[0], "unit": "nodes expanded/s", "cores": 1,
                                              "kind": "reference", "visited_per_s": pinfo["n_visited"] / secs[0],
                                              "sample": f"the reference's own bfs (baseline/_ref, pure Python) on AK(3) at budget {pyb}: "
                                                        f"{secs[0]:.1f} s on one core, {pinfo['n_expanded']} nodes expanded"}
    return out


def bench_greedy(args, world=1, dist=None):
    """BASELINE.json configs[2]: greedy_search over all 1190 Miller-Schupp presentations of the shipped
    all_presentations.txt, 1e6 nodes each, batched per max_relator_length group (one CTA per search).
    N GPUs: the searches are independent and are dealt round-robin to the ranks (no collective).
    Checked in the run: 533 solved and every stored reference path reproduced (greedy_search_paths.txt
    holds action+1), 657 failures.  CPU baseline beside it: the C oracle on all host cores."""
    import torch
    from ast import literal_eval
    from concurrent.futures import ThreadPoolExecutor

    from ac_solver_b200.search.greedy import greedy_search_batch  # noqa: F401  (kept for interactive use)

    data = os.path.join(ROOT, "ac_solver_b200", "search", "miller_schupp", "data")
    with open(os.path.join(data, "all_presentations.txt")) as f:
        pres = [np.array(literal_eval(line), dtype=np.int8) for line in f if line.strip()]
    with open(os.path.join(data, "greedy_search_paths.txt")) as f:
        stored = [[(int(a) - 1, int(l)) for a, l in literal_eval(line)] for line in f if line.strip()]
    rank = dist.get_rank() if dist is not None else 0
    budget = args.greedy_budget
    groups = {}
    for k, p in enumerate(pres):
        if k % world == rank:
            groups.setdefault(p.size, []).append(k)

    from ac_solver_b200.search.greedy import greedy_search_groups

    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    mine, dev_s = {}, 0.0
    group_rows = list(groups.values())
    # engines are created first, then the length groups search concurrently (one stream each), see greedy_search_groups
    for rows, out in zip(group_rows, greedy_search_groups([np.stack([pres[k] for k in rows]) for rows in group_rows], budget)):
        dev_s = max(dev_s, out[0][2]["seconds_device"])
        for k, (solved, path, info) in zip(rows, out):
            mine[k] = (solved, path, info["n_visited"], info["n_expanded"], info["rounds"])
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    if dist is not None:
        gathered = [None] * world if rank == 0 else None
        dist.gather_object((mine, dev_s, wall), gathered, dst=0)
        if rank != 0:
            return None
        mine = {k: v for part, _, _ in gathered for k, v in part.items()}
        dev_s = max(d for _, d, _ in gathered)
        wall = max(w for _, _, w in gathered)
    n_solved = sum(1 for v in mine.values() if v[0])
    paths_ok = sum(1 for k in range(len(stored)) if mine[k][0] and mine[k][1] == stored[k])
    visited = sum(v[2] for v in mine.values())
    out = {
        "metric": "greedy sweep seconds (1190 Miller-Schupp presentations, budget 1e6 each)",
        "workload": "BASELINE.json configs[2]; one CTA per search, bucket-batched speculative pops (csrc/greedy_bucket.cuh)",
        "n_gpus": world, "budget": budget, "seconds_wall": wall, "seconds_device_max_group": dev_s,
        "visited_total": visited, "visited_per_s_wall": visited / wall,
        "parity": {"solved": n_solved, "expected_solved": len(stored), "stored_paths_reproduced": paths_ok,
                   "failures": len(pres) - n_solved, "solved_rows_beyond_533": sum(1 for k in range(len(stored), len(pres)) if mine[k][0]),
                   "checked": "every stored reference path (greedy_search_paths.txt, action+1 convention) reproduced exactly"},
        "heap_kernel_fallbacks": sum(1 for v in mine.values() if v[4] < 0),
    }
    if world == 1:
        from oracle import oracle as O

        cores = host_threads()
        unsolved = list(range(len(stored), len(pres)))
        sample = unsolved[:: max(1, len(unsolved) // (2 * cores))][: 2 * cores]
        c0 = time.perf_counter()
        with ThreadPoolExecutor(max_workers=cores) as tp:
            cv = list(tp.map(lambda k: O.greedy_search(pres[k], budget)[2]["n_visited"], sample))
        cs = time.perf_counter() - c0
        est = cs / len(sample) * len(unsolved)
        out["cpu_baseline"] = {"value": est, "unit": "s (extrapolated sweep)", "cores": cores, "kind": "port",
                               "sample": f"C oracle greedy_search on {len(sample)} of the {len(unsolved)} unsolved rows at budget "
                                         f"{budget}, one search per thread on {cores} threads: {cs:.1f} s; the 533 solved rows are cheap",
                               "speedup_vs_allcore_port_wall": est / wall, "speedup_vs_allcore_port_device": est / dev_s}
        if not getattr(args, "skip_python_baseline", False):
            # BASELINE.md section 3, config 3: the reference's own greedy_search on 16 sampled unsolved rows at budget 1e4,
            # spread over the host cores, extrapolated linearly in the budget to 1e6 x 657 unsolved rows
            pyb = 10_000
            psample = unsolved[:: max(1, len(unsolved) // 16)][:16]
            p0 = time.perf_counter()
            secs = python_pool_map(_py_greedy_worker, [(pres[k].tolist(), pyb) for k in psample], cores)
            if secs:
                per_row = sum(secs) / len(secs) * (budget / pyb)
                out["cpu_baseline_python"] = {
                    "value": per_row * len(unsolved) / cores, "unit": "s (extrapolated sweep, all cores)", "cores": cores, "kind": "reference",
                    "core_seconds_per_unsolved_row_at_budget": per_row,
                    "sample": f"the reference's own greedy_search (baseline/_ref) on {len(psample)} unsolved rows at budget {pyb}: "
                              f"{sum(secs) / len(secs):.2f} core-s per row ({time.perf_counter() - p0:.1f} s wall on {cores} cores); "
                              f"EXTRAPOLATED x{budget // pyb} in the budget and to the {len(unsolved)} unsolved rows"}
    return out


def bench_vecenv(args):
    """BASELINE.json configs[3]: PPO rollout, environment side -- 4096 GPU-resident environments, horizon
    200, the reference's 2x512 tanh actor (agents/ppo_agent.py:39-49) sampling actions on the device, reward
    NormalizeReward + clip and the curriculum reset of training.py:169-224 all on the device; policy forward,
    sampling, env step, reset and reward transform are ONE CUDA graph.  Reported: environment steps / s.
    CPU beside it: the C oracle stepping the same 4096 rows, and the reference's own ACEnv.step loop."""
    import torch
    from ast import literal_eval

    from ac_solver_b200.envs.vector_env import ACVectorEnv

    n_envs, horizon, replays = 4096, 200, 1000
    data = os.path.join(ROOT, "ac_solver_b200", "search", "miller_schupp", "data", "all_presentations.txt")
    with open(data) as f:
        rows = [np.array(literal_eval(line), dtype=np.int8) for line in f if line.strip()]
    pad = np.zeros((len(rows), 72), np.int8)
    for k, r in enumerate(rows):  # change_max_relator_length_of_presentation(., 36) (environment.py:88-93)
        m = r.size // 2
        pad[k, :m], pad[k, 36 : 36 + m] = r[:m], r[m:]
    pool = pad[np.arange(2 * n_envs) % len(pad)]
    env = ACVectorEnv(pool[:n_envs], horizon_length=horizon, clip_rewards=(-10, 1000), norm_rewards=True, gamma=0.99)
    env.reset()
    env.enable_curriculum(pool, repeat_solved_prob=0.25, seed=0)
    torch.manual_seed(0)
    actor = torch.nn.Sequential(torch.nn.Linear(72, 512), torch.nn.Tanh(), torch.nn.Linear(512, 512), torch.nn.Tanh(),
                                torch.nn.Linear(512, 12)).cuda()

    from ac_solver_b200 import _lib as _L

    lib = _L.lib()
    dev = env.dev
    # Categorical sampling (Gumbel-max) + the rollout record of one step in ONE kernel (csrc/ppo_kernels.cu), as in
    # agents/training.py; the record buffers hold a single time slot here
    ctr = torch.zeros(2, dtype=torch.int64, device=dev)
    rec_obs = torch.zeros((1, n_envs, 72), dtype=torch.int8, device=dev)
    rec_f = [torch.zeros((1, n_envs), device=dev) for _ in range(3)]
    rec_act = torch.zeros((1, n_envs), dtype=torch.int64, device=dev)
    act8 = torch.zeros(n_envs, dtype=torch.uint8, device=dev)
    zeros_n = torch.zeros(n_envs, device=dev)

    def rollout_step():
        with torch.no_grad():
            logits = actor(env.state.float())
            _L.check(lib.acs_rollout_sample_record(
                env.state.data_ptr(), zeros_n.data_ptr(), logits.data_ptr(), zeros_n.data_ptr(), ctr.data_ptr(), rec_obs.data_ptr(),
                rec_f[0].data_ptr(), rec_f[1].data_ptr(), rec_f[2].data_ptr(), rec_act.data_ptr(), act8.data_ptr(), n_envs, 1, 72, 12, 7,
                torch.cuda.current_stream(dev).cuda_stream))
            ctr[1:2].add_(1)  # next draw; the time slot stays 0
            env.step_device(act8)
            return env.transformed_reward()

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            rollout_step()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        rollout_step()
    for _ in range(20):
        graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(replays):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    env.check_errors()
    # the environment side alone (no policy): actions drawn on the device, same step / reward wrappers / curriculum
    def env_only_step():
        env.step_device(torch.randint(0, 12, (n_envs,), device=env.dev, dtype=torch.uint8))
        return env.transformed_reward()

    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            env_only_step()
    torch.cuda.current_stream().wait_stream(side)
    graph2 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph2):
        env_only_step()
    for _ in range(20):
        graph2.replay()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(replays):
        graph2.replay()
    e1.record()
    torch.cuda.synchronize()
    ms_env = e0.elapsed_time(e1)
    env.check_errors()
    c = env.curriculum_counters()
    out = {
        "metric": "PPO rollout env steps/sec (env side)", "workload": "BASELINE.json configs[3]: 4096 envs, horizon 200, "
        "torch 2x512 actor on device, fused sampling kernel, device-side NormalizeReward+clip and curriculum reset, one CUDA graph per vector step",
        "env_steps_per_s": n_envs * replays / (ms * 1e-3), "us_per_vector_step": 1e3 * ms / replays,
        "episodes_finished": c["episodes"], "states_solved": c["n_solved"], "host_syncs_per_step": 0,
        "env_only_steps_per_s": n_envs * replays / (ms_env * 1e-3), "env_only_us_per_vector_step": 1e3 * ms_env / replays,
        "env_only_note": "same graph without the actor: random actions drawn on the device; the policy GEMMs (fp32, cuBLAS) are the rest",
    }
    from oracle import oracle as O

    S, sc = pool[:n_envs].copy(), np.zeros(n_envs, np.int32)
    A = np.random.default_rng(0).integers(0, 12, size=n_envs).astype(np.uint8)
    for threads in (1, host_threads()):
        O.env_step_batch(S, A, sc, horizon, nthreads=threads)
        t0, reps = time.perf_counter(), 0
        while time.perf_counter() - t0 < 1.0:
            O.env_step_batch(S, A, sc, horizon, nthreads=threads)
            reps += 1
        out[f"cpu_port_env_steps_per_s_{threads}_threads"] = n_envs * reps / (time.perf_counter() - t0)
    try:  # the reference's own ACEnv.step loop (pure Python), 64 environments x 200 steps, one core
        sys.path.insert(0, os.path.join(ROOT, "baseline", "_ref"))
        from ac_solver.envs.ac_env import ACEnv, ACEnvConfig

        envs = [ACEnv(ACEnvConfig(initial_state=pool[k].copy(), horizon_length=horizon)) for k in range(64)]
        rng = np.random.default_rng(1)
        t0, steps = time.perf_counter(), 0
        for _ in range(200):
            for e in envs:
                try:
                    _, _, d, tr, _ = e.step(int(rng.integers(0, 12)))
                except AssertionError:
                    d = True
                if d or tr:
                    e.reset()
                steps += 1
        out["cpu_baseline_python"] = {"value": steps / (time.perf_counter() - t0), "unit": "env steps/s", "cores": 1,
                                      "kind": "reference", "sample": "the reference's ACEnv.step, 64 envs x 200 steps, one core"}
    except Exception as e:
        out["cpu_baseline_python"] = {"unavailable": repr(e)}
    return out


def bench_config1():
    """BASELINE.json configs[0]: bfs() on the README presentation AK(2), default budget 10 000 -- the reference's own
    CPU-runnable case.  Value is parity (result, visited count; the visited array is pinned by the tests), the wall time
    of the drop-in call is reported beside the reference's own bfs() (pure Python, staged under baseline/_ref) and the C
    oracle."""
    import contextlib
    import io

    from ac_solver_b200 import bfs
    from ac_solver_b200.search.breadth_first import bfs_device
    from oracle import oracle as O

    ak2 = np.array([1, 1, -2, -2, -2, 0, 0, 1, 2, 1, -2, -1, -2, 0])
    with contextlib.redirect_stdout(io.StringIO()):
        bfs(ak2)  # warm-up
        t0 = time.perf_counter()
        reps = 20
        for _ in range(reps):
            res = bfs(ak2)
        gpu_s = (time.perf_counter() - t0) / reps
        _, _, info = bfs_device(ak2.astype(np.int8), 10000)
    t0 = time.perf_counter()
    es, ep, ei = O.bfs(ak2, 10000)
    port_s = time.perf_counter() - t0
    out = {"workload": "bfs([1,1,-2,-2,-2,0,0,1,2,1,-2,-1,-2,0]) with the default max_nodes_to_explore=10000",
           "result": [bool(res[0]), res[1]], "visited": int(info["n_visited"]), "expanded": int(info["n_expanded"]),
           "parity": {"result_equals_oracle": (bool(res[0]), res[1]) == (bool(es), ep), "visited_equals_oracle": int(info["n_visited"]) == int(ei["n_visited"]),
                      "expected": "(False, None), 10002 visited (SURVEY 8d)"},
           "seconds_per_call": gpu_s, "c_port_seconds": port_s}
    try:
        sys.path.insert(0, os.path.join(ROOT, "baseline", "_ref"))
        from ac_solver.search.breadth_first import bfs as ref_bfs

        with contextlib.redirect_stdout(io.StringIO()):
            t0 = time.perf_counter()
            rr = ref_bfs(ak2.copy(), max_nodes_to_explore=10000)
            out["reference_python_seconds"] = time.perf_counter() - t0
        out["parity"]["result_equals_reference_python"] = (bool(rr[0]), rr[1]) == (bool(res[0]), res[1])
    except Exception as e:
        out["reference_python_seconds"] = None
        out["reference_python_error"] = repr(e)
    return out


def bench_ppo(args):
    """SURVEY 8f-4: the whole PPO iteration on the device at BASELINE.json configs[3]'s size (4096 environments,
    horizon 200, the reference's 2x512 tanh actor and critic): rollout graph (policy, sampling, env step, reward
    wrappers, curriculum) + acs_gae + graphed minibatch updates (fused loss/gradient kernel, clip, Adam).
    Reported: training timesteps / s over whole updates, wall clock around ppo_training_loop after its warm-up."""
    import torch

    from ac_solver_b200.agents.args import parse_args as ppo_args
    from ac_solver_b200.agents.environment import get_env
    from ac_solver_b200.agents.ppo_agent import Agent
    from ac_solver_b200.agents import training as T

    n_envs, steps, updates = 4096, 200, 8
    a = ppo_args(["--num-envs", str(n_envs), "--num-steps", str(steps), "--horizon-length", "200", "--nodes-counts", "512", "512",
                  "--total-timesteps", str(n_envs * steps * updates), "--num-minibatches", "4", "--update-epochs", "1",
                  "--norm-rewards", "--states-type", "all"])
    import contextlib
    import io

    with contextlib.redirect_stdout(io.StringIO()):
        a.num_envs = min(n_envs, 1190)  # get_env asserts num_envs <= number of distinct initial states (environment.py:80-83)
        envs, initial_states, curr, rec, hist, processed = get_env(a)
    # 4096 environments over the 1190-state pool: the vector env is rebuilt at full width on the same pool
    from ac_solver_b200.envs.vector_env import ACVectorEnv

    pool = np.stack(initial_states)
    rows = pool[np.arange(n_envs) % len(pool)]
    pool_x = np.concatenate([rows, pool])
    envs = ACVectorEnv(rows, horizon_length=a.horizon_length, clip_rewards=(a.min_rew, a.max_rew), norm_rewards=True, gamma=a.gamma)
    envs.enable_curriculum(pool_x, repeat_solved_prob=a.repeat_solved_prob, seed=a.seed)
    a.num_envs, a.batch_size = n_envs, n_envs * steps
    a.minibatch_size = a.batch_size // a.num_minibatches
    dev = torch.device("cuda")
    torch.manual_seed(0)
    agent = Agent(envs, a.nodes_counts).to(dev)
    opt = torch.optim.Adam(agent.parameters(), lr=torch.tensor(a.learning_rate, device=dev), eps=a.epsilon, capturable=True)
    cwd = os.getcwd()
    os.chdir("/tmp")
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            a.total_timesteps = n_envs * steps * updates
            torch.cuda.synchronize()
            log = T.ppo_training_loop(envs, a, dev, opt, agent, list(range(n_envs)), {"solved": set(), "unsolved": set()}, {},
                                      set(), initial_states, checkpoint_every=0, progress=False)
            torch.cuda.synchronize()
    finally:
        os.chdir(cwd)
    # the first update captures the two CUDA graphs and sizes the allocator's pools: steady state = the later updates
    secs = sorted(log["perf/update_seconds"][2:])
    dt = secs[len(secs) // 2] * updates  # median whole-iteration time x updates
    return {"metric": "PPO training timesteps/sec (rollout + GAE + update, whole iterations)",
            "workload": f"{n_envs} envs x {steps} steps per update, {updates} updates, 2x512 tanh actor+critic fp32, 4 minibatches x 1 epoch, "
                        "NormalizeReward + clip and curriculum on the device; median whole-iteration wall time of updates 3.." + str(updates)
                        + " of one ppo_training_loop call (updates 1-2 capture the CUDA graphs)",
            "timesteps_per_s": n_envs * steps * updates / dt, "seconds_per_update": dt / updates,
            "update_seconds": [round(x, 4) for x in log["perf/update_seconds"]],
            "value_loss": log["losses/value_loss"], "policy_loss": log["losses/policy_loss"], "entropy": log["losses/entropy_loss"],
            "approx_kl": log["losses/approx_kl"], "episodes": log["charts/episode"],
            "note": "the reference's loop steps 4096 Python environments one by one on the host: at its measured "
                    "ACEnv.step rate (vecenv.cpu_baseline_python) the rollout alone is ~40 s per update"}


def bench_barcode(args):
    """SURVEY 8f-3: radius-5 ball sizes of all 1190 Miller-Schupp presentations (the workload of
    barcode_analysis/5_steps_neibourhoods) on the GPU, with a bounded sample through the reference's own C++ tool
    (oracle/_ref/neibourhoods_ref, compiled from the reference's sources) timed and compared beside it."""
    import subprocess
    import tempfile
    from ast import literal_eval

    from ac_solver_b200.barcode import neighbourhood_sizes

    data = os.path.join(ROOT, "ac_solver_b200", "search", "miller_schupp", "data", "all_presentations.txt")
    lines = [l.strip() for l in open(data) if l.strip()]
    pres = [literal_eval(l) for l in lines]
    neighbourhood_sizes(pres[:2], radius=2)
    t0 = time.perf_counter()
    sizes = neighbourhood_sizes(pres, radius=5)
    gpu_s = time.perf_counter() - t0
    out = {"metric": "radius-5 neighbourhood sizes of the 1190 Miller-Schupp presentations (12 prime moves)",
           "rows": len(pres), "states_total": int(sum(sizes)), "seconds": gpu_s, "states_per_s": sum(sizes) / gpu_s}
    exe = os.path.join(ROOT, "oracle", "_ref", "neibourhoods_ref")
    if os.path.exists(exe):
        idx = list(range(0, len(lines), len(lines) // 12))[:12]
        with tempfile.TemporaryDirectory() as d:
            src, dst = os.path.join(d, "in.txt"), os.path.join(d, "out.txt")
            with open(src, "w") as f:
                f.write("\n".join(lines[i] for i in idx) + "\n")
            t0 = time.perf_counter()
            subprocess.run([exe, src, dst, "5", "0"], check=True, stdout=subprocess.DEVNULL)
            ref_s = time.perf_counter() - t0
            ref = [int(x) for x in open(dst).read().split()]
        out["parity"] = {"rows_compared": len(idx), "mismatches": sum(1 for k, i in enumerate(idx) if ref[k] != sizes[i]),
                         "checked": "ball sizes vs the reference's own C++ tool run here"}
        out["cpu_baseline"] = {"value": sum(ref) / ref_s, "unit": "states/s", "cores": 1, "kind": "reference",
                               "sample": f"oracle/_ref/neibourhoods_ref (the reference's neibourhoods.cpp compiled by oracle/Makefile) "
                                         f"on {len(idx)} of the 1190 rows: {ref_s:.1f} s",
                               "extrapolated_seconds_all_rows_1core": ref_s * sum(sizes) / max(sum(ref), 1)}
    return out


def bfs_traffic(world):
    """DRAM bytes per expansion from the committed ncu launch list of the 1-GPU search (profiles/)."""
    try:
        with open(os.path.join(ROOT, "profiles", "pbfs_r2_ncu_summary.json")) as f:
            d = json.load(f)
        return {"dram_bytes_per_expansion": d["dram_bytes_per_expansion"], "source": d["source"]} if world == 1 else None
    except Exception:
        return None


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
