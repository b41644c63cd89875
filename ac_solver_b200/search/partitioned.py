"""Hash-partitioned breadth-first search, native driver (csrc/pbfs.cu).

Drop-in for the reference's ``bfs`` (ac_solver/search/breadth_first.py:15-97) on one GPU and on
the GPUs of one node, one process per GPU (``torchrun``).  The chunk loop lives in the library:
it is enqueued on CUDA streams without host synchronisation, and newly generated states are
written straight into the owner rank's inbox by peer stores over NVLink -- the expansion kernel
*is* the all-to-all.  ``torch.distributed`` is used for plumbing only: the all-gather of the
64-byte cudaIpc handles at set-up, the parent-chain walk of a solved search and the final gather
of the visited states.

Results (path, visited array in insertion order, stdout) are bit-identical to the reference for
every world size.  For tests ``sim_world=k`` runs k ranks inside one process on one device.
"""

from __future__ import annotations

import ctypes as C

import numpy as np

from .. import _lib
from ._common import _raise_for, check_row, search_info


def _info(res, stats_list):
    info = search_info(res)
    st = stats_list[0]
    info.update(n_local=[int(s[0]) for s in stats_list], chunks=int(st[1]),
                records_sent=[int(s[2]) for s in stats_list], records_recv=[int(s[3]) for s in stats_list],
                chunk_cap=int(st[4]), log_cap=int(st[5]), arena_bytes=int(st[6]), table_slots=int(st[7]))
    return info


class PartitionedBfs:
    """One rank (or, with ``sim_world``, all ranks) of the partitioned search; reusable across
    ``run`` calls with the same geometry (mrl, budget, cyclical)."""

    def __init__(self, mrl, max_nodes, cyclical=False, group=None, sim_world=None, chunk_parents=0, device=None,
                 timeout_s=None):
        import torch

        self.torch = torch
        self.L = _lib.lib()
        if not torch.cuda.is_available():
            raise _lib.AcsError("no CUDA device visible; the partitioned search has no CPU fallback")
        self.mrl, self.budget, self.cyclical = int(mrl), int(max_nodes), int(bool(cyclical))
        self.group = group
        self.handles = []
        dist = torch.distributed
        self.dist_on = sim_world is None and dist.is_available() and dist.is_initialized() and \
            dist.get_world_size(group) > 1
        dev = _lib.default_device() if device is None else int(device)
        self.device = dev
        if sim_world is not None:
            self.world, self.rank = int(sim_world), 0
            for r in range(self.world):
                self.handles.append(self._create(dev, r, self.world, chunk_parents))
            arr = (C.c_void_p * self.world)(*[h.value for h in self.handles])
            _lib.check(self.L.acs_pbfs_connect_local(arr, self.world))
        elif self.dist_on:
            self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
            h = self._create(dev, self.rank, self.world, chunk_parents)
            self.handles.append(h)
            blob = (C.c_ubyte * 64)()
            _lib.check(self.L.acs_pbfs_export(h, blob))
            mine = torch.tensor(list(blob), dtype=torch.uint8, device=torch.device("cuda", dev))
            allh = [torch.empty_like(mine) for _ in range(self.world)]
            dist.all_gather(allh, mine, group=group)
            packed = bytes(torch.cat(allh).cpu().numpy().tobytes())
            _lib.check(self.L.acs_pbfs_connect(h, packed))
            dist.barrier(group=group)
        else:
            self.world, self.rank = 1, 0
            self.handles.append(self._create(dev, 0, 1, chunk_parents))
        if timeout_s:
            for h in self.handles:
                _lib.check(self.L.acs_pbfs_set_timeout(h, float(timeout_s)))

    def _create(self, dev, rank, world, chunk_parents):
        h = C.c_void_p()
        _lib.check(self.L.acs_pbfs_create(dev, rank, world, self.mrl, self.budget, self.cyclical,
                                          int(chunk_parents or 0), C.byref(h)))
        return h

    def close(self):
        for h in self.handles:
            self.L.acs_pbfs_destroy(h)
        self.handles = []

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ------------------------------------------------------------------------------------------
    def run(self, presentation, want_visited=False):
        """-> (solved, path|None, info), identical on every rank."""
        torch = self.torch
        p8 = check_row(presentation)
        if p8.size != 2 * self.mrl:
            raise ValueError("presentation length does not match this search's max_relator_length")
        n = len(self.handles)
        arr = (C.c_void_p * n)(*[h.value for h in self.handles])
        cap = 1 << 16
        path = np.zeros((cap, 2), np.int32)
        res = _lib.SearchResult()
        rc = self.L.acs_pbfs_run(arr, n, p8.ctypes.data, path.ctypes.data, cap, C.byref(res))
        if self.dist_on:  # a rank-local failure must not leave the others inside a collective
            flag = torch.tensor([rc], dtype=torch.int64, device=torch.device("cuda", self.device))
            torch.distributed.all_reduce(flag, op=torch.distributed.ReduceOp.MIN, group=self.group)
            if int(flag.item()) != 0 and rc == 0:
                raise _lib.AcsError("partitioned bfs failed on another rank")
        _lib.check(rc)
        stats = []
        for h in self.handles:
            s = (C.c_int64 * 8)()
            _lib.check(self.L.acs_pbfs_stats(h, s))
            stats.append(list(s))
        info = _info(res, stats)
        info["world"] = self.world
        plist = None
        if res.solved:
            if self.dist_on:
                plist = self._walk_path(int(res.n_moves) - 1)
            else:
                plist = [(int(a), int(l)) for a, l in path[: res.path_len]]
        if want_visited and res.status == 0:
            info["visited"] = self._gather_visited(int(res.n_visited))
        _raise_for(res.status)
        return bool(res.solved), plist, info

    def _walk_path(self, sol_gid):
        """Parent chain of the solving candidate across ranks: exactly one rank owns each id."""
        torch, dist = self.torch, self.torch.distributed
        chain, g = [], sol_gid // 12
        dev = torch.device("cuda", self.device)
        while g >= 0:
            out = (C.c_int64 * 4)()
            _lib.check(self.L.acs_pbfs_lookup(self.handles[0], int(g), out))
            rec = torch.tensor(list(out), dtype=torch.int64, device=dev)
            if not out[0]:
                rec.zero_()
            dist.all_reduce(rec, group=self.group)
            rec = rec.cpu().numpy()
            assert rec[0] == 1, "global id not found on exactly one rank"
            chain.append((int(rec[2]), int(rec[3])))
            g = int(rec[1])
        return chain[::-1] + [(sol_gid % 12, 2)]

    def _gather_visited(self, n_nodes):
        parts = []
        for h in self.handles:
            s = (C.c_int64 * 8)()
            _lib.check(self.L.acs_pbfs_stats(h, s))
            nl = int(s[0])
            gids = np.zeros(max(nl, 1), np.int64)
            rows = np.zeros((max(nl, 1), 2 * self.mrl), np.int8)
            n_out = C.c_int64(0)
            _lib.check(self.L.acs_pbfs_visited(h, gids.ctypes.data, rows.ctypes.data, nl, C.byref(n_out)))
            parts.append((gids[: n_out.value], rows[: n_out.value]))
        if self.dist_on:
            dist = self.torch.distributed
            gathered = [None] * self.world if self.rank == 0 else None
            dist.gather_object(parts[0], gathered, dst=0, group=self.group)
            if self.rank != 0:
                return None
            parts = gathered
        gids = np.concatenate([g for g, _ in parts])
        rows = np.concatenate([r for _, r in parts])
        order = np.argsort(gids, kind="stable")
        assert np.array_equal(gids[order], np.arange(n_nodes)), "global ids are not a permutation of the FIFO positions"
        return rows[order]


def bfs_partitioned(presentation, max_nodes_to_explore=10000, cyclically_reduce_after_moves=False, group=None,
                    want_visited=False, chunk_parents=0, sim_world=None, verbose=False, device=None):
    """Partitioned ``bfs``: call on every rank of the process group with the same arguments.
    Returns ``(solved, path|None, info)`` on every rank; ``info["visited"]`` (rank 0, on request)
    holds the visited states in the reference's insertion order."""
    p8 = check_row(presentation)
    with PartitionedBfs(p8.size // 2, max_nodes_to_explore, cyclically_reduce_after_moves, group=group,
                        sim_world=sim_world, chunk_parents=chunk_parents, device=device) as eng:
        solved, path, info = eng.run(p8, want_visited=want_visited)
        rank0 = eng.rank == 0
    if verbose and rank0:
        for m in info["minlen_log"]:
            print(f"New minimal length found: {m}")
    if info["budget_hit"] and rank0 and verbose is not None:
        print(f"Exiting search as number of explored nodes = {info['n_visited']} has exceeded the limit "
              f"{int(max_nodes_to_explore)}")
    return solved, path, info
