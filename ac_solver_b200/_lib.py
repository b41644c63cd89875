"""ctypes loader of libacsolver_b200.so -- the only bridge between the Python host code
and the CUDA kernels.  There is NO CPU fallback: if the library is missing, or no CUDA
device is visible, every compute entry point raises."""

from __future__ import annotations

import ctypes as C
import os
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libacsolver_b200.so")

ACS_OK = 0
ACS_ERR_INVALID, ACS_ERR_CUDA, ACS_ERR_UNSUPPORTED, ACS_ERR_NOMEM, ACS_ERR_NO_DEVICE = -1, -2, -3, -4, -5
ROW_OK, ROW_ASSERT, ROW_INDEX = 0, 1, 2
OP_ACMOVE, OP_CONCAT_RAW, OP_CONJ_RAW, OP_SIMPLIFY_RELATOR, OP_SIMPLIFY_PRESENTATION = range(5)
FLAG_CYCLICAL, FLAG_NORMALIZED, FLAG_LENS_VALID = 1, 2, 4


class AcsError(RuntimeError):
    pass


class SearchResult(C.Structure):
    _fields_ = [
        ("solved", C.c_int32),
        ("status", C.c_int32),
        ("budget_hit", C.c_int32),
        ("path_len", C.c_int32),
        ("n_visited", C.c_int64),
        ("n_expanded", C.c_int64),
        ("n_moves", C.c_int64),
        ("frontier_left", C.c_int64),
        ("n_levels", C.c_int32),
        ("n_minlen", C.c_int32),
        ("minlen_log", C.c_int32 * 128),
        ("seconds_device", C.c_double),
    ]


class SbfsArgs(C.Structure):
    """Mirror of ``acs_sbfs_args`` (include/acsolver_b200.h)."""

    _fields_ = [
        ("keys", C.c_void_p), ("parent", C.c_void_p), ("gid", C.c_void_p), ("table", C.c_void_p),
        ("tmask", C.c_uint64), ("n_local", C.c_int64), ("l0", C.c_int64), ("l1", C.c_int64),
        ("head", C.c_int64), ("nparents", C.c_int64), ("n_nodes", C.c_int64), ("budget", C.c_int64),
        ("limit", C.c_int64),
        ("mrl", C.c_int32), ("cyclical", C.c_int32), ("trusted", C.c_int32), ("world", C.c_int32),
        ("rank", C.c_int32), ("min_len", C.c_int32), ("W", C.c_int32), ("pad_", C.c_int32),
        ("dest_count", C.c_void_p), ("dest_cursor", C.c_void_p), ("send_keys", C.c_void_p),
        ("send_c", C.c_void_p), ("ctrl", C.c_void_p), ("recv_keys", C.c_void_p), ("recv_c", C.c_void_p),
        ("n_recv", C.c_int64), ("rec_slot", C.c_void_p), ("bitmap_local", C.c_void_p),
        ("bitmap_global", C.c_void_p), ("prefix_local", C.c_void_p), ("prefix_global", C.c_void_p),
        ("cut", C.c_void_p),
    ]


class CurriculumArgs(C.Structure):
    """Mirror of ``acs_curriculum_args`` (include/acsolver_b200.h)."""

    _fields_ = [
        ("state", C.c_void_p), ("pool", C.c_void_p), ("pool_lens", C.c_void_p), ("lens", C.c_void_p),
        ("action", C.c_void_p), ("reward", C.c_void_p), ("done", C.c_void_p), ("truncated", C.c_void_p),
        ("step_count", C.c_void_p), ("cur_state", C.c_void_p), ("solved", C.c_void_p), ("solved_list", C.c_void_p),
        ("best", C.c_void_p), ("best_actions", C.c_void_p), ("action_log", C.c_void_p), ("final_obs", C.c_void_p),
        ("final_steps", C.c_void_p), ("counters", C.c_void_p), ("err", C.c_void_p),
        ("n", C.c_int64), ("n_states", C.c_int32), ("mrl", C.c_int32), ("horizon", C.c_int32),
        ("log_stride", C.c_int32), ("flags", C.c_int32), ("repeat_solved_prob", C.c_float), ("seed", C.c_uint64),
    ]


_lib = None
_lock = threading.Lock()
_ctx = {}

_P = C.c_void_p
_SIGS = {
    "acs_version": (C.c_int, []),
    "acs_last_error": (C.c_char_p, []),
    "acs_device_count": (C.c_int, []),
    "acs_ctx_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "acs_ctx_destroy": (None, [_P]),
    "acs_moves_batch": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int64, C.c_int, C.c_int, _P]),
    "acs_moves_batch_host": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int64, C.c_int, C.c_int]),
    "acs_env_step_batch": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int64, C.c_int, C.c_int, C.c_int, _P]),
    "acs_env_step_host": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, C.c_int64, C.c_int, C.c_int, C.c_int,
                                    C.POINTER(C.c_int64)]),
    "acs_vecenv_step": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int, _P, _P, _P, C.c_int64, C.c_int,
                                  C.c_int, C.c_int, _P]),
    "acs_reward_transform": (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_double, C.c_double, C.c_int, C.c_int, C.c_double,
                                       C.c_double, _P]),
    "acs_vecenv_curriculum_step": (C.c_int, [_P, _P]),
    "acs_validate_batch": (C.c_int, [_P, _P, C.c_int64, C.c_int, _P]),
    "acs_validate_batch_host": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int]),
    "acs_generic_batch": (C.c_int, [C.c_int, _P, _P, _P, _P, _P, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int,
                                    C.c_int, _P]),
    "acs_generic_host": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, _P, C.c_int64, C.c_int, C.c_int, C.c_int,
                                   C.c_int, C.c_int]),
    "acs_bfs_create": (C.c_int, [_P, C.c_int, C.c_int, C.c_int64, C.c_int, C.POINTER(_P)]),
    "acs_bfs_run": (C.c_int, [_P, _P, _P, C.c_int, C.POINTER(SearchResult)]),
    "acs_bfs_visited": (C.c_int, [_P, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "acs_bfs_destroy": (None, [_P]),
    "acs_bfs_batch_bytes": (C.c_int, [C.c_int, C.c_int, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "acs_bfs_batch_create": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, C.c_int, C.c_int64, C.POINTER(_P)]),
    "acs_bfs_batch_run": (C.c_int, [_P, _P, _P, C.c_int, C.POINTER(SearchResult)]),
    "acs_bfs_batch_paths": (C.c_int, [_P, _P, C.c_int]),
    "acs_bfs_batch_visited": (C.c_int, [_P, C.c_int, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "acs_bfs_batch_destroy": (None, [_P]),
    "acs_bfs_batch_set_goals": (C.c_int, [_P, _P, C.c_int]),
    "acs_bfs_batch_goal_hits": (C.c_int, [_P, _P]),
    "acs_canonical_form": (C.c_int, [C.c_int, C.c_int, _P, C.c_int64, _P, _P]),
    "acs_bfs_batch_set_symmetric": (C.c_int, [_P, C.c_int]),
    "acs_bfs_batch_goal_hit_elements": (C.c_int, [_P, _P]),
    "acs_beam_bytes": (C.c_int, [C.c_int, C.c_int, C.c_int64, _P, C.c_int, C.POINTER(C.c_int64)]),
    "acs_beam_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int64, _P, C.c_int, C.c_int, C.POINTER(_P)]),
    "acs_beam_set_goals": (C.c_int, [_P, _P]),
    "acs_beam_run": (C.c_int, [_P, _P, _P, C.c_int, C.POINTER(SearchResult)]),
    "acs_beam_paths": (C.c_int, [_P, _P, C.c_int]),
    "acs_beam_visited": (C.c_int, [_P, C.c_int, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "acs_beam_goal_hits": (C.c_int, [_P, _P]),
    "acs_beam_goal_hit_elements": (C.c_int, [_P, _P]),
    "acs_beam_destroy": (None, [_P]),
    "acs_goalset_from_rows_symmetric": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, C.c_int64, C.POINTER(_P)]),
    "acs_goalset_is_symmetric": (C.c_int, [_P, C.POINTER(C.c_int)]),
    "acs_goalset_path_frame": (C.c_int, [_P, C.c_int64, C.POINTER(C.c_int), _P, C.c_int, C.POINTER(C.c_int),
                                         C.POINTER(C.c_int)]),
    "acs_greedy_goal_hit_elements": (C.c_int, [_P, _P]),
    "acs_goalset_from_rows": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, C.c_int64, C.POINTER(_P)]),
    "acs_goalset_from_bfs_batch": (C.c_int, [_P, C.POINTER(_P)]),
    "acs_goalset_size": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "acs_goalset_path": (C.c_int, [_P, C.c_int64, C.POINTER(C.c_int), _P, C.c_int, C.POINTER(C.c_int)]),
    "acs_goalset_destroy": (None, [_P]),
    "acs_greedy_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, C.POINTER(_P)]),
    "acs_greedy_run": (C.c_int, [_P, _P, _P, _P]),
    "acs_greedy_visited": (C.c_int, [_P, C.c_int, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "acs_greedy_destroy": (None, [_P]),
    "acs_greedy_set_goals": (C.c_int, [_P, _P]),
    "acs_greedy_goal_hits": (C.c_int, [_P, _P]),
    "acs_sbfs_pack_root": (C.c_int, [_P, C.c_int, _P, _P, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "acs_sbfs_owner": (C.c_int, [C.c_uint64, C.c_int]),
    "acs_sbfs_expand": (C.c_int, [_P, C.c_int, _P]),
    "acs_sbfs_insert_mark": (C.c_int, [_P, _P]),
    "acs_sbfs_scan": (C.c_int, [_P, _P, C.c_int64, _P]),
    "acs_sbfs_cut": (C.c_int, [_P, _P]),
    "acs_sbfs_rank_at": (C.c_int, [_P, _P, _P]),
    "acs_sbfs_commit": (C.c_int, [_P, _P]),
    "acs_sbfs_lower_bound": (C.c_int, [_P, C.c_int64, C.c_int64, _P, _P]),
    "acs_sbfs_lookup": (C.c_int, [_P, C.c_int64, _P, _P]),
    "acs_sbfs_unpack": (C.c_int, [_P, _P, C.c_int64, C.c_int, _P]),
    "acs_ball_explore": (C.c_int, [C.c_int, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, C.POINTER(C.c_int64), _P,
                                   _P, C.c_int64, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "acs_gae": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.c_int, C.c_int64, C.c_double, C.c_double, _P]),
    "acs_ppo_loss_workspace_bytes": (C.c_int, []),
    "acs_ppo_loss": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int,
                               C.c_double, C.c_double, C.c_double, _P]),
    "acs_rollout_sample_record": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int64, C.c_int64, C.c_int, C.c_int,
                                            C.c_uint64, _P]),
    "acs_rollout_finish": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int64, C.c_int64, C.c_int, _P]),
    "acs_ball_sizes": (C.c_int, [C.c_int, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int64, _P]),
    "acs_pbfs_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int64, C.POINTER(_P)]),
    "acs_pbfs_export": (C.c_int, [_P, _P]),
    "acs_pbfs_connect": (C.c_int, [_P, C.c_char_p]),
    "acs_pbfs_connect_local": (C.c_int, [_P, C.c_int]),
    "acs_pbfs_run": (C.c_int, [_P, C.c_int, _P, _P, C.c_int, C.POINTER(SearchResult)]),
    "acs_pbfs_lookup": (C.c_int, [_P, C.c_int64, _P]),
    "acs_pbfs_visited": (C.c_int, [_P, _P, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "acs_pbfs_stats": (C.c_int, [_P, _P]),
    "acs_pbfs_set_timeout": (C.c_int, [_P, C.c_double]),
    "acs_pbfs_destroy": (None, [_P]),
}


def exported_symbols():
    """Names include/acsolver_b200.h declares (used by the CPU-side ABI test)."""
    return sorted(_SIGS)


def lib():
    """Load the shared library (no device needed for this step)."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise AcsError(
                    f"{LIB_PATH} is missing: build it with `python -m ac_solver_b200.build` "
                    "(there is no CPU fallback for the AC-move kernels)"
                )
            L = C.CDLL(LIB_PATH)
            for name, (res, args) in _SIGS.items():
                fn = getattr(L, name)
                fn.restype = res
                fn.argtypes = args
            _lib = L
    return _lib


def check(rc: int):
    if rc != ACS_OK:
        msg = lib().acs_last_error()
        raise AcsError(f"libacsolver_b200 error {rc}: {msg.decode() if msg else ''}")


def ctx(device: int = 0):
    """Per-device context (streams + scratch).  Raises without a GPU."""
    L = lib()
    with _lock:
        if device not in _ctx:
            h = _P()
            rc = L.acs_ctx_create(int(device), C.byref(h))
            if rc != ACS_OK:
                msg = L.acs_last_error()
                raise AcsError(f"cannot create a CUDA context on device {device}: {msg.decode() if msg else rc}")
            _ctx[device] = h
        return _ctx[device]


def default_device() -> int:
    """LOCAL_RANK under torchrun, else 0."""
    return int(os.environ.get("LOCAL_RANK", "0"))
