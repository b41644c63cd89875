"""ac_solver_b200 -- B200-native implementation of AC-Solver's AC-move / search hot path.

Same public names as the reference package (``ac_solver/__init__.py:1-6``) for the path this
repo rebuilds: ``ACEnv``, ``ACEnvConfig``, ``ACMove``, ``bfs``, ``greedy_search``.  All compute
runs in hand-written sm_100a CUDA kernels behind the C ABI in ``include/acsolver_b200.h``;
importing the package needs no GPU, calling a compute function does (no CPU fallback).
"""

from .envs.ac_env import ACEnv, ACEnvConfig  # noqa: F401
from .envs.ac_moves import ACMove, ac_moves_batch, concatenate_relators, conjugate  # noqa: F401
from .search.beam import beam_meet_in_the_middle, beam_search, beam_search_batch  # noqa: F401
from .search.breadth_first import bfs, bfs_batch, bfs_groups, canonical_form  # noqa: F401
from .search.goals import GoalSet, bfs_meet_in_the_middle, greedy_meet_in_the_middle, trivial_ball  # noqa: F401
from .search.greedy import greedy_search, greedy_search_batch  # noqa: F401

__all__ = ["ACEnv", "ACEnvConfig", "ACMove", "ac_moves_batch", "bfs", "bfs_batch", "bfs_groups", "canonical_form", "GoalSet",
           "trivial_ball",
           "beam_search", "beam_search_batch", "beam_meet_in_the_middle",
           "bfs_meet_in_the_middle", "greedy_meet_in_the_middle", "greedy_search", "greedy_search_batch",
           "concatenate_relators", "conjugate"]
__version__ = "0.1.0"
