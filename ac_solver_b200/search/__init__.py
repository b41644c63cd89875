from .beam import beam_meet_in_the_middle, beam_search, beam_search_batch  # noqa: F401
from .breadth_first import bfs, bfs_batch, bfs_device, bfs_groups, canonical_form  # noqa: F401
from .goals import GoalSet, bfs_meet_in_the_middle, greedy_meet_in_the_middle, trivial_ball  # noqa: F401
from .greedy import greedy_search, greedy_search_batch, greedy_search_groups  # noqa: F401
