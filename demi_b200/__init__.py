"""demi_b200 — B200-native schedule-space exploration engine behind DEMi's
Scheduler / TestOracle plugin surface.  See DESIGN.md."""
from . import _native  # noqa: F401
from .events import (Start, Kill, HardKill, Send, WaitQuiescence, Partition, UnPartition,  # noqa: F401
                     pack_externals, unpack_externals, raft5_program, pingpong3_program, bcast32_program)
from .schedulers import (DemiError, SchedulerConfig, Engine, RandomScheduler, STSScheduler, ReplayScheduler,  # noqa: F401
                         DDMin, MinimizationStats, DPORwHeuristics, STSSchedMinimizer, LeftToRightOneAtATime, SrcDstFIFORemoval,
                         ProvenanceTracker, ResumableDPOR, IncrementalDDMin, ArvindDistanceOrdering,
                         DefaultBacktrackOrdering, mask_of, events_of, program_of, random_ddmin)
