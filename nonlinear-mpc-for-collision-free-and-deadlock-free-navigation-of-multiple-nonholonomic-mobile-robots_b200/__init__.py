"""B200-native batched NMPC solver for multi-robot unicycle navigation (hot path only).

Python host over the C-ABI library csrc/ -> libnmpc_b200.so (include/nmpc_b200.h).
"""
from ._cabi import LIB_PATH, NSTATS, STATUS, SYMBOLS, NmpcError, lib  # noqa: F401
from .solver import DM, NlpSolver, Problem, SmallOcp, closed_loop, distributed_loop, horzcat, nlpsol, repmat, reshape, vertcat  # noqa: F401
from . import _cabi, mpc_loop, odometry, sharding, workload  # noqa: F401,E402
