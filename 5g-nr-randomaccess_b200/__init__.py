"""rach_b200: B200-native engine for the 5G NR RACH UE state machine (see DESIGN.md).

Import with importlib (the directory name is not a Python identifier):
    rach = importlib.import_module("5g-nr-randomaccess_b200")
"""
from .api import (RachSim, RaParams, RaStats, RaOptions, RachError, default_params, arrival_schedule, validate_params,  # noqa: F401
                  load_lib, LIB_PATH, SYMBOLS, DUMP_NAMES, RA_DUMP_FIELDS, STATS_DTYPE, hist_bins, HIST_DELAY, HIST_TX,
                  HIST_FAIL)
from .build import build_lib, build_host  # noqa: F401
from .shard import shard_plan, local_counter_vector, allreduce_counters, COUNTER_KEYS  # noqa: F401
