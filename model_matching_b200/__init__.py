"""model_matching_b200 -- B200-native StoCS hot path (drop-in for kuwt/model_matching's
stocs::stocs_estimator online methods).  The product is libstocs_b200.so (CUDA, sm_100a) behind
the C ABI in include/stocs_b200.h; this package holds its sources (csrc/), the C++ host shim
and CLIs (host/), a ctypes binding (_capi) and the synthetic-workload generators (synth)."""
from ._capi import (Context, Group, RECORD, StocsError, lib, LIB_PATH, SYMBOLS, shard_range,  # noqa: F401
                    comm_unique_id, upload_scenes, run_pipelines)

__all__ = ["Context", "Group", "RECORD", "StocsError", "lib", "LIB_PATH", "SYMBOLS", "shard_range", "comm_unique_id",
           "upload_scenes", "run_pipelines"]
