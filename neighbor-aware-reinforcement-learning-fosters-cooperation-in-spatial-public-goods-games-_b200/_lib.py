"""ctypes binding of ``libspgg_b200.so`` (C ABI declared in ``include/spgg.h``).

The library is built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a).  There
is no CPU fallback: if the shared object is missing or no CUDA device is present
every computing call raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SPGG_B200_LIB selects another build of the same library (kernel tuning experiments)
LIB_PATH = os.environ.get("SPGG_B200_LIB") or os.path.join(_HERE, "libspgg_b200.so")
NSTAT = 40

# stat-row columns (include/spgg.h: enum spgg_stat)
ST_NC_OLD, ST_N_CD, ST_N_DC, ST_NC_NEW = 0, 1, 2, 3
ST_SUM_P, ST_SUM_P_C, ST_SUM_P_D, ST_SUM_WP_P = 4, 5, 6, 7
ST_SUM_REW_C, ST_SUM_REW_D, ST_SUM_RATIO = 8, 9, 10
ST_GROUP0 = 11
ST_SUM_R = 17
ST_SUM_Q, ST_SUM_Q_C, ST_SUM_Q_D = 18, 22, 26
ST_SUM_NI, ST_N_BEST_POS, ST_N_BEST_2ND, ST_GMAX = 30, 31, 32, 33

PREC_FP32, PREC_FP64 = 0, 1
STATE_REPUTATION, STATE_ACTION = 0, 1
ALGO_QLEARNING, ALGO_SARSA, ALGO_EXPECTED_SARSA, ALGO_DOUBLE_QLEARNING = 0, 1, 2, 3
RSTORE_AUTO, RSTORE_INT8, RSTORE_FP32 = 0, 1, 2
E_INVALID, E_CUDA, E_STATE, E_UNSUPPORTED = -1, -2, -3, -4
CLUSTER_PERIODIC = 1
BLOCK_R, BLOCK_Q = 1, 2
HIST_R, HIST_Q = 1, 2
MAX_SNAPSHOTS = 8
SNAP_R, SNAP_Q = 1, 2


class Params(C.Structure):
    """``spgg_params_t``"""
    _fields_ = [("L", C.c_int32), ("rows", C.c_int32), ("row0", C.c_int32), ("M", C.c_int32),
                ("state_mode", C.c_int32), ("precision", C.c_int32), ("algorithm", C.c_int32),
                ("r_storage", C.c_int32),
                ("r", C.c_double), ("c", C.c_double), ("cost", C.c_double),
                ("alpha", C.c_double), ("gamma", C.c_double),
                ("epsilon", C.c_double), ("epsilon_decay", C.c_double),
                ("epsilon_min", C.c_double), ("kappa", C.c_double),
                ("lambda_eps", C.c_double), ("rep_gain_C", C.c_double),
                ("delta_R_D", C.c_double), ("R_min", C.c_double), ("R_max", C.c_double),
                ("wP", C.c_double), ("seed", C.c_uint64)]


class Status(C.Structure):
    """``spgg_status_t``"""
    _fields_ = [("iteration", C.c_int64), ("stopped_at", C.c_int64), ("epsilon", C.c_double),
                ("n_replicas", C.c_int32), ("r_is_int8", C.c_int32),
                ("kernel_launches", C.c_int64), ("speculative_launches", C.c_int64),
                ("speculation_failures", C.c_int64)]


EXPORTS = (
    "spgg_create", "spgg_destroy", "spgg_set_state", "spgg_get_state", "spgg_set_replay",
    "spgg_set_replay_pairs",
    "spgg_step", "spgg_sync", "spgg_get_stats", "spgg_query", "spgg_halo_bytes",
    "spgg_halo_pack", "spgg_halo_unpack", "spgg_phase_kernel", "spgg_phase_gmax",
    "spgg_gmax_device_ptr", "spgg_begin_steps", "spgg_end_steps", "spgg_last_error",
    "spgg_abi_version", "spgg_init_random", "spgg_describe", "spgg_set_progress",
    "spgg_state_digest", "spgg_phase_iteration", "spgg_strip_can_speculate", "spgg_strip_iteration",
    "spgg_strip_report_ptr", "spgg_strip_verify", "spgg_strip_failed", "spgg_strip_rewind",
    "spgg_r_histogram", "spgg_ipc_export", "spgg_ipc_attach", "spgg_ring_export", "spgg_ring_attach",
    "spgg_clusters", "spgg_cluster_sizes", "spgg_cluster_labels",
    "spgg_strip_cluster_record_bytes", "spgg_strip_clusters", "spgg_strip_clusters_resolve",
    "spgg_pair_counts", "spgg_strip_pair_record_bytes", "spgg_strip_pair_record", "spgg_strip_pair_counts",
    "spgg_block_fields", "spgg_value_ranges", "spgg_histograms",
    "spgg_snapshot", "spgg_snapshot_info", "spgg_snapshot_free", "spgg_overlap",
)

_lib = None


def load():
    """Load the shared object (no CUDA call is made until ``spgg_create``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing - build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    lib.spgg_create.argtypes = [C.POINTER(Params), i32, i32, C.POINTER(vp)]
    lib.spgg_destroy.argtypes = [vp]
    lib.spgg_destroy.restype = None
    lib.spgg_set_state.argtypes = [vp, i32, vp, vp, vp]
    lib.spgg_get_state.argtypes = [vp, i32, vp, vp, vp]
    lib.spgg_set_replay.argtypes = [vp, i32, vp, vp]
    lib.spgg_set_replay_pairs.argtypes = [vp, i32, i32, vp, vp]
    lib.spgg_step.argtypes = [vp, i32, vp]
    lib.spgg_sync.argtypes = [vp]
    lib.spgg_get_stats.argtypes = [vp, i32, i32, i32, vp]
    lib.spgg_query.argtypes = [vp, i32, C.POINTER(Status)]
    lib.spgg_halo_bytes.argtypes = [vp]
    lib.spgg_halo_bytes.restype = i64
    lib.spgg_halo_pack.argtypes = [vp, vp, vp, vp]
    lib.spgg_halo_unpack.argtypes = [vp, vp, vp, vp]
    lib.spgg_phase_kernel.argtypes = [vp, i32, i32, vp]
    lib.spgg_phase_gmax.argtypes = [vp, vp]
    lib.spgg_phase_iteration.argtypes = [vp, i32, vp]
    lib.spgg_strip_can_speculate.argtypes = [vp, i32]
    lib.spgg_strip_iteration.argtypes = [vp, i32, vp]
    lib.spgg_strip_report_ptr.argtypes = [vp]
    lib.spgg_strip_report_ptr.restype = vp
    lib.spgg_strip_verify.argtypes = [vp, vp]
    lib.spgg_strip_failed.argtypes = [vp]
    lib.spgg_strip_rewind.argtypes = [vp, i32]
    lib.spgg_r_histogram.argtypes = [vp, i32, i32, vp, vp]
    lib.spgg_clusters.argtypes = [vp, i32, i32, i32, C.POINTER(i64)]
    lib.spgg_cluster_sizes.argtypes = [vp, vp, i64]
    lib.spgg_cluster_labels.argtypes = [vp, vp]
    lib.spgg_strip_cluster_record_bytes.argtypes = [vp]
    lib.spgg_strip_cluster_record_bytes.restype = i64
    lib.spgg_strip_clusters.argtypes = [vp, i32, i32, vp]
    lib.spgg_strip_clusters_resolve.argtypes = [vp, i32, i32, vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]
    lib.spgg_pair_counts.argtypes = [vp, i32, i32, vp]
    lib.spgg_strip_pair_record_bytes.argtypes = [vp, i32, i32]
    lib.spgg_strip_pair_record_bytes.restype = i64
    lib.spgg_strip_pair_record.argtypes = [vp, i32, i32, vp]
    lib.spgg_strip_pair_counts.argtypes = [vp, i32, i32, vp, i32, i32, vp]
    lib.spgg_block_fields.argtypes = [vp, i32, i32, i32, vp, vp]
    lib.spgg_value_ranges.argtypes = [vp, i32, i32, i32, vp]
    lib.spgg_histograms.argtypes = [vp, i32, i32, i32, i32, vp, vp, vp]
    lib.spgg_snapshot.argtypes = [vp, i32, i32, i32, i32]
    lib.spgg_snapshot_info.argtypes = [vp, i32, vp, vp, vp, vp]
    lib.spgg_snapshot_free.argtypes = [vp, i32]
    lib.spgg_overlap.argtypes = [vp, i32, i32, i32, i32, vp, vp, vp]
    lib.spgg_ipc_export.argtypes = [vp, vp]
    lib.spgg_ipc_attach.argtypes = [vp, i32, vp, i32, i32]
    lib.spgg_ring_export.argtypes = [vp, vp]
    lib.spgg_ring_attach.argtypes = [vp, i32, i32, vp]
    lib.spgg_gmax_device_ptr.argtypes = [vp]
    lib.spgg_gmax_device_ptr.restype = vp
    lib.spgg_begin_steps.argtypes = [vp, i32, vp]
    lib.spgg_end_steps.argtypes = [vp, vp]
    lib.spgg_init_random.argtypes = [vp, i32, C.c_uint64]
    lib.spgg_describe.argtypes = [vp, C.c_char_p, i32]
    lib.spgg_set_progress.argtypes = [vp, i64, vp]
    lib.spgg_state_digest.argtypes = [vp, i32, vp]
    lib.spgg_last_error.restype = C.c_char_p
    lib.spgg_abi_version.restype = i32
    _lib = lib
    return lib


def check(rc: int):
    """Map the C error convention onto the exceptions the reference raises
    (ValueError for bad arguments, spgg.py:118,309; RuntimeError otherwise)."""
    if rc == 0:
        return
    msg = load().spgg_last_error().decode("utf-8", "replace")
    if rc in (E_INVALID, E_UNSUPPORTED):
        raise ValueError(msg)
    raise RuntimeError(msg)
