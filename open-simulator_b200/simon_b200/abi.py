"""ctypes mirror of include/simon_gpu.h (structs + marshalling of a Compiled cluster)."""
from __future__ import annotations

import ctypes as C

import numpy as np

N_FAIL_CODES = 24
OPT_RECORD_SCORES = 1
OPT_NO_PIN_FAST = 2


class SimonSnapshot(C.Structure):
    _fields_ = [
        ("n_nodes", C.c_uint32), ("n_scalars", C.c_uint32), ("n_label_words", C.c_uint32),
        ("n_taint_words", C.c_uint32), ("n_topos", C.c_uint32), ("n_node_classes", C.c_uint32),
        ("n_log", C.c_uint32), ("reserved", C.c_uint32),
        ("topo_ndom", C.c_void_p), ("alloc_mcpu", C.c_void_p), ("alloc_mem", C.c_void_p), ("alloc_eph", C.c_void_p),
        ("alloc_scalar", C.c_void_p), ("alloc_pods", C.c_void_p), ("node_flags", C.c_void_p),
        ("label_bits", C.c_void_p), ("taint_hard", C.c_void_p), ("taint_soft", C.c_void_p),
        ("topo_dom", C.c_void_p), ("node_class", C.c_void_p), ("gpu_count", C.c_void_p),
        ("gpu_dev_mem", C.c_void_p), ("gpu_total_mem", C.c_void_p), ("log_table", C.c_void_p),
    ]


class SimonPodset(C.Structure):
    _fields_ = [
        ("n_classes", C.c_uint32), ("n_pods", C.c_uint32), ("n_counters", C.c_uint32),
        ("n_static_rows", C.c_uint32), ("n_extra_rows", C.c_uint32), ("n_static_sigs", C.c_uint32),
        ("class_off", C.c_void_p), ("class_blob", C.c_void_p), ("pod_class", C.c_void_p),
        ("pod_fixed_node", C.c_void_p), ("pod_pin_node", C.c_void_p), ("counter_topo", C.c_void_p), ("simon_raw", C.c_void_p),
        ("extra_score", C.c_void_p),
    ]


class SimonCtxOpts(C.Structure):
    _fields_ = [("device", C.c_int32), ("cluster_ctas", C.c_uint32), ("threads_per_cta", C.c_uint32),
                ("flags", C.c_uint32)]


class SimonScenario(C.Structure):
    _fields_ = [("n_nodes", C.c_uint32), ("reserved", C.c_uint32), ("nodes", C.c_void_p)]


class SimonScenarioResult(C.Structure):
    _fields_ = [("n_unscheduled", C.c_uint32), ("n_scheduled", C.c_uint32),
                ("req_mcpu", C.c_int64), ("alloc_mcpu", C.c_int64), ("req_mem", C.c_int64), ("alloc_mem", C.c_int64),
                ("elapsed_ms", C.c_float), ("reserved", C.c_uint32)]


class SimonMovesResult(C.Structure):
    _fields_ = [("best_key", C.c_uint64), ("n_feasible", C.c_uint32), ("n_topk", C.c_uint32),
                ("kernel_ms", C.c_float), ("reserved", C.c_uint32)]


class SimonDrainResult(C.Structure):
    _fields_ = [("n_evicted", C.c_uint32), ("n_rescheduled", C.c_uint32), ("n_unscheduled", C.c_uint32),
                ("n_daemon", C.c_uint32), ("n_bound", C.c_uint32), ("reserved", C.c_uint32),
                ("req_mcpu", C.c_int64), ("alloc_mcpu", C.c_int64), ("req_mem", C.c_int64), ("alloc_mem", C.c_int64),
                ("elapsed_ms", C.c_float), ("reserved2", C.c_uint32)]


MOVE_NOOP, MOVE_NOT_PLACED, MOVE_NOT_MOVABLE, MOVE_BAD_INDEX = 1 << 24, 1 << 25, 1 << 26, 1 << 27
MOVE_GAIN_BIAS = 1000


_SNAP_DTYPES = {
    "topo_ndom": np.uint32, "alloc_mcpu": np.int64, "alloc_mem": np.int64, "alloc_eph": np.int64,
    "alloc_scalar": np.int64, "alloc_pods": np.int32, "node_flags": np.uint32, "label_bits": np.uint64,
    "taint_hard": np.uint64, "taint_soft": np.uint64, "topo_dom": np.int32, "node_class": np.int32,
    "gpu_count": np.int32, "gpu_dev_mem": np.int64, "gpu_total_mem": np.int64, "log_table": np.float64,
}
_PODS_DTYPES = {
    "class_off": np.uint64, "class_blob": np.int64, "pod_class": np.int32, "pod_fixed_node": np.int32,
    "counter_topo": np.uint32, "simon_raw": np.int64, "extra_score": np.int32, "pod_pin_node": np.int32,
}
_PODS_OPTIONAL = ("pod_pin_node",)       # NULL when the pod list has no pinned class (columns stored before ABI 3)


def ptr(a: np.ndarray) -> int:
    return a.ctypes.data


def marshal(compiled):
    """-> (SimonSnapshot, SimonPodset, keepalive list). Arrays are made contiguous with the ABI dtypes."""
    keep = []
    snap = SimonSnapshot()
    for k, v in compiled.snap_dims.items():
        setattr(snap, k, int(v))
    for k, dt in _SNAP_DTYPES.items():
        a = np.ascontiguousarray(compiled.snap[k], dtype=dt)
        keep.append(a)
        setattr(snap, k, ptr(a))
    pods = SimonPodset()
    for k, v in compiled.pods_dims.items():
        setattr(pods, k, int(v))
    for k, dt in _PODS_DTYPES.items():
        if k in _PODS_OPTIONAL and compiled.pods.get(k) is None:
            setattr(pods, k, None)
            continue
        a = np.ascontiguousarray(compiled.pods[k], dtype=dt)
        keep.append(a)
        setattr(pods, k, ptr(a))
    return snap, pods, keep
