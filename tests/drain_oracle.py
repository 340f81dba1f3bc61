"""ctypes binding of tests/drain_oracle.c (TEST INFRASTRUCTURE ONLY): the CPU oracle plus simon_oracle_drain, the checker of
simon_drain_run.  The library is compiled on first use into a temporary directory keyed by the sources' contents, so a read-only
tree works as well."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from simon_b200 import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_SRCS = [os.path.join(_HERE, "drain_oracle.c"), os.path.join(_ROOT, "oracle", "simon_oracle.c"), os.path.join(_ROOT, "include", "simon_gpu.h")]
# the oracle's own flags (oracle/Makefile)
_CFLAGS = ["-O2", "-fPIC", "-shared", "-std=c11", "-D_GNU_SOURCE", "-pthread", "-Wall", "-Wextra", "-ffp-contract=off", "-fno-fast-math"]
_LIB = None


def build() -> str:
    h = hashlib.sha256()
    for p in _SRCS:
        with open(p, "rb") as f:
            h.update(f.read())
    h.update(" ".join(_CFLAGS).encode())
    so = os.path.join(tempfile.gettempdir(), f"simon_drain_oracle_{os.getuid()}_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.check_call([os.environ.get("CC", "gcc")] + _CFLAGS + ["-o", tmp, _SRCS[0], "-lm"])
        os.replace(tmp, so)
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        L.simon_oracle_create.restype = C.c_void_p
        L.simon_oracle_create.argtypes = [C.c_void_p, C.c_void_p]
        L.simon_oracle_destroy.argtypes = [C.c_void_p]
        L.simon_oracle_set_active.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
        L.simon_oracle_schedule.restype = C.c_int
        L.simon_oracle_schedule.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
        L.simon_oracle_set_threads.restype = C.c_int
        L.simon_oracle_set_threads.argtypes = [C.c_void_p, C.c_int]
        L.simon_oracle_drain.restype = C.c_int
        L.simon_oracle_drain.argtypes = [C.c_void_p] + [C.c_void_p] * 2 + [C.c_uint32] + [C.c_void_p] * 5
        _LIB = L
    return _LIB


class DrainOracle:
    """The CPU oracle on one compiled cluster: the live run (schedule) and node drains on it (drain)."""

    def __init__(self, compiled, threads: int = 1):
        self.c = compiled
        self.snap, self.pods, self._keep = abi.marshal(compiled)
        self.h = lib().simon_oracle_create(C.byref(self.snap), C.byref(self.pods))
        if not self.h:
            raise MemoryError("simon_oracle_create failed")
        if threads > 1:
            lib().simon_oracle_set_threads(self.h, int(threads))

    def close(self):
        if self.h:
            lib().simon_oracle_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def schedule(self):
        """Every pod in order on all nodes (the live run): -> out_node."""
        P = self.c.pods_dims["n_pods"]
        out = np.full(max(P, 1), -9, np.int32)
        n_fail = C.c_uint32(0)
        rc = lib().simon_oracle_schedule(self.h, 0, P, out.ctypes.data, None, None, None, 0, C.byref(n_fail))
        if rc != 0:
            raise RuntimeError(f"simon_oracle_schedule rc={rc}")
        return out[:P]

    def drain(self, placement, survivors):
        """Node drain on the CURRENT (live) state: placement[pod] = the pod's node, survivors = surviving nodes in their scheduling
        order.  -> (counts dict, pod, node, fail_counts [n, 24], sums dict); the state is left as it was."""
        P = self.c.pods_dims["n_pods"]
        pl = np.ascontiguousarray(placement, dtype=np.int32)
        sv = np.ascontiguousarray(survivors, dtype=np.uint32)
        counts = np.zeros(5, np.uint32)
        pod = np.zeros(max(P, 1), np.uint32)
        node = np.zeros(max(P, 1), np.int32)
        fc = np.zeros((max(P, 1), abi.N_FAIL_CODES), np.uint32)
        sums = np.zeros(4, np.int64)
        rc = lib().simon_oracle_drain(self.h, pl.ctypes.data, sv.ctypes.data if len(sv) else None, len(sv), counts.ctypes.data,
                                      pod.ctypes.data, node.ctypes.data, fc.ctypes.data, sums.ctypes.data)
        if rc != 0:
            raise RuntimeError(f"simon_oracle_drain rc={rc}")
        n = int(counts[0])
        cd = dict(zip(["n_evicted", "n_rescheduled", "n_unscheduled", "n_daemon", "n_bound"], [int(x) for x in counts]))
        sd = dict(zip(["req_mcpu", "alloc_mcpu", "req_mem", "alloc_mem"], [int(x) for x in sums]))
        return cd, pod[:n], node[:n], fc[:n], sd
