"""ctypes binding of libsimon_gpu.so — the C-ABI engine (include/simon_gpu.h).

There is NO CPU fallback: if the shared library is missing or no CUDA device can be opened, constructing an
Engine raises EngineUnavailable.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional

import numpy as np

from . import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SIMON_GPU_LIB") or os.path.join(_HERE, "libsimon_gpu.so")    # the override is for kernel experiments
_LIB = None

EXPORTS = ["simon_gpu_version", "simon_ctx_create", "simon_ctx_destroy", "simon_last_error", "simon_snapshot_upload",
           "simon_pods_upload", "simon_state_reset", "simon_schedule", "simon_results_download", "simon_last_kernel_ms",
           "simon_launch_count", "simon_state_download", "simon_scenarios_run", "simon_replay", "simon_stats",
           "simon_gpu_slots_download", "simon_state_download_ext", "simon_debug_set_dump_pod", "simon_debug_dump_read",
           "simon_moves_upload", "simon_moves_run", "simon_moves_replay", "simon_host_go118_sort",
           "simon_host_last_error", "simon_host_compile", "simon_host_plan_free", "simon_host_plan_columns", "simon_host_plan_describe",
           "simon_host_simulate", "simon_host_free", "simon_host_quantity_probe", "simon_host_plan_fit_error", "simon_host_capacity_search",
           "simon_drain_run", "simon_drain_download"]


class EngineUnavailable(RuntimeError):
    pass


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise EngineUnavailable(f"{LIB_PATH} not built: run __graft_entry__.build() (nvcc, sm_100a)")
    L = C.CDLL(LIB_PATH)
    L.simon_gpu_version.restype = C.c_int
    L.simon_ctx_create.restype = C.c_int
    L.simon_ctx_create.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    L.simon_ctx_destroy.argtypes = [C.c_void_p]
    L.simon_last_error.restype = C.c_char_p
    L.simon_last_error.argtypes = [C.c_void_p]
    L.simon_snapshot_upload.restype = C.c_int
    L.simon_snapshot_upload.argtypes = [C.c_void_p, C.c_void_p]
    L.simon_pods_upload.restype = C.c_int
    L.simon_pods_upload.argtypes = [C.c_void_p, C.c_void_p]
    L.simon_state_reset.restype = C.c_int
    L.simon_state_reset.argtypes = [C.c_void_p]
    L.simon_schedule.restype = C.c_int
    L.simon_schedule.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_uint32, C.c_void_p]
    L.simon_results_download.restype = C.c_int
    L.simon_results_download.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]
    L.simon_replay.restype = C.c_int
    L.simon_replay.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_float)]
    L.simon_stats.restype = C.c_int
    L.simon_stats.argtypes = [C.c_void_p, C.c_void_p]
    L.simon_last_kernel_ms.restype = C.c_float
    L.simon_last_kernel_ms.argtypes = [C.c_void_p]
    L.simon_launch_count.restype = C.c_uint64
    L.simon_launch_count.argtypes = [C.c_void_p]
    L.simon_state_download.restype = C.c_int
    L.simon_state_download.argtypes = [C.c_void_p] + [C.c_void_p] * 6
    L.simon_scenarios_run.restype = C.c_int
    L.simon_scenarios_run.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
    try:
        L.simon_gpu_slots_download.restype = C.c_int
        L.simon_gpu_slots_download.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
        L.simon_state_download_ext.restype = C.c_int
        L.simon_state_download_ext.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.simon_debug_set_dump_pod.restype = C.c_int
        L.simon_debug_set_dump_pod.argtypes = [C.c_void_p, C.c_uint32]
        L.simon_debug_dump_read.restype = C.c_int
        L.simon_debug_dump_read.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.simon_moves_upload.restype = C.c_int
        L.simon_moves_upload.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32]
        L.simon_moves_run.restype = C.c_int
        L.simon_moves_run.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.simon_moves_replay.restype = C.c_int
        L.simon_moves_replay.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_float)]
        L.simon_host_go118_sort.restype = C.c_int
        L.simon_host_go118_sort.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
        L.simon_drain_run.restype = C.c_int
        L.simon_drain_run.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
        L.simon_drain_download.restype = C.c_int
        L.simon_drain_download.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    except AttributeError:
        if not os.environ.get("SIMON_GPU_LIB"):       # an experiment library may lack the newer entry points; the shipped one may not
            raise
    _LIB = L
    return L


class Engine:
    """One device context holding one compiled cluster (snapshot + ordered pod list)."""

    def __init__(self, compiled, device: int = 0, record_scores: bool = False, cluster_ctas: int = 0,
                 threads_per_cta: int = 0, pin_fast: bool = True):
        L = lib()
        self.c = compiled
        self.h = C.c_void_p()
        # pin_fast=False: DaemonSet pods take the general one-decision-at-a-time path (SIMON_OPT_NO_PIN_FAST; same results)
        opts = abi.SimonCtxOpts(device, cluster_ctas, threads_per_cta,
                                (abi.OPT_RECORD_SCORES if record_scores else 0) | (0 if pin_fast else abi.OPT_NO_PIN_FAST))
        rc = L.simon_ctx_create(C.byref(opts), C.byref(self.h))
        if rc != 0 or not self.h:
            raise EngineUnavailable(f"simon_ctx_create failed (rc={rc}): no usable CUDA device {device}; "
                                    "the engine has no CPU path")
        self.record_scores = record_scores
        self.snap, self.pods, self._keep = abi.marshal(compiled)
        self._check(L.simon_snapshot_upload(self.h, C.byref(self.snap)))
        self._check(L.simon_pods_upload(self.h, C.byref(self.pods)))

    def _check(self, rc: int):
        if rc != 0:
            msg = lib().simon_last_error(self.h)
            raise RuntimeError(f"simon engine error {rc}: {msg.decode() if msg else ''}")

    def close(self):
        if getattr(self, "h", None):
            lib().simon_ctx_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self):
        self._check(lib().simon_state_reset(self.h))

    def schedule(self, first: int = 0, count: Optional[int] = None, max_fail: Optional[int] = None, download: bool = True):
        """Place pods [first, first+count). Returns (out_node, out_score, fail_counts, fail_pod)."""
        P = self.c.pods_dims["n_pods"]
        count = P - first if count is None else count
        max_fail = count if max_fail is None else max_fail
        n_fail = C.c_uint32(0)
        if not download:
            self._check(lib().simon_schedule(self.h, first, count, None, None, None, None, 0, C.byref(n_fail)))
            return None, None, None, None
        out_node = np.full(count, -9, np.int32)
        out_score = np.zeros(count, np.int64)
        fail_counts = np.zeros((max(max_fail, 1), abi.N_FAIL_CODES), np.uint32)
        fail_pod = np.zeros(max(max_fail, 1), np.uint32)
        self._check(lib().simon_schedule(self.h, first, count, out_node.ctypes.data,
                                         out_score.ctypes.data if self.record_scores else None,
                                         fail_counts.ctypes.data, fail_pod.ctypes.data, max_fail, C.byref(n_fail)))
        nf = min(n_fail.value, max_fail)
        return out_node, out_score, fail_counts[:nf], fail_pod[:nf]

    def results(self, first: int = 0, count: Optional[int] = None):
        P = self.c.pods_dims["n_pods"]
        count = P - first if count is None else count
        out_node = np.full(count, -9, np.int32)
        self._check(lib().simon_results_download(self.h, first, count, out_node.ctypes.data, None))
        return out_node

    def replay(self, steps: int = 1) -> float:
        """steps x (reset + place every pod), device-timed; returns total ms. Results stay on the device."""
        ms = C.c_float(0)
        self._check(lib().simon_replay(self.h, steps, C.byref(ms)))
        return float(ms.value)

    def stats(self):
        a = np.zeros(32, np.uint64)
        self._check(lib().simon_stats(self.h, a.ctypes.data))
        return dict(decisions=int(a[0]), class_switches=int(a[1]), summary_rebuilds=int(a[2]), redone=int(a[3]), static_evals=int(a[4]), single_flip_fast=int(a[6]),
                    merged_decisions=int(a[7] & 0xffffffff), merged_redone=int(a[7] >> 32),
                    cycles=dict(zip(['loop', 'fixed', 'class_change_tail', 'r1', 'p1', 'reduce_steady', 'reduce_summary', 'p3', 'argmax', 'commit',
                                     'cc_pre', 'cc_sync', 'cc_blob', 'cc_entry', 'cc_static', 'pts_pass_steady'],
                                    [int(x) for x in a[8:24]])),
                    reductions=dict(zip(['allreduce_bar', 'allreduce_exchange', 'allreduce_n', 'argmax_bar', 'argmax_exchange', 'argmax_n'],
                                        [int(x) for x in a[24:30]])),
                    owner_commit=dict(cycles=int(a[30]), n=int(a[31])), spec_own=dict(cycles=int(a[27]), n=int(a[5])))

    def last_kernel_ms(self) -> float:
        return float(lib().simon_last_kernel_ms(self.h))

    def launch_count(self) -> int:
        return int(lib().simon_launch_count(self.h))

    def state(self):
        N = self.c.n_nodes
        arrs = [np.zeros(N, np.int64) for _ in range(5)] + [np.zeros(N, np.int32)]
        self._check(lib().simon_state_download(self.h, *[a.ctypes.data for a in arrs]))
        return dict(zip(["req_mcpu", "req_mem", "req_eph", "nz_mcpu", "nz_mem", "num_pods"], arrs))

    def gpu_slots(self, first: int = 0, count: Optional[int] = None):
        """GPU-share Reserve results: per pod a list of device ids (one per GPU slot, ascending), [] if none."""
        P = self.c.pods_dims["n_pods"]
        count = P - first if count is None else count
        a = np.zeros(max(count, 1), np.uint32)
        self._check(lib().simon_gpu_slots_download(self.h, first, count, a.ctypes.data))
        out = []
        for v in a[:count]:
            v = int(v)
            out.append([d for d in range(8) for _ in range((v >> (4 * d)) & 15)])
        return out

    def state_ext(self):
        N, K = self.c.n_nodes, int(self.c.snap_dims["n_scalars"])
        rs = np.zeros((max(K, 1), max(N, 1)), np.int64)
        gu = np.zeros((8, max(N, 1)), np.int64)
        self._check(lib().simon_state_download_ext(self.h, rs.ctypes.data, gu.ctypes.data))
        return dict(req_scalar=rs[:K, :N], gpu_used=gu[:, :N])

    def dump_pod(self, pod: int):
        """From the EMPTY state, schedule up to and including `pod`; return (out_node of the range, per-node totals,
        per-node filter verdicts of that pod).  Leaves the context in that partial state."""
        self.reset()
        self._check(lib().simon_debug_set_dump_pod(self.h, pod))
        out = self.schedule(0, pod + 1)[0]
        self._check(lib().simon_debug_set_dump_pod(self.h, 0xffffffff))
        N = self.c.n_nodes
        tot = np.zeros(max(N, 1), np.int64)
        code = np.zeros(max(N, 1), np.int32)
        self._check(lib().simon_debug_dump_read(self.h, tot.ctypes.data, code.ctypes.data))
        return out, tot[:N], code[:N]

    # ---- candidate-move scoring (config 5) ----
    def moves_upload(self, moves: np.ndarray, move_base: int = 0):
        """moves: uint32 array [n, 2] of (pod index, target node)."""
        a = np.ascontiguousarray(moves, dtype=np.uint32).reshape(-1, 2)
        self._moves_keep = a
        self._check(lib().simon_moves_upload(self.h, a.ctypes.data, len(a), move_base))
        return len(a)

    def moves_run(self, k: int = 0, want_arrays: bool = True, want_per_pod: bool = False):
        """-> dict(best_key, n_feasible, kernel_ms, gain, code, best_per_pod, topk=[(move, gain)...])."""
        n = len(self._moves_keep)
        gain = np.zeros(max(n, 1), np.int32) if want_arrays else None
        code = np.zeros(max(n, 1), np.uint32) if want_arrays else None
        bpp = np.zeros(max(self.c.pods_dims["n_pods"], 1), np.uint64) if want_per_pod else None
        topk = np.zeros((max(k, 1), 2), np.int32)
        res = abi.SimonMovesResult()
        self._check(lib().simon_moves_run(self.h, k, gain.ctypes.data if want_arrays else None, code.ctypes.data if want_arrays else None,
                                          bpp.ctypes.data if want_per_pod else None, topk.ctypes.data if k else None, C.byref(res)))
        return dict(best_key=int(res.best_key), n_feasible=int(res.n_feasible), kernel_ms=float(res.kernel_ms),
                    gain=None if gain is None else gain[:n], code=None if code is None else code[:n],
                    best_per_pod=bpp, topk=[(int(topk[q, 0]) & 0xffffffff, int(topk[q, 1])) for q in range(res.n_topk)])

    def moves_replay(self, steps: int = 1) -> float:
        ms = C.c_float(0)
        self._check(lib().simon_moves_replay(self.h, steps, C.byref(ms)))
        return float(ms.value)

    @staticmethod
    def _scenario_array(scenarios: List[np.ndarray]):
        """The simon_scenario array of node lists, and the uint32 arrays it points into (to be kept alive across the call)."""
        arr = (abi.SimonScenario * max(len(scenarios), 1))()
        keep = [np.ascontiguousarray(nodes, dtype=np.uint32) for nodes in scenarios]
        for i, a in enumerate(keep):
            arr[i].n_nodes = len(a)
            arr[i].nodes = a.ctypes.data
        return arr, keep

    def run_scenarios(self, scenarios: List[np.ndarray], want_nodes: bool = False):
        """scenarios: list of uint32 arrays (active node indices in scenario order)."""
        n = len(scenarios)
        arr, keep = self._scenario_array(scenarios)
        res = (abi.SimonScenarioResult * n)()
        P = self.c.pods_dims["n_pods"]
        out_node = np.full((n, P), -9, np.int32) if want_nodes else None
        self._check(lib().simon_scenarios_run(self.h, arr, n, res, out_node.ctypes.data if want_nodes else None))
        out = [dict(n_unscheduled=r.n_unscheduled, n_scheduled=r.n_scheduled, req_mcpu=r.req_mcpu, alloc_mcpu=r.alloc_mcpu,
                    req_mem=r.req_mem, alloc_mem=r.alloc_mem, elapsed_ms=r.elapsed_ms) for r in res]
        return out, out_node

    def drain(self, scenarios: List[np.ndarray]):
        """Node drains on the live state (simon_drain_run): scenarios = surviving node indices in their scheduling order
        (drain.survivor_order).  -> (results, off, pod, node, fail_counts): one dict per scenario (counts and sums over the
        survivors) and, per evicted pod, scenario s owning entries off[s]:off[s+1]: pod index, new node (-1: unschedulable),
        failure histogram [n, SIMON_N_FAIL_CODES] (zero for placed pods)."""
        n = len(scenarios)
        arr, keep = self._scenario_array(scenarios)
        res = (abi.SimonDrainResult * max(n, 1))()
        off = np.zeros(n + 1, np.uint64)
        self._check(lib().simon_drain_run(self.h, arr, n, res, off.ctypes.data))
        tot = int(off[-1])
        pod = np.zeros(max(tot, 1), np.uint32)
        node = np.zeros(max(tot, 1), np.int32)
        fc = np.zeros((max(tot, 1), abi.N_FAIL_CODES), np.uint32)
        self._check(lib().simon_drain_download(self.h, pod.ctypes.data, node.ctypes.data, fc.ctypes.data))
        out = [dict(n_evicted=r.n_evicted, n_rescheduled=r.n_rescheduled, n_unscheduled=r.n_unscheduled, n_daemon=r.n_daemon,
                    n_bound=r.n_bound, req_mcpu=r.req_mcpu, alloc_mcpu=r.alloc_mcpu, req_mem=r.req_mem, alloc_mem=r.alloc_mem,
                    elapsed_ms=r.elapsed_ms) for r in res[:n]]
        return out, off.astype(np.int64), pod[:tot], node[:tot], fc[:tot]
