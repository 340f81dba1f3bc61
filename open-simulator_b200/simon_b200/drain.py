"""Node drains: "if I remove node X (or nodes X, Y, Z), where do its pods go, and do they all still fit?"

The pod-migration use case of the reference (README.md:16: scaling a cluster down, defragmenting it).  The reference has the
primitives - NodeInfo.RemovePod (vendor/k8s.io/kubernetes/pkg/scheduler/framework/types.go:539-585) and nodeTree.removeNode
(.../scheduler/internal/cache/node_tree.go:70-100) - but no implementation, so the definition is this library's
(include/simon_gpu.h, "node drains"): on the cluster as Simulate() leaves it, the pods of the drained nodes are classified
(DaemonSet pods vanish with their node, pre-bound pods are deleted, every other pod is evicted), and the evicted pods go through
the full scheduling path again, in pod order, on the surviving nodes in removeNode order; everything else stays where it is.
Many drains run at once on the device (simon_drain_run), each from a fork of the live state.

    Drain(cluster, apps, candidates=None, *opts, bound_pods="block", max_cpu=100, max_mem=100) -> DrainResult
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np

from . import objects as O
from .capacity import occupancy_ok
from .compiler import Compiled, compile_cluster, get_zone_key
from .simulator import (SimulateResult, SimulatorOptions, UnscheduledPod, build_result, format_fit_error, plan,
                        MAX_GPU_FAIL_DETAIL)
from .workloads import PodRec

SCW_FLAGS, SCW_GUARD_NODE = 9, 13        # class-blob words (include/simon_gpu.h, enum simon_class_word)
CLS_PINNED = 16


def survivor_order(compiled: Compiled, drained: Iterable[int]) -> np.ndarray:
    """nodeTree.list() after removeNode of every drained node (compiled node indices in, compiled indices out).

    Zones keep the order in which the cluster's nodes first introduced them and a zone disappears only when it empties; nodes keep
    their insertion order (node_orig_index) inside their zone.  This is not node_tree_list() of the survivors: a zone's position
    comes from ALL of the cluster's nodes, drained ones included."""
    N = compiled.n_nodes
    d = [int(x) for x in drained]
    if any(x < 0 or x >= N for x in d):
        raise ValueError(f"drained node index out of range [0, {N})")
    if len(set(d)) != len(d):
        raise ValueError("drained node listed twice")
    gone = set(d)
    zones: List[str] = []
    tree: Dict[str, List[int]] = {}
    for i in sorted(range(N), key=lambda i: compiled.node_orig_index[i]):       # addNode in insertion order
        z = get_zone_key(compiled.node_objs[i])
        if z not in tree:
            tree[z] = []
            zones.append(z)
        tree[z].append(i)
    for i in d:                                                                   # removeNode
        z = get_zone_key(compiled.node_objs[i])
        tree[z].remove(i)
        if not tree[z]:
            del tree[z]
            zones.remove(z)
    out: List[int] = []
    total = N - len(gone)
    k = 0
    while len(out) < total:                                                       # list(): zone round robin
        for z in zones:
            if k < len(tree[z]):
                out.append(tree[z][k])
        k += 1
    return np.array(out, dtype=np.uint32)


@dataclass
class DrainOutcome:
    """One candidate set of nodes drained from the live cluster."""
    Nodes: List[str]
    Feasible: bool
    Evicted: List[Tuple[PodRec, str, Optional[str]]] = field(default_factory=list)    # (pod, from node, to node or None)
    UnscheduledPods: List[UnscheduledPod] = field(default_factory=list)
    DaemonSetPods: List[PodRec] = field(default_factory=list)
    BoundPods: List[PodRec] = field(default_factory=list)
    Occupancy: Dict[str, int] = field(default_factory=dict)                            # sums over the survivors after re-placement


@dataclass
class DrainResult:
    Simulate: SimulateResult
    Drains: List[DrainOutcome]


def pod_kinds(compiled: Compiled) -> Tuple[np.ndarray, np.ndarray]:
    """Per pod: (is a DaemonSet pod - pinned class or guard node -, is pre-bound) as the drain classifies them."""
    pods = compiled.pods
    blob, off, cls = pods["class_blob"], pods["class_off"], pods["pod_class"]
    flags = np.array([int(blob[int(off[c]) + SCW_FLAGS]) for c in range(len(off) - 1)], np.int64)
    guard = np.array([int(blob[int(off[c]) + SCW_GUARD_NODE]) for c in range(len(off) - 1)], np.int64)
    pin = pods.get("pod_pin_node")
    g = guard[cls] if len(cls) else np.zeros(0, np.int64)
    if pin is not None:
        g = np.where(g == -3, np.asarray(pin, np.int64), g)
    daemon = ((flags[cls] & CLS_PINNED) != 0) | (g >= 0) if len(cls) else np.zeros(0, bool)
    bound = ~daemon & (np.asarray(pods["pod_fixed_node"]) >= 0)
    return daemon, bound


def _resolve(compiled: Compiled, candidates) -> List[List[int]]:
    if candidates is None:
        order = sorted(range(compiled.n_nodes), key=lambda i: compiled.node_orig_index[i])
        return [[i] for i in order]
    sets = []
    for cand in candidates:
        names = [cand] if isinstance(cand, str) else list(cand)
        idx = []
        for nm in names:
            i = compiled.node_index(nm)
            if i < 0:
                raise ValueError(f"Drain: unknown node {nm!r}")
            if i in idx:
                raise ValueError(f"Drain: node {nm!r} listed twice in one candidate set")
            idx.append(i)
        sets.append(idx)
    return sets


def Drain(cluster: O.ResourceTypes, apps: List[O.AppResource], candidates: Optional[Sequence] = None, *opts,
          bound_pods: str = "block", max_cpu: int = 100, max_mem: int = 100) -> DrainResult:
    """Simulate() the cluster and apps, then drain every candidate set of node names from the result (None: every node alone).

    Feasible = no evicted pod is left unschedulable, no pre-bound pod is lost (unless bound_pods="drop") and the survivors' CPU and
    memory occupancy passes satisfyResourceSetting (capacity.occupancy_ok with max_cpu / max_mem).  Failure texts are FitError's over
    the survivors ("0/(N-|D|) nodes are available: ..."); Open-Gpu-Share's per-node "Node:<name>" detail is not re-evaluated for
    drains (count-only text).  Raises EngineUnavailable without a CUDA device, ValueError for unknown or repeated node names."""
    if bound_pods not in ("block", "drop"):
        raise ValueError("Drain: bound_pods must be 'block' or 'drop'")
    options = SimulatorOptions()
    for o in opts:
        o(options)
    if options.schedulerConfig or options.kubeconfig or options.extraRegistry:
        raise NotImplementedError("Drain: only the default scheduler configuration and in-memory clusters are supported")
    with O.gc_paused():
        p = plan(cluster, apps)
        compiled = compile_cluster(p.nodes, p.pods, p.ctx)
    sets = _resolve(compiled, candidates)
    from .engine import Engine          # raises EngineUnavailable without libsimon_gpu.so / a CUDA device
    orders = [survivor_order(compiled, s) for s in sets]
    gpu_fail_nodes = {}
    with Engine(compiled, device=options.device) as eng:
        out_node, _scores, fail_counts, fail_pod = eng.schedule()
        results, off, epod, enode, efc = eng.drain(orders)
        # Simulate()'s own Open-Gpu-Share detail re-runs pods from an empty state: after the drains, which need the live state
        todo = [int(pod) for j, pod in enumerate(fail_pod) if j < len(fail_counts) and int(fail_counts[j][19]) > 0][:MAX_GPU_FAIL_DETAIL]
        for pod in todo:
            _o, _t, code = eng.dump_pod(pod)
            gpu_fail_nodes[pod] = [compiled.node_names[g] for g in np.nonzero(code & (1 << 19))[0]]
    live = np.asarray(out_node).copy()
    sim = build_result(compiled, p, out_node, fail_counts, fail_pod, gpu_fail_nodes)
    daemon, bound = pod_kinds(compiled)
    names = compiled.node_names
    recs = p.pods
    drains = []
    static_memo: dict = {}
    for s, (idx, order, r) in enumerate(zip(sets, orders, results)):
        gone = np.zeros(compiled.n_nodes + 1, bool)
        gone[idx] = True
        on = np.nonzero((live >= 0) & gone[np.where(live >= 0, live, compiled.n_nodes)])[0]
        out = DrainOutcome(Nodes=[names[i] for i in idx], Feasible=False)
        out.DaemonSetPods = [recs[q] for q in on if daemon[q]]
        out.BoundPods = [recs[q] for q in on if bound[q] and not daemon[q]]
        act = [int(x) for x in order]
        for j in range(int(off[s]), int(off[s + 1])):
            q, to = int(epod[j]), int(enode[j])
            out.Evicted.append((recs[q], names[live[q]], names[to] if to >= 0 else None))
            if to < 0:
                out.UnscheduledPods.append(UnscheduledPod(recs[q], format_fit_error(compiled, recs[q], efc[j], active=act,
                                                                                    static_memo=static_memo)))
        out.Occupancy = dict(req_mcpu=int(r["req_mcpu"]), alloc_mcpu=int(r["alloc_mcpu"]), req_mem=int(r["req_mem"]),
                             alloc_mem=int(r["alloc_mem"]))
        out.Feasible = (r["n_unscheduled"] == 0 and (r["n_bound"] == 0 or bound_pods == "drop")
                        and occupancy_ok(out.Occupancy, max_cpu, max_mem))
        drains.append(out)
    return DrainResult(Simulate=sim, Drains=drains)
