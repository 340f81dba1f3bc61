"""Node drains (include/simon_gpu.h, "node drains"): the survivor order of nodeTree.removeNode, the oracle's restatement
(pinned against a re-simulation with the surviving pods pre-bound, and by hand-derived cases), the Python validation, and on the GPU
the engine (fork + pod-list placement kernel) against the oracle, bit for bit."""
import os
import random

import numpy as np
import pytest

from simon_b200 import objects as O, simulator, synth
from simon_b200.compiler import compile_cluster, get_zone_key
from util import make_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCW_GPU_MEM = 7


# ---- survivor order ------------------------------------------------------------------------------------------------------------
def _node(name, zone=None, cpu="4", taints=None, labels=None):
    lab = {"kubernetes.io/hostname": name}
    if zone:
        lab["topology.kubernetes.io/zone"] = zone
    lab.update(labels or {})
    n = {"apiVersion": "v1", "kind": "Node", "metadata": {"name": name, "labels": lab}, "spec": {},
         "status": {"allocatable": {"cpu": cpu, "memory": "8Gi", "pods": "20"}, "capacity": {"cpu": cpu, "memory": "8Gi", "pods": "20"}}}
    if taints:
        n["spec"]["taints"] = taints
    return n


def _pod(name, labels=None, node_name=None, anti=None, cpu="100m"):
    spec = {"containers": [{"name": "c", "image": "app:v1", "resources": {"requests": {"cpu": cpu, "memory": "64Mi"}}}]}
    if node_name:
        spec["nodeName"] = node_name
    if anti:
        spec["affinity"] = {"podAntiAffinity": {"requiredDuringSchedulingIgnoredDuringExecution": [
            {"labelSelector": {"matchLabels": a}, "topologyKey": "topology.kubernetes.io/zone"} for a in anti]}}
    return {"apiVersion": "v1", "kind": "Pod", "metadata": {"name": name, "namespace": "default", "labels": labels or {"app": name}},
            "spec": spec}


def _compile(nodes, pods=(), daemonsets=()):
    cluster = O.ResourceTypes(Nodes=list(nodes), Pods=list(pods), DaemonSets=list(daemonsets))
    p = simulator.plan(cluster, [])
    return p, compile_cluster(p.nodes, p.pods, p.ctx)


def _names(c, idx):
    return [c.node_names[int(i)] for i in idx]


def _tree_after_remove(nodes, drained):
    """nodeTree restated from node_tree.go: addNode in order, removeNode, list()."""
    zones, tree = [], {}
    for nd in nodes:
        z = get_zone_key(nd)
        if z not in tree:
            zones.append(z)
            tree[z] = []
        tree[z].append(O.name_of(nd))
    for nd in drained:
        z = get_zone_key(nd)
        tree[z].remove(O.name_of(nd))
        if not tree[z]:
            del tree[z]
            zones.remove(z)
    out, k = [], 0
    while len(out) < sum(len(v) for v in tree.values()):
        for z in zones:
            if k < len(tree[z]):
                out.append(tree[z][k])
        k += 1
    return out


def test_survivor_order_is_remove_node_order():
    from simon_b200.drain import survivor_order
    _p, c = _compile([_node("a1", "A"), _node("b1", "B"), _node("a2", "A")])
    assert c.node_names == ["a1", "b1", "a2"]
    # draining a1: zone A keeps its place in front of B -> [a2, b1] (recomputing from the survivors would give [b1, a2])
    assert _names(c, survivor_order(c, [c.node_index("a1")])) == ["a2", "b1"]
    assert _names(c, survivor_order(c, [])) == ["a1", "b1", "a2"]
    # a zone that empties disappears: zones A, B, C -> drain both A nodes
    _p, c = _compile([_node("a1", "A"), _node("b1", "B"), _node("c1", "C"), _node("a2", "A"), _node("b2", "B")])
    assert _names(c, survivor_order(c, [c.node_index("a1"), c.node_index("a2")])) == ["b1", "c1", "b2"]
    assert _names(c, survivor_order(c, [c.node_index("b1")])) == ["a1", "b2", "c1", "a2"]


def test_survivor_order_random_sets():
    from simon_b200.drain import survivor_order
    rng = random.Random(11)
    for it in range(200):
        n = rng.randint(1, 14)
        zones = [None, "A", "B", "C", "D"][:rng.randint(1, 5)]
        nodes = [_node(f"n{i}", rng.choice(zones)) for i in range(n)]
        _p, c = _compile(nodes)
        k = rng.randint(0, n)
        drained = rng.sample(range(n), k)
        got = _names(c, survivor_order(c, [c.node_index(f"n{i}") for i in drained]))
        assert got == _tree_after_remove(nodes, [nodes[i] for i in drained]), it


def test_survivor_order_rejects_bad_indices():
    from simon_b200.drain import survivor_order
    _p, c = _compile([_node("a1", "A"), _node("b1", "B")])
    with pytest.raises(ValueError):
        survivor_order(c, [2])
    with pytest.raises(ValueError):
        survivor_order(c, [-1])
    with pytest.raises(ValueError):
        survivor_order(c, [0, 0])


# ---- oracle ---------------------------------------------------------------------------------------------------------------------
class _Sub:
    """A compiled cluster with another pod list over the same classes (what Oracle / Engine consume)."""

    def __init__(self, c, pods, dims):
        self.snap, self.snap_dims, self.n_nodes = c.snap, c.snap_dims, c.n_nodes
        self.pods, self.pods_dims = pods, dims
        self.node_orig_index, self.node_objs, self.node_names = c.node_orig_index, c.node_objs, c.node_names


def _with_pods(c, idx, fixed=None):
    idx = np.asarray(idx, np.int64)
    pods = dict(c.pods)
    pods["pod_class"] = np.asarray(c.pods["pod_class"])[idx]
    pods["pod_fixed_node"] = np.asarray(c.pods["pod_fixed_node"])[idx] if fixed is None else np.asarray(fixed, np.int32)
    if c.pods.get("pod_pin_node") is not None:
        pods["pod_pin_node"] = np.asarray(c.pods["pod_pin_node"])[idx]
    dims = dict(c.pods_dims)
    dims["n_pods"] = len(idx)
    return _Sub(c, pods, dims)


def _no_gpu_share(c):
    blob, off = c.pods["class_blob"], c.pods["class_off"]
    keep = [q for q, k in enumerate(c.pods["pod_class"]) if blob[int(off[k]) + SCW_GPU_MEM] <= 0]
    return _with_pods(c, keep)


def _drain_sets(c, rng, n_multi):
    from simon_b200.drain import survivor_order
    N = c.n_nodes
    sets = [[g] for g in range(N)]
    for _ in range(n_multi):
        sets.append(rng.sample(range(N), rng.randint(2, max(2, min(N - 1, 6)))))
    return [(s, survivor_order(c, s)) for s in sets]


def test_oracle_drain_equals_resimulation_with_survivors_prebound():
    """Draining D = simulating a pod list made of the surviving placed pods, pre-bound to their live node in pod order, followed
    by the evicted pods, on the survivors in removeNode order: identical placements, failure histograms and sums.  (GPU-share pods
    are left out: a pre-bound pod holds no GPU memory, so the re-simulation would not see their reservations.)"""
    from drain_oracle import DrainOracle
    from oracle.binding import Oracle
    from simon_b200.drain import pod_kinds
    rng = random.Random(5)
    for seed in (101, 104, 107):
        _p, c0 = make_case("mix", seed_no=seed)
        c = _no_gpu_share(c0)
        o = DrainOracle(c)
        live = o.schedule()
        np.testing.assert_array_equal(live, Oracle(c).schedule()[0])
        daemon, bound = pod_kinds(c)
        checked = 0
        for drained, order in _drain_sets(c, rng, 20):
            counts, pod, node, fc, sums = o.drain(live, order)
            gone = set(drained)
            on = [q for q in range(len(live)) if live[q] >= 0 and int(live[q]) in gone]
            ev = [q for q in on if not daemon[q] and not bound[q]]
            assert list(pod) == ev
            assert counts["n_daemon"] == sum(1 for q in on if daemon[q]) and counts["n_bound"] == sum(1 for q in on if bound[q] and not daemon[q])
            keep = [q for q in range(len(live)) if live[q] >= 0 and int(live[q]) not in gone]
            sub = _with_pods(c, keep + ev, [int(live[q]) for q in keep] + [-1] * len(ev))
            r = Oracle(sub)
            r.set_active(order)
            out, _sc, rfc, rfp = r.schedule()
            tail = out[len(keep):]
            np.testing.assert_array_equal(node, tail)
            want = np.zeros_like(fc)
            for j, q in enumerate(rfp):
                want[int(q) - len(keep)] = rfc[j]
            np.testing.assert_array_equal(fc, want)
            st = r.state()
            assert sums["req_mcpu"] == int(sum(st["req_mcpu"][g] for g in order))
            assert sums["req_mem"] == int(sum(st["req_mem"][g] for g in order))
            assert counts["n_rescheduled"] == int((tail >= 0).sum()) and counts["n_unscheduled"] == int((tail < 0).sum())
            checked += len(ev)
            r.close()
        assert checked > 20
        o.close()


def _kat_order_tie():
    # three identical empty nodes, insertion order a1(A), b1(B), a2(A): live order [a1, b1, a2], so Z (first pod, ties) -> a1.
    # Drain a1: removeNode order [a2, b1] -> Z -> a2.  Recomputed ([b1, a2]) or live-minus-D ([b1, a2]) orders give b1.
    return _compile([_node("a1", "A"), _node("b1", "B"), _node("a2", "A")], [_pod("z")])


def _kat_counter():
    # X and Y: app=x, required anti-affinity to app=x over zones.  X -> a1 (ties), Y -> b1 (zone A holds X).  Drain a1: with X's
    # increments released, zone A is free again -> X -> a2; without the release a2 (zone A) and b1 (Y) both fail: unschedulable.
    lab = {"app": "x"}
    return _compile([_node("a1", "A"), _node("b1", "B"), _node("a2", "A")],
                    [_pod("x", labels=lab, anti=[lab]), _pod("y", labels=lab, anti=[lab])])


def _kat_classes():
    # Z (plain, anti-affinity over zones to role=bound) -> a1 (b1 is tainted, a1 first); B is pre-bound to a1 afterwards and carries
    # role=bound; DaemonSet d runs on a1 only (pool=x).  Drain a1: d -> n_daemon, B -> n_bound, neither placed; Z -> a2 only if B's
    # zone-A count was released (b1 stays tainted).
    taint = [{"key": "t", "value": "y", "effect": "NoSchedule"}]
    ds = {"apiVersion": "apps/v1", "kind": "DaemonSet", "metadata": {"name": "d", "namespace": "kube-system"},
          "spec": {"selector": {"matchLabels": {"ds": "d"}}, "template": {"metadata": {"labels": {"ds": "d"}}, "spec": {
              "nodeSelector": {"pool": "x"},
              "containers": [{"name": "c", "image": "d:v1", "resources": {"requests": {"cpu": "100m", "memory": "64Mi"}}}]}}}}
    return _compile([_node("a1", "A", labels={"pool": "x"}), _node("b1", "B", taints=taint), _node("a2", "A")],
                    [_pod("z", anti=[{"role": "bound"}]), _pod("b", labels={"role": "bound"}, node_name="a1")], [ds])


def _oracle_drain_by_name(p, c, names):
    from drain_oracle import DrainOracle as Oracle
    from simon_b200.drain import survivor_order
    o = Oracle(c)
    live = o.schedule()
    order = survivor_order(c, [c.node_index(n) for n in names])
    res = o.drain(live, order)
    o.close()
    return live, order, res


def test_kat_order_tie():
    p, c = _kat_order_tie()
    live, order, (counts, pod, node, fc, sums) = _oracle_drain_by_name(p, c, ["a1"])
    assert c.node_names[live[0]] == "a1"
    assert counts["n_evicted"] == 1 and list(pod) == [0] and c.node_names[node[0]] == "a2"


def test_kat_counter_decrement():
    p, c = _kat_counter()
    live, order, (counts, pod, node, fc, sums) = _oracle_drain_by_name(p, c, ["a1"])
    assert _names(c, live) == ["a1", "b1"]
    assert list(pod) == [0] and c.node_names[node[0]] == "a2" and counts["n_unscheduled"] == 0


def test_kat_classification():
    p, c = _kat_classes()
    live, order, (counts, pod, node, fc, sums) = _oracle_drain_by_name(p, c, ["a1"])
    kinds = [r.tmpl.workload_kind for r in p.pods]
    assert _names(c, live) == ["a1", "a1", "a1"] and kinds[2] == "DaemonSet"
    assert counts == dict(n_evicted=1, n_rescheduled=1, n_unscheduled=0, n_daemon=1, n_bound=1)
    assert list(pod) == [0] and c.node_names[node[0]] == "a2"
    # the pods left behind still count on the survivors: Z's 100m on a2, nothing else
    assert sums["req_mcpu"] == 100 and sums["alloc_mcpu"] == 8000


# ---- Python layer without a device ---------------------------------------------------------------------------------------------
def _small_cluster():
    return synth.make_c2(n_nodes=10, n_workloads=2, replicas=3)


def test_drain_rejects_bad_node_names():
    from simon_b200.drain import Drain
    cluster, apps = _small_cluster()
    name = O.name_of(cluster.Nodes[0])
    with pytest.raises(ValueError):
        Drain(cluster, apps, [["no-such-node"]])
    with pytest.raises(ValueError):
        Drain(cluster, apps, [[name, name]])
    with pytest.raises(ValueError):
        Drain(cluster, apps, None, bound_pods="keep")


def test_drain_needs_a_device():
    import torch
    from simon_b200.drain import Drain
    from simon_b200.engine import EngineUnavailable
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    cluster, apps = _small_cluster()
    with pytest.raises(EngineUnavailable):
        Drain(cluster, apps)


# ---- GPU: engine == oracle ------------------------------------------------------------------------------------------------------
def _case_sets(c, rng, n_multi=29):
    """Every single-node drain, a whole zone, the empty set, all nodes but one, and random multi-node sets (32 multi-node sets)."""
    from simon_b200.drain import survivor_order
    N = c.n_nodes
    sets = [[g] for g in range(N)]
    zones = {}
    for g in range(N):
        zones.setdefault(get_zone_key(c.node_objs[g]), []).append(g)
    sets.append(max(zones.values(), key=len))
    sets.append([])
    sets.append(list(range(1, N)))
    for _ in range(n_multi):
        sets.append(rng.sample(range(N), rng.randint(2, max(2, min(N - 1, 8)))))
    return sets, [survivor_order(c, s) for s in sets]


def _engine_vs_oracle(c, sets, orders, **engine_kw):
    from drain_oracle import DrainOracle as Oracle
    from simon_b200.engine import Engine
    o = Oracle(c)
    live = o.schedule()
    with Engine(c, device=0, **engine_kw) as eng:
        out = eng.schedule()[0]
        np.testing.assert_array_equal(out, live)
        res, off, pod, node, fc = eng.drain(orders)
    for s, order in enumerate(orders):
        counts, rpod, rnode, rfc, sums = o.drain(live, order)
        got = {k: res[s][k] for k in counts}
        assert got == counts, (s, sets[s])
        assert {k: res[s][k] for k in sums} == sums, (s, sets[s])
        a, b = int(off[s]), int(off[s + 1])
        np.testing.assert_array_equal(pod[a:b], rpod)
        np.testing.assert_array_equal(node[a:b], rnode)
        np.testing.assert_array_equal(fc[a:b], rfc)
    o.close()
    return res


@pytest.mark.gpu
def test_gpu_drain_matches_oracle_mix():
    rng = random.Random(3)
    n_ev = 0
    for seed in range(100, 122):
        _p, c = make_case("mix", seed_no=seed)
        sets, orders = _case_sets(c, rng)
        res = _engine_vs_oracle(c, sets, orders)
        n_ev += sum(r["n_evicted"] for r in res)
    for build in (_kat_order_tie, _kat_counter, _kat_classes):
        _p, c = build()
        sets, orders = _case_sets(c, rng, n_multi=2)
        _engine_vs_oracle(c, sets, orders)
    assert n_ev > 1000


@pytest.mark.gpu
def test_gpu_drain_matches_oracle_c2_1000_nodes():
    _p, c = make_case("c2", n_nodes=1000, n_workloads=100, replicas=60)
    sets, orders = _case_sets(c, random.Random(4))
    res = _engine_vs_oracle(c, sets, orders)
    assert sum(r["n_evicted"] for r in res) > 1000


@pytest.mark.gpu
def test_gpu_drain_matches_oracle_c3_3000_nodes():
    _p, c = make_case("c3", n_nodes=3000, n_workloads=300, replicas=100, n_apps=2, seed_no=3)
    sets, orders = _case_sets(c, random.Random(5))
    res = _engine_vs_oracle(c, sets, orders)
    assert sum(r["n_evicted"] for r in res) > 3000


@pytest.mark.gpu
def test_gpu_drain_results_do_not_depend_on_the_batch(monkeypatch):
    from simon_b200.engine import Engine
    _p, c = make_case("mix", seed_no=111)
    sets, orders = _case_sets(c, random.Random(6))
    with Engine(c, device=0) as eng:
        eng.schedule()
        whole = eng.drain(orders)
        single = [eng.drain([o]) for o in orders]
        monkeypatch.setenv("SIMON_DRAIN_CHUNK", "3")
        chunked = eng.drain(orders)
    for r in (chunked,):
        assert [{k: v for k, v in x.items() if k != "elapsed_ms"} for x in r[0]] == \
               [{k: v for k, v in x.items() if k != "elapsed_ms"} for x in whole[0]]
        for a, b in zip(r[1:], whole[1:]):
            np.testing.assert_array_equal(a, b)
    for s, one in enumerate(single):
        a, b = int(whole[1][s]), int(whole[1][s + 1])
        assert {k: v for k, v in one[0][0].items() if k != "elapsed_ms"} == {k: v for k, v in whole[0][s].items() if k != "elapsed_ms"}
        np.testing.assert_array_equal(one[2], whole[2][a:b])
        np.testing.assert_array_equal(one[3], whole[3][a:b])
        np.testing.assert_array_equal(one[4], whole[4][a:b])


@pytest.mark.gpu
def test_gpu_drain_leaves_the_live_state_alone():
    from simon_b200 import moves as M
    from simon_b200.engine import Engine
    _p, c = make_case("mix", seed_no=113)
    sets, orders = _case_sets(c, random.Random(7))
    with Engine(c, device=0) as eng:
        out = eng.schedule()[0]
        mv = M.sample_moves(len(out), c.n_nodes, 500, seed=2, placement=out)

        def snapshot():
            eng.moves_upload(mv)
            m = eng.moves_run(k=8)
            return eng.state(), eng.state_ext(), eng.results(), m

        before = snapshot()
        first = eng.drain(orders)
        after = snapshot()
        second = eng.drain(orders)
    for a, b in zip(before[:2], after[:2]):
        for k in a:
            np.testing.assert_array_equal(a[k], b[k])
    np.testing.assert_array_equal(before[2], after[2])
    np.testing.assert_array_equal(before[3]["gain"], after[3]["gain"])
    np.testing.assert_array_equal(before[3]["code"], after[3]["code"])
    assert before[3]["topk"] == after[3]["topk"]
    for a, b in zip(first[1:], second[1:]):
        np.testing.assert_array_equal(a, b)


@pytest.mark.gpu
def test_gpu_drain_needs_the_live_state():
    from simon_b200.engine import Engine
    _p, c = make_case("mix", seed_no=102)
    order = [np.arange(1, c.n_nodes, dtype=np.uint32)]
    with Engine(c, device=0) as eng:
        with pytest.raises(RuntimeError, match="error -3"):
            eng.drain(order)                    # nothing scheduled yet
        eng.schedule()
        eng.drain(order)
        eng.reset()
        with pytest.raises(RuntimeError, match="error -3"):
            eng.drain(order)
        eng.schedule(0, c.pods_dims["n_pods"] // 2)
        with pytest.raises(RuntimeError, match="error -3"):
            eng.drain(order)
        eng.schedule(c.pods_dims["n_pods"] // 2)
        eng.drain(order)                        # the two halves in order make a complete live run
        with pytest.raises(RuntimeError, match="error -1"):
            eng.drain([np.array([0, 0], np.uint32)])


@pytest.mark.gpu
def test_gpu_drain_api_on_the_reference_example():
    """Drain() over the reference example (demo_1 with the simple and complicate apps), every node alone: each outcome is the
    oracle's drain, and each failure text is FitError's over the survivors."""
    from drain_oracle import DrainOracle as Oracle
    from simon_b200.drain import Drain, pod_kinds, survivor_order
    base = os.path.join(ROOT, "tests", "golden", "example")
    cluster = O.create_cluster_resource_from_cluster_config(os.path.join(base, "cluster", "demo_1"))
    apps = [O.AppResource(nm, O.get_object_from_yaml_content(O.get_yaml_content_from_directory(os.path.join(base, "application", d))))
            for nm, d in (("simple", "simple"), ("complicated", "complicate"))]
    res = Drain(cluster, apps)
    p = simulator.plan(cluster, apps)
    c = compile_cluster(p.nodes, p.pods, p.ctx)
    o = Oracle(c)
    live = o.schedule()
    daemon, bound = pod_kinds(c)
    assert len(res.Drains) == len(cluster.Nodes)
    for nd, out in zip(cluster.Nodes, res.Drains):
        assert out.Nodes == [O.name_of(nd)]
        g = c.node_index(O.name_of(nd))
        order = survivor_order(c, [g])
        counts, pod, node, fc, sums = o.drain(live, order)
        assert [(r.name, frm, to) for r, frm, to in out.Evicted] == \
               [(p.pods[q].name, c.node_names[g], c.node_names[n] if n >= 0 else None) for q, n in zip(pod, node)]
        assert len(out.DaemonSetPods) == counts["n_daemon"] and len(out.BoundPods) == counts["n_bound"]
        assert out.Occupancy == sums
        want = [simulator.format_fit_error(c, p.pods[q], fc[j], active=[int(x) for x in order]) for j, q in enumerate(pod) if node[j] < 0]
        assert [u.Reason for u in out.UnscheduledPods] == want
        for u in out.UnscheduledPods:
            assert f"0/{c.n_nodes - 1} nodes are available" in u.Reason
    o.close()
