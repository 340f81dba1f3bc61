"""The NATIVE host side (csrc/simon_host.cpp + csrc/host/*.h, inside libsimon_gpu.so) against its Python mirror.

The reference's host side is compiled Go; without a Go toolchain the drop-in host side is C++ behind the C ABI
(include/simon_gpu.h: simon_host_compile / simon_host_simulate).  The Python package stays as the test-side mirror, so parity of
the native path is asserted here at three levels:
  * resource.Quantity (parse / Value / MilliValue / AsApproximateFloat64) against simon_b200/quantity.py (whose arithmetic the
    hand-derived Simon KAT pins) on a sweep of quantity strings, incl. the inf.Dec fallbacks and the error cases;
  * the compiled columns: every array and dimension of simon_snapshot / simon_podset, node order, pod order and identity, for
    synthetic clusters (C2 / C3 shapes, 40 random feature mixes with DaemonSets, GPU share, images), the hand-derived plugin KATs,
    the DaemonSet cluster and the reference's own example cluster + applications (config 1, stored in tests/golden/example/);
  * (-m gpu) simulator.Simulate: simon_host_simulate == simon_b200.simulator.Simulate: per-node pod lists in placement order and
    every UnscheduledPod reason string.
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))

from simon_b200 import native_host, simulator, synth  # noqa: E402
from simon_b200.compiler import compile_cluster  # noqa: E402
from simon_b200.objects import AppResource, ResourceTypes  # noqa: E402


def _diff(cluster, apps):
    """-> list of differences between the Python compiler and the native one (empty = identical)."""
    p = simulator.plan(cluster, apps)
    c = compile_cluster(p.nodes, p.pods, p.ctx)
    n = native_host.compile_native(cluster, apps)
    bad = []
    if n.node_names != list(c.node_names):
        bad.append("node_names")
    if list(n.node_orig_index) != list(c.node_orig_index):
        bad.append("node_orig_index")
    if n.scalar_names != list(c.scalar_names):
        bad.append("scalar_names")
    for k, v in c.snap_dims.items():
        if int(n.snap_dims[k]) != int(v):
            bad.append(f"snap_dims.{k}: {n.snap_dims[k]} != {v}")
    for k, v in c.pods_dims.items():
        if int(n.pods_dims[k]) != int(v):
            bad.append(f"pods_dims.{k}: {n.pods_dims[k]} != {v}")
    for name, mine, theirs in (("snap", c.snap, n.snap), ("pods", c.pods, n.pods)):
        for k, v in mine.items():
            a, b = np.asarray(v), theirs[k]
            if a.shape != b.shape or not np.array_equal(a.astype(b.dtype), b):
                bad.append(f"{name}.{k} {a.shape} vs {b.shape}")
    if [r.key() for r in p.pods] != n.pod_keys():
        bad.append("pod order / identity")
    segs = [(s["name"], s["first"], s["count"]) for s in n.info["segments"]]
    if segs != [(s[0], s[1], s[2]) for s in p.segments]:
        bad.append("segments")
    return bad


def _kat_inputs(kat):
    cluster = ResourceTypes()
    cluster.Nodes.extend(kat["nodes"])
    cluster.Pods.extend(kat["running"])
    cluster.Services.extend(kat["services"])
    app = AppResource("kat", ResourceTypes())
    app.Resource.Pods.extend(kat["pod"] if isinstance(kat["pod"], list) else [kat["pod"]])
    apps = [app]
    if kat.get("pod2"):
        app2 = AppResource("kat2", ResourceTypes())
        app2.Resource.Pods.extend(kat["pod2"])
        apps.append(app2)
    return cluster, apps


def test_native_host_symbols_are_exported():
    L = native_host.lib()
    for name in ("simon_host_compile", "simon_host_plan_free", "simon_host_plan_columns", "simon_host_plan_describe",
                 "simon_host_simulate", "simon_host_free", "simon_host_last_error", "simon_host_quantity_probe", "simon_host_plan_fit_error", "simon_host_capacity_search"):
        assert hasattr(L, name)


QUANTITIES = ["0", "1", "100m", "1500m", "0.5", "1.5", "2.75", "4", "64", "16Gi", "1.5Gi", "0.5Mi", "128974848", "129e6", "129M", "123Mi",
              "1e3", "1E3", "1e-3", "5e-1", "100Ki", "1Ti", "2Pi", "1Ei", "7Ei", "8Ei", "9223372036854775807", "9223372036854775808",
              "92233720368547758070", "1n", "1u", "999u", "1000000n", "0.000000001", "0.0000000001", "+3", "-3", "-1500m", "-0.5Gi",
              "12345678901234567890123", "1.000000000000000001", "3.14159Gi", "100000000000000000000m", "1k", "1M", "1G", "1T", "1P",
              "1E", "9E", "10E", "0.1Ki", "1.0", "01", "00.50", ".5", "5.", "1.5e3", "1.5E+3", "250Mi", "32", "110", "3900m", "15258Mi", "e3", "Gi", "m"]
BAD_QUANTITIES = ["", "abc", "1.2.3", "1Kii", "1 Gi", "--1", "1e", "1ee3", "1mi", "1e3e", "1.5.Gi"]


@pytest.mark.parametrize("text", QUANTITIES)
def test_native_quantity_matches_the_python_restatement(text):
    from simon_b200.quantity import Quantity
    q = Quantity.parse(text)
    L = native_host.lib()
    L.simon_host_quantity_probe.restype = C.c_int
    L.simon_host_quantity_probe.argtypes = [C.c_char_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_double)]
    v, m, a = C.c_int64(0), C.c_int64(0), C.c_double(0)
    want_v, want_m = q.int_value(), q.milli_value()
    assert L.simon_host_quantity_probe(text.encode(), None, None, C.byref(a)) == 0, L.simon_host_last_error()
    assert a.value == q.as_approximate_float64()          # bit-identical doubles
    for want, ref in ((want_v, v), (want_m, m)):
        rc = L.simon_host_quantity_probe(text.encode(), C.byref(ref) if ref is v else None, C.byref(ref) if ref is m else None, None)
        if -(1 << 63) <= want < (1 << 63):
            assert rc == 0 and ref.value == want
        else:
            assert rc != 0          # beyond int64: refused, never wrapped


@pytest.mark.parametrize("text", BAD_QUANTITIES)
def test_native_quantity_rejects_what_the_python_restatement_rejects(text):
    from simon_b200.quantity import Quantity, QuantityError
    with pytest.raises(QuantityError):
        Quantity.parse(text)
    L = native_host.lib()
    L.simon_host_quantity_probe.restype = C.c_int
    L.simon_host_quantity_probe.argtypes = [C.c_char_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_double)]
    v = C.c_int64(0)
    assert L.simon_host_quantity_probe(text.encode(), C.byref(v), None, None) != 0


def test_native_columns_match_python_c3_and_c2_shapes():
    assert _diff(*synth.make_c3(n_nodes=300, n_workloads=60, replicas=10, n_apps=2, seed_no=7)) == []
    assert _diff(*synth.make_c3(n_nodes=1200, n_workloads=120, replicas=12, n_apps=3, seed_no=11)) == []
    assert _diff(*synth.make_c2(n_nodes=100, n_workloads=10, replicas=10)) == []


@pytest.mark.parametrize("seed", list(range(100, 140)))
def test_native_columns_match_python_on_random_feature_mixes(seed):
    assert _diff(*synth.make_mix(seed_no=seed, n_nodes=30 + 10 * (seed % 4), n_workloads=25, max_replicas=5,
                                 with_images=bool(seed % 3 == 0))) == []


def test_native_columns_match_python_on_the_plugin_kats():
    import kat_plugins
    for name, kat in kat_plugins.CASES.items():
        assert _diff(*_kat_inputs(kat)) == [], name


def test_native_columns_match_python_on_the_daemonset_cluster():
    import test_daemonset_pins as T
    assert _diff(*T._cluster()) == []


@pytest.mark.parametrize("case", ["simple", "complicate", "more_pods", "gpushare", "config_sequence"])
def test_native_compiles_the_reference_example_inputs_to_the_stored_columns(case):
    """BASELINE config 1: example/cluster/demo_1 x example/application/* through the NATIVE compiler == the columns stored in
    tests/golden/config1_<case>.npz (which the oracle, the object-level restatement and the engine are pinned to)."""
    import make_config1
    from simon_b200 import objects as O
    cluster = O.create_cluster_resource_from_cluster_config(os.path.join(make_config1.REF, "cluster", "demo_1"))
    apps = [O.AppResource(a, O.get_object_from_yaml_content(O.get_yaml_content_from_directory(
        os.path.join(make_config1.REF, "application", a)))) for a in make_config1.CASES[case]]
    n = native_host.compile_native(cluster, apps)
    z = np.load(os.path.join(HERE, "golden", f"config1_{case}.npz"))
    for k in z.files:
        if k.startswith("snap__"):
            np.testing.assert_array_equal(n.snap[k[6:]], z[k], err_msg=k)
        elif k.startswith("pods__"):
            np.testing.assert_array_equal(n.pods[k[6:]], z[k], err_msg=k)


def test_native_refusals_match_the_python_compiler():
    """Inputs the engine does not implement are refused with SIMON_ERR_LIMIT (never narrowed or ignored), like compiler.CompileError."""
    def node(name):
        return {"kind": "Node", "metadata": {"name": name, "labels": {"kubernetes.io/hostname": name}},
                "status": {"allocatable": {"cpu": "4", "memory": "8Gi", "pods": "110"}, "capacity": {"cpu": "4", "memory": "8Gi", "pods": "110"}}}

    def pod(name, **spec):
        s = {"containers": [{"name": "c", "image": "x", "resources": {"requests": {"cpu": "100m"}}}]}
        s.update(spec)
        return {"kind": "Pod", "metadata": {"name": name, "namespace": "default"}, "spec": s}

    cluster = ResourceTypes(Nodes=[node("a"), node("b")])
    # mixed priorities -> DefaultPreemption would matter
    app = AppResource("x", ResourceTypes(Pods=[pod("p1", priority=0), pod("p2", priority=10)]))
    with pytest.raises(native_host.NativeHostError) as e:
        native_host.compile_native(cluster, [app])
    assert e.value.rc == -4 and "priority" in e.value.msg
    # a StatefulSet that requests open-local storage
    sts = {"kind": "StatefulSet", "metadata": {"name": "s", "namespace": "default"},
           "spec": {"replicas": 1, "template": {"metadata": {"labels": {"a": "b"}}, "spec": pod("t")["spec"]},
                    "volumeClaimTemplates": [{"spec": {"storageClassName": "open-local-lvm", "resources": {"requests": {"storage": "1Gi"}}}}]}}
    with pytest.raises(native_host.NativeHostError) as e:
        native_host.compile_native(cluster, [AppResource("x", ResourceTypes(StatefulSets=[sts]))])
    assert e.value.rc == -4 and "open-local" in e.value.msg
    # duplicate taints on a node
    n2 = node("c")
    n2["spec"] = {"taints": [{"key": "k", "value": "v", "effect": "NoSchedule"}, {"key": "k", "value": "v", "effect": "NoSchedule"}]}
    with pytest.raises(native_host.NativeHostError) as e:
        native_host.compile_native(ResourceTypes(Nodes=[n2]), [AppResource("x", ResourceTypes(Pods=[pod("p")]))])
    assert e.value.rc == -4 and "duplicate taint" in e.value.msg
    # malformed requests
    L = native_host.lib()
    h = C.c_void_p()
    assert L.simon_host_compile(b"{not json", 9, C.byref(h)) == -1 and b"JSON" in L.simon_host_last_error()
    assert L.simon_host_compile(b"{}", 2, C.byref(h)) == -1
    # a pod without containers: MakeValidPod's validation error
    with pytest.raises(native_host.NativeHostError) as e:
        native_host.compile_native(cluster, [AppResource("x", ResourceTypes(Pods=[{"kind": "Pod", "metadata": {"name": "e"}, "spec": {}}]))])
    assert "spec.containers" in e.value.msg


@pytest.mark.parametrize("seed", [5, 101, 104, 107, 110, 113])
def test_native_failure_messages_match_the_python_mirror(seed):
    """FitError text for every pod of a mixed cluster (taints, node selectors / affinity incl. matchFields, cordoned nodes), with an
    empty and with a synthetic dynamic histogram: simon_host_plan_fit_error == simulator.format_fit_error."""
    cluster, apps = synth.make_mix(seed_no=seed, n_nodes=40, n_workloads=25, max_replicas=3)
    cluster.Nodes[3].setdefault("spec", {})["unschedulable"] = True
    names = [n["metadata"]["name"] for n in cluster.Nodes]
    base = {"containers": [{"name": "c", "image": "x", "resources": {"requests": {"cpu": "100m"}}}]}
    R = "requiredDuringSchedulingIgnoredDuringExecution"
    extra = [
        # matchFields (node names) and spec.nodeName defeat the per-node-group memo of the native path
        {"kind": "Pod", "metadata": {"name": "by-field", "namespace": "default"}, "spec": dict(base, affinity={"nodeAffinity": {R: {
            "nodeSelectorTerms": [{"matchFields": [{"key": "metadata.name", "operator": "In", "values": [names[5]]}]},
                                  {"matchExpressions": [{"key": "kubernetes.io/hostname", "operator": "NotIn", "values": names[:7]}]}]}}})},
        {"kind": "Pod", "metadata": {"name": "by-name", "namespace": "default"}, "spec": dict(base, nodeName=names[2])},
        {"kind": "Pod", "metadata": {"name": "tolerant", "namespace": "default"}, "spec": dict(
            base, tolerations=[{"operator": "Exists"}], nodeSelector={"no-such-label": "x"})},
        {"kind": "Pod", "metadata": {"name": "cordon-ok", "namespace": "default"}, "spec": dict(
            base, tolerations=[{"key": "node.kubernetes.io/unschedulable", "operator": "Exists", "effect": "NoSchedule"}])},
    ]
    apps.append(AppResource("extra", ResourceTypes(Pods=extra)))
    p = simulator.plan(cluster, apps)
    c = compile_cluster(p.nodes, p.pods, p.ctx)
    L = native_host.lib()
    L.simon_host_plan_fit_error.restype = C.c_int
    L.simon_host_plan_fit_error.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.POINTER(C.c_void_p)]
    req = native_host.request_json(cluster, apps)
    h = C.c_void_p()
    assert L.simon_host_compile(req, len(req), C.byref(h)) == 0
    try:
        counts = np.zeros(24, np.uint32)
        counts[[1, 2, 3, 4, 5, 14, 15, 16, 17, 18]] = [1, 2, 3, 4, 5, 6, 7, 8, 9, 10]
        for k in range(len(c.scalar_names)):
            counts[6 + k] = 11 + k
        seen = set()
        for i, rec in enumerate(p.pods):
            if id(rec.tmpl) in seen:
                continue
            seen.add(id(rec.tmpl))
            for cnt in (np.zeros(24, np.uint32), counts):
                out = C.c_void_p()
                assert L.simon_host_plan_fit_error(h, i, cnt.ctypes.data, C.byref(out)) == 0
                got = C.string_at(out).decode()
                L.simon_host_free(out)
                assert got == simulator.format_fit_error(c, rec, cnt)
    finally:
        L.simon_host_plan_free(h)


def test_native_simulate_needs_a_device():
    """No CPU scheduling path: without a CUDA device the native Simulate fails loudly (SIMON_ERR_CUDA), like Engine()."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    cluster, apps = synth.make_c2(n_nodes=10, n_workloads=2, replicas=3)
    with pytest.raises(native_host.NativeHostError) as e:
        native_host.simulate_native(cluster, apps)
    assert e.value.rc == -2


def _simulate_both(cluster, apps):
    import copy
    res = simulator.Simulate(copy.deepcopy(cluster), copy.deepcopy(apps))
    nat = native_host.simulate_native(cluster, apps)
    t = nat["templates"]
    keys = []
    for ti, name, o in zip(nat["podTemplate"], nat["podName"], nat["podOrdinal"]):
        tt = t[ti]
        keys.append((tt["kind"], tt["namespace"], name if tt["kind"] == "Pod" else tt["workload"], o))
    assert nat["nodes"] == [(s.Node.get("metadata") or {}).get("name") for s in res.NodeStatus]
    for i, st in enumerate(res.NodeStatus):
        assert [keys[k] for k in nat["nodeStatus"][i]] == [r.key() for r in st.Pods], nat["nodes"][i]
    assert [(keys[u["pod"]], u["reason"]) for u in nat["unscheduledPods"]] == [(u.Pod.key(), u.Reason) for u in res.UnscheduledPods]
    return res, nat


@pytest.mark.gpu
def test_native_simulate_matches_python_simulate_gpu():
    res, nat = _simulate_both(*synth.make_c3(n_nodes=300, n_workloads=60, replicas=10, n_apps=2, seed_no=7))
    assert sum(len(x) for x in nat["nodeStatus"]) + len(nat["unscheduledPods"]) == len(nat["podNode"])
    assert len(nat["unscheduledPods"]) > 0          # the case exercises the failure messages
    # a small, over-committed cluster: most messages are resource reasons
    _simulate_both(*synth.make_c2(n_nodes=20, n_workloads=10, replicas=30))


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [100, 101, 102, 103, 104, 105, 106, 107])
def test_native_simulate_matches_python_on_feature_mixes_gpu(seed):
    _simulate_both(*synth.make_mix(seed_no=seed, n_nodes=30 + 10 * (seed % 4), n_workloads=25, max_replicas=5, with_images=bool(seed % 2)))


@pytest.mark.gpu
def test_native_simulate_gpu_share_failure_names_the_nodes_gpu():
    """Open-Gpu-Share failure reasons name each rejecting node (pkg/simulator/plugin/open-gpu-share.go:66-79): the native path
    collects them with the per-node verdict dump exactly as the Python mirror does."""
    import kat_plugins
    kat = kat_plugins.CASES["gpu_share_per_device_fit"]
    cluster, apps = _kat_inputs(kat)
    big = dict(kat["pod"][0] if isinstance(kat["pod"], list) else kat["pod"])
    big = __import__("copy").deepcopy(big)
    big["metadata"]["name"] = "too-big"
    big["metadata"].setdefault("annotations", {})["alibabacloud.com/gpu-mem"] = "1024Gi"
    apps[0].Resource.Pods.append(big)
    res, nat = _simulate_both(cluster, apps)
    assert any("Node:" in u["reason"] for u in nat["unscheduledPods"])


def _c4_small():
    cluster, apps, specs = synth.make_c4(n_nodes=60, n_workloads=6, replicas=12, seed_no=4)
    specs = specs[:3]
    # a spec WITHOUT labels: utils.NewFakeNodes mutates its template across copies (pkg/utils/utils.go:890-899), so the first copy has
    # no hostname label and the later ones do - both host sides must reproduce that
    bare = {"kind": "Node", "metadata": {"name": "bare-spec"}, "status": dict(specs[0]["status"])}
    return cluster, apps, specs + [bare]


def test_native_capacity_scenarios_match_python():
    """simon_host_capacity_search (dryRun): superset cluster and per-scenario node lists == capacity.build_scenarios."""
    import copy
    from simon_b200 import capacity
    cluster, apps, specs = _c4_small()
    ks = [0, 1, 2, 4, 8]
    ss = capacity.build_scenarios(copy.deepcopy(cluster), copy.deepcopy(apps), copy.deepcopy(specs), ks=ks)
    nat = native_host.capacity_search_native(cluster, apps, specs, ks, dry_run=True)
    assert nat["nodeNames"] == list(ss.compiled.node_names) and nat["nBase"] == ss.n_base and nat["nScenarios"] == len(ss.scenarios)
    assert [(a["sid"], a["spec"], a["k"], a["nodes"]) for a in nat["scenarios"]] == [(b.sid, b.spec, b.k, b.nodes.tolist()) for b in ss.scenarios]
    shard = native_host.capacity_search_native(cluster, apps, specs, ks, dry_run=True, rank=1, world=3)
    assert [a["sid"] for a in shard["scenarios"]] == [b.sid for b in ss.scenarios if b.sid % 3 == 1]
    assert shard["bestKey"] == 1 << 62


@pytest.mark.gpu
def test_native_capacity_search_matches_python_gpu():
    """Same scenarios, same device results, same packed key as capacity.search with the GPU runner (and so as the oracle, which
    tests/test_capacity.py pins that path to)."""
    import copy
    from simon_b200 import capacity
    cluster, apps, specs = _c4_small()
    ks = [0, 1, 2, 4, 8]
    ss = capacity.build_scenarios(copy.deepcopy(cluster), copy.deepcopy(apps), copy.deepcopy(specs), ks=ks)
    best, by_sid = capacity.search(ss, capacity.gpu_runner(0), max_cpu=100, max_mem=100)
    nat = native_host.capacity_search_native(cluster, apps, specs, ks, max_cpu=100, max_mem=100)
    assert nat["bestKey"] == best
    for a in nat["scenarios"]:
        r = by_sid[a["sid"]]
        assert all(int(a[q]) == int(r[q]) for q in ("n_unscheduled", "n_scheduled", "req_mcpu", "alloc_mcpu", "req_mem", "alloc_mem")), a
    # two ranks: the MIN of the local keys is the global key
    k0 = native_host.capacity_search_native(cluster, apps, specs, ks, rank=0, world=2)["bestKey"]
    k1 = native_host.capacity_search_native(cluster, apps, specs, ks, rank=1, world=2)["bestKey"]
    assert min(k0, k1) == best
    # occupancy caps (satisfyResourceSetting) move the answer the same way on both sides
    best50, _ = capacity.search(ss, capacity.gpu_runner(0), max_cpu=50, max_mem=100)
    assert native_host.capacity_search_native(cluster, apps, specs, ks, max_cpu=50, max_mem=100)["bestKey"] == best50


def test_native_host_survives_malformed_requests():
    """Truncated and corrupted requests come back as error codes with a message - no crash, no exception across the C boundary
    (the cgo rule of include/simon_gpu.h) - and well-formed but odd JSON (escapes, nesting, number forms) parses like json.loads."""
    import random
    cluster, apps = synth.make_mix(seed_no=103, n_nodes=12, n_workloads=8, max_replicas=2)
    req = native_host.request_json(cluster, apps)
    L = native_host.lib()
    rng = random.Random(7)
    for _ in range(150):
        cut = rng.randrange(1, len(req) - 1)
        h = C.c_void_p()
        rc = L.simon_host_compile(req[:cut], cut, C.byref(h))
        assert rc != 0 and not h and L.simon_host_last_error()
    ok = 0
    for _ in range(150):
        b = bytearray(req)
        for _k in range(rng.randrange(1, 4)):
            b[rng.randrange(len(b))] = rng.choice(b'{}[]",:0a\\ ')
        h = C.c_void_p()
        rc = L.simon_host_compile(bytes(b), len(b), C.byref(h))
        if rc == 0:
            ok += 1
            L.simon_host_plan_free(h)
        else:
            assert L.simon_host_last_error()
    # a request large enough for the multi-threaded array parser (elements parsed by worker threads): errors inside an element,
    # between elements and truncation must all surface as error codes
    big_cluster, big_apps = synth.make_c3(n_nodes=1500, n_workloads=30, replicas=5, n_apps=1, seed_no=9)
    big = native_host.request_json(big_cluster, big_apps)
    assert len(big) > (1 << 19)
    h = C.c_void_p()
    assert L.simon_host_compile(big, len(big), C.byref(h)) == 0
    L.simon_host_plan_free(h)
    for _ in range(40):
        b = bytearray(big)
        if rng.random() < 0.5:
            b = b[:rng.randrange(1, len(b) - 1)]
        else:
            for _k in range(rng.randrange(1, 3)):
                b[rng.randrange(len(b))] = rng.choice(b'{}[]",:\\')
        h = C.c_void_p()
        rc = L.simon_host_compile(bytes(b), len(b), C.byref(h))
        if rc == 0:
            L.simon_host_plan_free(h)
        else:
            assert L.simon_host_last_error()
    # escapes / unicode / exponent numbers in names and quantities
    node = {"kind": "Node", "metadata": {"name": "n\u00e9-\"q\"\\\t\U0001F600", "labels": {"k": "v"}},
            "status": {"allocatable": {"cpu": 4, "memory": 8.0e9, "pods": "110"}, "capacity": {"cpu": 4, "memory": 8.0e9, "pods": "110"}}}
    pod = {"kind": "Pod", "metadata": {"name": "p", "namespace": "default"},
           "spec": {"containers": [{"name": "c", "image": "x", "resources": {"requests": {"cpu": 0.5, "memory": 1e9}}}]}}
    cl, ap = ResourceTypes(Nodes=[node]), [AppResource("a", ResourceTypes(Pods=[pod]))]
    assert _diff(cl, ap) == []
    n = native_host.compile_native(cl, ap)
    assert n.node_names == [node["metadata"]["name"]] and int(n.snap["alloc_mem"][0]) == 8_000_000_000


def test_native_columns_match_python_on_rarely_used_object_shapes():
    """Branches the synthetic generators seldom reach: init containers and pod overhead, host ports (incl. hostIP / protocol), extended and
    hugepages resources, templates that preset spec.nodeName, Jobs and CronJobs (completions), a Service with an empty selector, ReplicaSet
    / StatefulSet owners for the default spread selector, spread constraints with a null selector, (anti)affinity terms with explicit
    namespaces, every node-selector operator incl. Gt / Lt and invalid ones, fractional / exponent / binary quantities, zone labels in
    their beta spelling, nodes without labels, duplicate node names."""
    R, P = "requiredDuringSchedulingIgnoredDuringExecution", "preferredDuringSchedulingIgnoredDuringExecution"

    def node(name, cpu="8", mem="16Gi", labels=None, taints=None, extra_alloc=None, unsched=False):
        alloc = {"cpu": cpu, "memory": mem, "pods": "110", "ephemeral-storage": "100Gi"}
        alloc.update(extra_alloc or {})
        n = {"kind": "Node", "metadata": {"name": name}, "status": {"allocatable": alloc, "capacity": dict(alloc)}}
        if labels is not None:
            n["metadata"]["labels"] = labels
        if taints or unsched:
            n["spec"] = {}
            if taints:
                n["spec"]["taints"] = taints
            if unsched:
                n["spec"]["unschedulable"] = True
        return n

    nodes = [
        node("a", labels={"kubernetes.io/hostname": "a", "failure-domain.beta.kubernetes.io/zone": "z1", "failure-domain.beta.kubernetes.io/region": "r1",
                          "tier": "gold", "gen": "7"}, extra_alloc={"example.com/fpga": "2", "hugepages-2Mi": "1Gi"}),
        node("b", cpu="7500m", mem="15.5Gi", labels={"kubernetes.io/hostname": "b", "topology.kubernetes.io/zone": "z2", "tier": "silver", "gen": "12"},
             taints=[{"key": "dedicated", "value": "x", "effect": "NoSchedule"}, {"key": "flaky", "effect": "PreferNoSchedule"}]),
        node("c", cpu="16", mem="64e9", labels={"kubernetes.io/hostname": "c", "topology.kubernetes.io/zone": "z1", "gen": "abc"},
             taints=[{"key": "evict", "value": "now", "effect": "NoExecute"}]),
        node("d", cpu="4", mem="8Gi"),                                  # no labels at all
        node("e", cpu="0.5", mem="512Mi", labels={"kubernetes.io/hostname": "e", "tier": "gold"}, unsched=True),
        node("a", cpu="64", labels={"kubernetes.io/hostname": "dup"}),    # duplicate name: skipped by nodeTree
    ]

    def tmpl(labels, **spec):
        s = {"containers": [{"name": "c", "image": "img", "resources": {"requests": {"cpu": "250m", "memory": "256Mi"}}}]}
        s.update(spec)
        return {"metadata": {"labels": labels}, "spec": s}

    heavy = tmpl({"app": "heavy"},
                 initContainers=[{"name": "i", "image": "init", "resources": {"requests": {"cpu": "2", "memory": "1Gi", "example.com/fpga": "1"}}}],
                 containers=[{"name": "c1", "image": "img1", "resources": {"requests": {"cpu": "0.3", "memory": "1e8", "hugepages-2Mi": "128Mi"}},
                              "ports": [{"containerPort": 80, "hostPort": 8080}, {"containerPort": 81, "hostPort": 8081, "hostIP": "10.0.0.1", "protocol": "UDP"}]},
                             {"name": "c2", "image": "img2", "resources": {"requests": {"ephemeral-storage": "1Gi"}, "limits": {"cpu": "1"}}}],
                 overhead={"cpu": "100m", "memory": "64Mi"})
    sel = tmpl({"app": "sel", "team": "t"}, nodeSelector={"tier": "gold"}, tolerations=[{"key": "dedicated", "operator": "Equal", "value": "x"}],
               affinity={"nodeAffinity": {
                   R: {"nodeSelectorTerms": [
                       {"matchExpressions": [{"key": "gen", "operator": "Gt", "values": ["5"]}, {"key": "tier", "operator": "NotIn", "values": ["bronze"]}]},
                       {"matchExpressions": [{"key": "gen", "operator": "Lt", "values": ["10"]}, {"key": "nope", "operator": "DoesNotExist"}]},
                       {"matchExpressions": [{"key": "gen", "operator": "Bogus", "values": ["1"]}]},
                       {}]},
                   P: [{"weight": 10, "preference": {"matchExpressions": [{"key": "tier", "operator": "Exists"}]}},
                       {"weight": 0, "preference": {"matchExpressions": [{"key": "tier", "operator": "In", "values": ["gold"]}]}},
                       {"weight": 5, "preference": {"matchFields": [{"key": "metadata.name", "operator": "NotIn", "values": ["b"]}]}}]}})
    spread = tmpl({"app": "spread"}, topologySpreadConstraints=[
        {"maxSkew": 1, "topologyKey": "topology.kubernetes.io/zone", "whenUnsatisfiable": "DoNotSchedule", "labelSelector": {"matchLabels": {"app": "spread"}}},
        {"maxSkew": 2, "topologyKey": "kubernetes.io/hostname", "whenUnsatisfiable": "ScheduleAnyway", "labelSelector": None},
        {"maxSkew": 3, "topologyKey": "tier", "whenUnsatisfiable": "ScheduleAnyway",
         "labelSelector": {"matchExpressions": [{"key": "app", "operator": "In", "values": ["spread", "sel"]}]}}])
    ipa = tmpl({"app": "ipa"}, tolerations=[{"operator": "Exists"}], affinity={
        "podAffinity": {R: [{"labelSelector": {"matchLabels": {"app": "heavy"}}, "topologyKey": "topology.kubernetes.io/zone", "namespaces": ["default", "other"]}],
                        P: [{"weight": 50, "podAffinityTerm": {"labelSelector": {"matchExpressions": [{"key": "team", "operator": "Exists"}]},
                                                               "topologyKey": "kubernetes.io/hostname"}}]},
        "podAntiAffinity": {R: [{"labelSelector": {"matchLabels": {"app": "ipa"}}, "topologyKey": "kubernetes.io/hostname"}],
                            P: [{"weight": 7, "podAffinityTerm": {"labelSelector": {"matchLabels": {"app": "spread"}}, "topologyKey": "tier",
                                                                  "namespaces": ["other"]}}]}})
    bound = tmpl({"app": "bound"}, nodeName="c")

    def wl(kind, name, template, ns="default", **spec):
        s = {"template": template}
        s.update(spec)
        return {"kind": kind, "metadata": {"name": name, "namespace": ns, "uid": "uid-" + name}, "spec": s}

    cluster = ResourceTypes(
        Nodes=nodes,
        Pods=[{"kind": "Pod", "metadata": {"name": "static-1", "namespace": "kube-system", "labels": {"app": "heavy"}},
               "spec": dict(heavy["spec"], nodeName="a")},
              {"kind": "Pod", "metadata": {"name": "ghost", "namespace": "kube-system"}, "spec": dict(tmpl({})["spec"], nodeName="no-such-node")}],
        Services=[{"kind": "Service", "metadata": {"name": "all", "namespace": "default"}, "spec": {"selector": {}}},
                  {"kind": "Service", "metadata": {"name": "sel", "namespace": "default"}, "spec": {"selector": {"app": "sel", "team": "t"}}},
                  {"kind": "Service", "metadata": {"name": "none", "namespace": "default"}, "spec": {}}],
        ReplicaSets=[wl("ReplicaSet", "rs-heavy", heavy, replicas=2, selector={"matchLabels": {"app": "heavy"}})],
        StatefulSets=[wl("StatefulSet", "sts-ipa", ipa, replicas=2, selector={"matchExpressions": [{"key": "app", "operator": "In", "values": ["ipa"]}]})],
        DaemonSets=[wl("DaemonSet", "ds", tmpl({"app": "ds"}, tolerations=[{"operator": "Exists"}], nodeSelector={"tier": "gold"}))])
    app = ResourceTypes(
        Deployments=[wl("Deployment", "d-sel", sel, replicas=3), wl("Deployment", "d-spread", spread, replicas=4), wl("Deployment", "d-bound", bound, replicas=2),
                     wl("Deployment", "d-zero", sel, replicas=0), wl("Deployment", "d-default", heavy)],
        Jobs=[wl("Job", "job", tmpl({"job": "j"}), completions=2), wl("Job", "job1", tmpl({"job": "j1"}))],
        CronJobs=[{"kind": "CronJob", "metadata": {"name": "cron", "namespace": "other"}, "spec": {"jobTemplate": {"spec": {"completions": 2, "template": ipa}}}}],
        StatefulSets=[wl("StatefulSet", "sts", spread, ns="other", replicas=2, volumeClaimTemplates=[{"spec": {"storageClassName": "standard", "resources": {"requests": {"storage": "5Gi"}}}}])],
        PodDisruptionBudgets=[{"kind": "PodDisruptionBudget", "metadata": {"name": "pdb"}, "spec": {"minAvailable": 1}}])
    assert _diff(cluster, [AppResource("first", app), AppResource("second", ResourceTypes(Deployments=[wl("Deployment", "again", ipa, replicas=2)]))]) == []
