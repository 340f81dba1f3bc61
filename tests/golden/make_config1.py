"""BASELINE config 1 from the reference's own input files, stored in tests/golden/example/ (a verbatim copy of the
open-simulator project's example/ inputs used here, Apache-2.0):

    cluster  example/cluster/demo_1           (example/simon-config.yaml:12-14 customConfig)
    apps     example/application/{simple,complicate,more_pods,gpushare}
             (the non-chart apps of example/simon-config.yaml:20-33 + the GPU-share example; open_local needs the
              Open-Local plugin, which is out of scope, and the yoda chart needs Helm rendering)

For every app (each on a fresh copy of the cluster) and for the config's own sequence simple -> complicate -> more_pods the
inputs are loaded with the repository's YAML loader, expanded and compiled; the COMPILED columns (numbers only - no
reference text) are stored in tests/golden/config1_<name>.npz together with
    * the placements of the C oracle and of the independent object-level restatement (they must agree),
    * the facts the reference itself pins for such runs (pkg/simulator/core_test.go:364-591): the number of unscheduled
      pods and the pod count per workload.
tests/test_config1.py replays the stored columns through the oracle (CPU suite) and through the CUDA engine (-m gpu);
it also re-derives the columns from the YAML and checks that nothing drifted.

    python tests/golden/make_config1.py
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (os.path.join(ROOT, "open-simulator_b200"), ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

REF = os.path.join(HERE, "example")
CASES = {
    "simple": ["simple"],
    "complicate": ["complicate"],
    "more_pods": ["more_pods"],
    "gpushare": ["gpushare"],
    "config_sequence": ["simple", "complicate", "more_pods"],     # appList order of example/simon-config.yaml
}


def build(case):
    from simon_b200 import objects as O, simulator
    from simon_b200.compiler import compile_cluster
    cluster = O.create_cluster_resource_from_cluster_config(os.path.join(REF, "cluster", "demo_1"))
    apps = [O.AppResource(a, O.get_object_from_yaml_content(O.get_yaml_content_from_directory(os.path.join(REF, "application", a))))
            for a in CASES[case]]
    p = simulator.plan(cluster, apps)
    return p, compile_cluster(p.nodes, p.pods, p.ctx)


def derive(case):
    from oracle.binding import Oracle
    from util import run_pyref
    p, c = build(case)
    o = Oracle(c)
    o_nodes, _, fc, fp = o.schedule()
    st = o.state()
    py = run_pyref(p, c)
    assert np.array_equal(o_nodes, py), f"{case}: C oracle and object-level restatement disagree"
    wl = {}
    for i, rec in enumerate(p.pods):
        k = "/".join((rec.tmpl.workload_kind, rec.tmpl.workload_namespace, rec.workload_name))
        e = wl.setdefault(k, [0, 0])
        e[0] += 1
        e[1] += int(o_nodes[i] >= 0)
    facts = {"n_pods": len(p.pods), "n_nodes": c.n_nodes, "unscheduled": int((o_nodes == -1).sum()),
             "segments": [[s[0], int(s[1]), int(s[2])] for s in p.segments],
             "node_names": list(c.node_names), "workloads": wl}
    arrays = {"out_node": o_nodes.astype(np.int32), "fail_pod": fp.astype(np.uint32), "fail_counts": fc.astype(np.uint32),
              "num_pods": st["num_pods"], "req_mcpu": st["req_mcpu"], "req_mem": st["req_mem"]}
    for k, v in c.snap.items():
        arrays["snap__" + k] = np.asarray(v)
    for k, v in c.pods.items():
        arrays["pods__" + k] = np.asarray(v)
    arrays["snap_dims"] = np.frombuffer(json.dumps({k: int(v) for k, v in c.snap_dims.items()}).encode(), dtype=np.uint8)
    arrays["pods_dims"] = np.frombuffer(json.dumps({k: int(v) for k, v in c.pods_dims.items()}).encode(), dtype=np.uint8)
    arrays["facts"] = np.frombuffer(json.dumps(facts, sort_keys=True).encode(), dtype=np.uint8)
    return arrays, facts


if __name__ == "__main__":
    for case in CASES:
        arrays, facts = derive(case)
        path = os.path.join(HERE, f"config1_{case}.npz")
        np.savez_compressed(path, **arrays)
        print(case, "pods", facts["n_pods"], "nodes", facts["n_nodes"], "unscheduled", facts["unscheduled"], os.path.getsize(path), "bytes")
