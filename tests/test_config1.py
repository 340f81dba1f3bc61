"""BASELINE config 1: the reference's own example inputs (example/cluster/demo_1 x example/application/*), compiled by
tests/golden/make_config1.py into tests/golden/config1_<case>.npz (columns + oracle placements + pinned count facts).

CPU suite : stored columns -> C oracle == stored placements; count facts; and the YAML (stored in tests/golden/example/) is
            re-loaded, re-expanded and re-compiled and must reproduce the stored columns and placements bit for bit
            (C oracle == object-level restatement is asserted by the generator).
GPU suite : stored columns -> CUDA engine (through the C ABI) == stored placements, failure histograms and aggregates.
"""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
from util import CompiledArrays  # noqa: E402

CASES = ["simple", "complicate", "more_pods", "gpushare", "config_sequence"]


def _load(case):
    z = np.load(os.path.join(HERE, "golden", f"config1_{case}.npz"))
    return z, CompiledArrays(z)


@pytest.mark.parametrize("case", CASES)
def test_config1_oracle_reproduces_stored_placements(case):
    from oracle.binding import Oracle
    z, c = _load(case)
    o = Oracle(c)
    out, _, fc, fp = o.schedule()
    st = o.state()
    np.testing.assert_array_equal(out, z["out_node"])
    np.testing.assert_array_equal(fp, z["fail_pod"])
    np.testing.assert_array_equal(fc, z["fail_counts"])
    np.testing.assert_array_equal(st["num_pods"], z["num_pods"])
    f = c.facts
    assert f["n_nodes"] == 4                       # demo_1: master-1..3 + worker-1 (BASELINE.json says "3-node"; SURVEY 8d)
    assert int((out == -1).sum()) == f["unscheduled"]
    assert sum(v[0] for v in f["workloads"].values()) == f["n_pods"] == len(out)
    # every placed pod sits on a node that can hold it: aggregates never exceed allocatable
    assert (st["req_mcpu"] <= c.snap["alloc_mcpu"]).all() and (st["req_mem"] <= c.snap["alloc_mem"]).all()
    assert (st["num_pods"] <= c.snap["alloc_pods"]).all()


def test_config1_pinned_count_facts():
    """Pod counts per workload as the reference's expansion rules give them (pkg/utils/utils.go:132-247; replicas /
    completions default to 1), read off example/application/simple/*.yaml by hand: Deployment busybox-deploy replicas 4
    (pods owned by the generated ReplicaSet), ReplicaSet calico-kube-controllers 2, StatefulSet busybox-sts-new 8,
    Job pi (no completions -> 1), Pod single-pod 1, DaemonSet busybox-ds (one pod per eligible node).  The same kind of
    fact is what the reference's own test pins (pkg/simulator/core_test.go:364-591)."""
    _, c = _load("simple")
    wl = {k: v[0] for k, v in c.facts["workloads"].items()}
    assert wl["ReplicaSet/simple/busybox-deploy"] == 4
    assert wl["ReplicaSet/kube-system/calico-kube-controllers"] == 2
    assert wl["StatefulSet/simple/busybox-sts-new"] == 8
    assert wl["Job/default/pi"] == 1
    assert wl["Pod/simple/single-pod"] == 1
    assert 1 <= wl["DaemonSet/simple/busybox-ds"] <= c.facts["n_nodes"]
    # demo_1's own workloads: 3 masters x 4 static pods, coredns / kube-proxy DaemonSets, metrics-server
    assert sum(1 for k in wl if k.startswith("Pod/kube-system/")) == 12
    assert wl["DaemonSet/kube-system/kube-proxy-master"] == 3 and wl["DaemonSet/kube-system/kube-proxy-worker"] == 1
    app = c.facts["segments"][1]
    assert c.facts["segments"][0][0] == "cluster" and app[0] == "simple" and app[1] + app[2] == c.facts["n_pods"]


@pytest.mark.parametrize("case", CASES)
def test_config1_yaml_still_compiles_to_the_stored_columns(case):
    import make_config1
    arrays, facts = make_config1.derive(case)
    z, c = _load(case)
    assert facts == c.facts
    for k in z.files:
        np.testing.assert_array_equal(arrays[k], z[k], err_msg=k)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_config1_engine_matches_stored_placements(case):
    from simon_b200.engine import Engine
    z, c = _load(case)
    with Engine(c, device=0) as eng:
        out, _, fc, fp = eng.schedule()
        st = eng.state()
    np.testing.assert_array_equal(out, z["out_node"])
    np.testing.assert_array_equal(fp, z["fail_pod"])
    np.testing.assert_array_equal(fc, z["fail_counts"])
    np.testing.assert_array_equal(st["num_pods"], z["num_pods"])
    np.testing.assert_array_equal(st["req_mcpu"], z["req_mcpu"])
    np.testing.assert_array_equal(st["req_mem"], z["req_mem"])
