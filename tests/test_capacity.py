"""Capacity-planning scenario search (C4): sharding + the single MIN all-reduce, on CPU with gloo (world_size 2),
and GPU parity of every scenario against the oracle."""
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _small_set():
    from simon_b200 import capacity, synth
    cluster, apps, specs = synth.make_c4(n_nodes=60, n_workloads=6, replicas=12, seed_no=4)
    return capacity.build_scenarios(cluster, apps, specs[:3], ks=[1, 2, 4, 8])


def oracle_runner(ss, shard):
    """Test-side runner: the CPU oracle restricted to each scenario's active node set."""
    from oracle.binding import Oracle
    o = Oracle(ss.compiled)
    alloc_mcpu = ss.compiled.snap["alloc_mcpu"]
    alloc_mem = ss.compiled.snap["alloc_mem"]
    out = []
    for sc in shard:
        o.reset()
        o.set_active(sc.nodes)
        nodes, _, _, _ = o.schedule()
        st = o.state()
        act = sc.nodes.astype(np.int64)
        out.append(dict(n_unscheduled=int((nodes == -1).sum()), n_scheduled=int(((nodes >= 0) & (ss.compiled.pods["pod_fixed_node"] == -1)).sum()),
                        req_mcpu=int(st["req_mcpu"][act].sum()), alloc_mcpu=int(alloc_mcpu[act].sum()),
                        req_mem=int(st["req_mem"][act].sum()), alloc_mem=int(alloc_mem[act].sum()), nodes=nodes))
    o.close()
    return out


def test_scenarios_single_process_monotone():
    from simon_b200 import capacity
    ss = _small_set()
    best, res = capacity.search(ss, oracle_runner)
    assert len(res) == len(ss.scenarios)
    # more nodes of the same spec never leave more pods unscheduled than fewer
    for spec in range(3):
        un = [res[sc.sid]["n_unscheduled"] for sc in ss.scenarios if sc.spec == spec]
        assert all(a >= b for a, b in zip(un, un[1:])), un
    keys = [capacity.scenario_key(sc, res[sc.sid], 100, 100) for sc in ss.scenarios]
    assert best == min(keys)


def _worker(rank, world, port, q):
    sys.path.insert(0, os.path.join(ROOT, "open-simulator_b200"))
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch.distributed as dist
    from simon_b200 import capacity
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    ss = _small_set()
    best, res = capacity.search(ss, oracle_runner, rank=rank, world=world, all_reduce_min=capacity.torch_all_reduce_min("cpu"))
    q.put((rank, best, sorted(res.keys())))
    dist.destroy_process_group()


def test_scenarios_sharded_gloo_world2():
    import torch.multiprocessing as mp
    from simon_b200 import capacity
    ss = _small_set()
    ref_best, _ = capacity.search(ss, oracle_runner)
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    sids = set()
    for rank, best, keys in got:
        assert best == ref_best                      # every rank holds the global minimum after the all-reduce
        assert all(k % 2 == rank for k in keys)      # round-robin sharding, no overlap
        sids.update(keys)
    assert sids == set(range(len(ss.scenarios)))


@pytest.mark.gpu
def test_scenarios_gpu_match_oracle():
    from simon_b200 import capacity
    from simon_b200.engine import Engine
    ss = _small_set()
    ref = oracle_runner(ss, ss.scenarios)
    with Engine(ss.compiled, device=0) as eng:
        out, nodes = eng.run_scenarios([sc.nodes for sc in ss.scenarios], want_nodes=True)
    for sc, r, g in zip(ss.scenarios, ref, out):
        np.testing.assert_array_equal(nodes[sc.sid], r["nodes"], err_msg=f"scenario {sc.sid}")
        for k in ("n_unscheduled", "req_mcpu", "alloc_mcpu", "req_mem", "alloc_mem"):
            assert g[k] == r[k], (sc.sid, k, g[k], r[k])
    best_gpu, _ = capacity.search(ss, capacity.gpu_runner(0))
    best_ref, _ = capacity.search(ss, oracle_runner)
    assert best_gpu == best_ref


def _oracle_factory(ss):
    return oracle_runner


def test_auto_add_nodes_sweep_and_bisect_agree():
    """The automatic replacement of the interactive add-node loop (pkg/apply/apply.go:203-259): the sweep over k and the
    bisection find the same minimal node count, and that count is tight (k-1 leaves pods unscheduled or breaks a cap)."""
    from simon_b200 import apply as A, capacity, synth
    cluster, apps, specs = synth.make_c4(n_nodes=12, n_workloads=8, replicas=15, seed_no=4)
    sweep = A.auto_add_nodes(cluster, apps, specs[1], _oracle_factory, kmax=24, method="sweep")
    bis = A.auto_add_nodes(cluster, apps, specs[1], _oracle_factory, kmax=24, method="bisect")
    assert sweep.new_node_num == bis.new_node_num and sweep.new_node_num > 0
    assert sweep.unscheduled_without_new_nodes > 0
    assert bis.scenarios_evaluated < sweep.scenarios_evaluated and bis.rounds <= 7
    k = sweep.new_node_num
    r1, r0 = sweep.per_k[k], sweep.per_k[k - 1]
    assert r1["n_unscheduled"] == 0 and capacity.occupancy_ok(r1)
    assert r0["n_unscheduled"] > 0 or not capacity.occupancy_ok(r0)
    # monotone: every k beyond the minimum is feasible as well
    assert all(sweep.per_k[q]["n_unscheduled"] == 0 for q in range(k, 25))


def test_apply_config_of_the_reference_example(tmp_path):
    """example/simon-config.yaml with `customConfig: example/cluster/demo_1` (the shipped file points at a developer's
    kubeConfig, SURVEY 8d C1) and the non-chart, non-open-local apps: the 4-node demo cluster cannot hold them, the search
    reports how many copies of example/newnode/demo_1 are needed.  The example inputs are stored in tests/golden/example/."""
    import yaml
    from simon_b200 import apply as A
    cfg = {"apiVersion": "simon/v1alpha1", "kind": "Config", "metadata": {"name": "simon-config"},
           "spec": {"cluster": {"customConfig": "example/cluster/demo_1"},
                    "appList": [{"name": "simple", "path": "example/application/simple"},
                                {"name": "complicated", "path": "example/application/complicate"},
                                {"name": "more_pods", "path": "example/application/more_pods"}],
                    "newNode": "example/newnode/demo_1"}}
    path = tmp_path / "simon-config.yaml"
    path.write_text(yaml.safe_dump(cfg))
    base = os.path.join(ROOT, "tests", "golden")
    cluster, apps, new_node = A.load_config(str(path), base_dir=base)
    assert len(cluster.Nodes) == 4 and len(apps) == 3 and new_node["metadata"]["name"] == "node-1"
    res = A.auto_add_nodes(cluster, apps, new_node, _oracle_factory, kmax=32, method="bisect")
    assert res.unscheduled_without_new_nodes > 0
    assert res.new_node_num > 0
    sweep = A.auto_add_nodes(cluster, apps, new_node, _oracle_factory, kmax=res.new_node_num + 2, method="sweep")
    assert sweep.new_node_num == res.new_node_num
    # the shipped config itself is refused for what it is (kubeConfig of a developer machine / Helm chart), not ignored
    with pytest.raises(NotImplementedError):
        A.load_config(os.path.join(base, "example", "simon-config.yaml"), base_dir=base)


@pytest.mark.gpu
def test_auto_add_nodes_gpu_matches_oracle():
    from simon_b200 import apply as A, capacity, synth
    from simon_b200.engine import Engine
    cluster, apps, specs = synth.make_c4(n_nodes=12, n_workloads=8, replicas=15, seed_no=4)
    want = A.auto_add_nodes(cluster, apps, specs[1], _oracle_factory, kmax=16, method="sweep")
    engines = []

    def factory(ss):
        e = Engine(ss.compiled, device=0)
        engines.append(e)
        return capacity.gpu_runner(0, engine=e)

    got = A.auto_add_nodes(cluster, apps, specs[1], factory, kmax=16, method="sweep")
    got_b = A.auto_add_nodes(cluster, apps, specs[1], factory, kmax=16, method="bisect")
    for e in engines:
        e.close()
    assert got.new_node_num == want.new_node_num == got_b.new_node_num
    assert got.per_k == want.per_k
