"""Node-drain batches on one GPU (simon_drain_run), checked against the CPU oracle on a sample; prints one JSON line.

Workloads: C3 (10,000 nodes, 120,500 pods) with every node drained alone, C3 with 256 random sets of 8 nodes, C2 (1,000 nodes) with
every node drained alone.  Per workload: wall time of one simon_drain_run call (host lists, fork, placement, downloads), the device
time of the placement kernels (simon_last_kernel_ms), the device time of the fork kernels and of the placement kernels from a
separate torch.profiler run, scenarios/s and re-placements/s, the totals, and `identical` against simon_oracle_drain on `--check`
sampled scenarios (tests/drain_oracle.c; its time is reported as the CPU reference rate of that sample)."""
import argparse
import json
import os
import random
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "open-simulator_b200"), ROOT, os.path.join(ROOT, "tests")):     # tests/: the drain oracle
    sys.path.insert(0, p)
import numpy as np

from simon_b200 import simulator, synth
from simon_b200.compiler import compile_cluster
from simon_b200.drain import survivor_order
from simon_b200.engine import Engine


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in q.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:       # noqa: BLE001 - reported, not hidden
        return dict(error=str(e))


def profiled_split(eng, orders):
    """Device time per kernel family of one drain call, from torch.profiler (CUDA activities)."""
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            eng.drain(orders)
            torch.cuda.synchronize()
        fork = place = other = 0.0
        for ev in prof.events():
            if ev.device_type.name != "CUDA":
                continue
            ms = ev.device_time_total / 1e3 if hasattr(ev, "device_time_total") else ev.cuda_time_total / 1e3
            if ev.name.startswith("simon_drain_"):
                fork += ms
            elif ev.name.startswith("simon_list_kernel"):
                place += ms
            else:
                other += ms
        return dict(fork_ms=round(fork, 3), place_kernel_ms=round(place, 3), other_device_ms=round(other, 3))
    except Exception as e:       # noqa: BLE001
        return dict(error=repr(e))


def run(name, c, sets, n_check, threads, seed):
    orders = [survivor_order(c, s) for s in sets]
    with Engine(c, device=0) as eng:
        eng.schedule()
        live = eng.results()
        eng.drain(orders[: min(len(orders), 64)])                      # warm-up: modules, pooled buffers
        t0 = time.perf_counter()
        res, off, pod, node, fc = eng.drain(orders)
        wall = time.perf_counter() - t0
        kernel_ms = eng.last_kernel_ms()
        t0 = time.perf_counter()
        res2, off2, pod2, node2, fc2 = eng.drain(orders)
        wall2 = time.perf_counter() - t0
        repeat_same = bool(np.array_equal(off, off2) and np.array_equal(node, node2) and np.array_equal(fc, fc2))
        split = profiled_split(eng, orders)
    n = len(orders)
    ev = sum(r["n_evicted"] for r in res)
    resched = sum(r["n_rescheduled"] for r in res)
    from drain_oracle import DrainOracle
    o = DrainOracle(c, threads=threads)
    t0 = time.perf_counter()
    olive = o.schedule()
    o_live_s = time.perf_counter() - t0
    sample = sorted(random.Random(seed).sample(range(n), min(n_check, n)))
    same = bool(np.array_equal(olive, live))
    t0 = time.perf_counter()
    for s in sample:
        counts, rpod, rnode, rfc, sums = o.drain(live, orders[s])
        a, b = int(off[s]), int(off[s + 1])
        same &= all(res[s][k] == v for k, v in counts.items()) and all(res[s][k] == v for k, v in sums.items())
        same &= bool(np.array_equal(pod[a:b], rpod) and np.array_equal(node[a:b], rnode) and np.array_equal(fc[a:b], rfc))
    o_ms = (time.perf_counter() - t0) * 1e3
    o.close()
    return dict(workload=name, nodes=c.n_nodes, pods=int(c.pods_dims["n_pods"]), scenarios=n,
                call_wall_ms=round(wall * 1e3, 2), call_wall_ms_repeat=round(wall2 * 1e3, 2), kernel_ms=round(kernel_ms, 3),
                profiled=split, scenarios_per_s=round(n / wall, 1), replacements_per_s=round(ev / wall, 1),
                evicted=ev, rescheduled=resched, unscheduled=sum(r["n_unscheduled"] for r in res),
                daemon=sum(r["n_daemon"] for r in res), bound=sum(r["n_bound"] for r in res),
                repeat_identical=repeat_same, identical=same, oracle_checked_scenarios=len(sample),
                oracle_sample=dict(threads=threads, live_schedule_s=round(o_live_s, 2), drain_ms=round(o_ms, 2),
                                   scenarios_per_s=round(len(sample) / (o_ms / 1e3), 2)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--check", type=int, default=16, help="scenarios per workload compared with the oracle")
    ap.add_argument("--threads", type=int, default=min(16, os.cpu_count() or 1), help="oracle host threads")
    ap.add_argument("--out", default="", help="also write the JSON line here")
    ap.add_argument("--small", action="store_true", help="small clusters (a rehearsal of the script, not a measurement)")
    a = ap.parse_args()
    out = dict(metric="node drains on one GPU", card=card())
    if a.small:
        c3 = synth.make_c3(n_nodes=300, n_workloads=60, replicas=10, n_apps=2, seed_no=7)
        c2 = synth.make_c2(n_nodes=100, n_workloads=10, replicas=30)
    else:
        c3 = synth.make_c3()
        c2 = synth.make_c2()
    rows = []
    p = simulator.plan(*c3)
    c = compile_cluster(p.nodes, p.pods, p.ctx)
    rows.append(run("C3 single-node drains", c, [[g] for g in range(c.n_nodes)], a.check, a.threads, 1))
    rng = random.Random(8)
    rows.append(run("C3 256 sets of 8 nodes", c, [rng.sample(range(c.n_nodes), 8) for _ in range(256)], a.check, a.threads, 2))
    p = simulator.plan(*c2)
    c = compile_cluster(p.nodes, p.pods, p.ctx)
    rows.append(run("C2 single-node drains", c, [[g] for g in range(c.n_nodes)], a.check, a.threads, 3))
    out["workloads"] = rows
    out["identical"] = all(r["identical"] for r in rows)
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
