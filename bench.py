#!/usr/bin/env python
"""bench.py — pod-placement decisions/s on the 10k-node synthetic cluster (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # the CUDA engine (through the C ABI)
  python bench.py --impl reference --steps K --warmup W    # the CPU restatement of the reference path

A "step" is one pass of the hot path over one batch: the whole ordered pod list of workload C3
(10,000 nodes x 100,000 pods, full predicate set) placed from the empty cluster state.
  value  : decisions/s, inputs resident in HBM, device-timed (CUDA events on the engine's stream), max over ranks
  e2e    : same metric through the C-ABI calls a caller makes with HOST buffers:
           simon_snapshot_upload + simon_pods_upload + simon_schedule(out_node -> host), wall clock
  N > 1  : a single scenario does not shard (each placement depends on the previous one) -> N independent
           replicas (distinct seeds), one per GPU, no data-path collective; scaling = weak.
Beside the headline the line carries the other BASELINE configurations as blocks:
  c2               1k nodes x 10k pods, Fit-only predicates (config 2)
  batch            concurrent what-if replicas of C3 on one GPU at the best residency (aggregate decisions/s)
  capacity_search  config 4: 2,000-node base, 5,000 pending pods, 8 specs x 32 node counts = 256 scenarios sharded over the
                   ranks, ONE all_reduce(MIN) inside the timed region
  move_scoring     config 5: 1,000,000 candidate moves on a 10k-node live snapshot (~300k running pods), moves partitioned
                   contiguously over the ranks, one all_reduce(MAX) + one all_gather of the per-rank top-k
--dump-outputs DIR writes what the last timed step left for its caller (rank 0): DIR/out_node.npy (the node of every pod of
the list, -1 = unschedulable) and the per-node totals of simon_state_download (DIR/req_mcpu.npy, ...), as float32 / float64.
The inputs are generated from fixed seeds, so two builds run with the same arguments can be compared array for array.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(ROOT, "open-simulator_b200"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "pod-placement decisions/sec on 10k-node synthetic cluster"
ALGO_BYTES_PER_NODE_DECISION = 180      # SURVEY.md section 8(d), C3 full predicate set
ALGO_BYTES_PER_NODE_DECISION_C2 = 80    # SURVEY.md section 8(d), C2 Fit + default scores
ALGO_BYTES_PER_MOVE = 280               # DESIGN.md section 3: move 8 + pod 8 + class 56 + target 96 + source 96 + verdict 8 + out 8


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def go_probe() -> str:
    """BASELINE.md section 3 / SURVEY 8c step 4: the reference itself can only be timed where a Go >= 1.18 toolchain exists."""
    exe = shutil.which("go")
    if not exe:
        return "go: not found on this box (the reference's Go path cannot be built or timed here)"
    try:
        return subprocess.run([exe, "version"], capture_output=True, text=True, timeout=20).stdout.strip()
    except Exception as e:       # noqa: BLE001
        return f"go: probe failed ({e})"


def build_workload(args, seed_no):
    from simon_b200 import simulator, synth
    from simon_b200.compiler import compile_cluster
    cluster, apps = synth.make_c3(n_nodes=args.nodes, n_workloads=args.workloads, replicas=args.replicas,
                                  n_apps=10, seed_no=seed_no)
    # host_compile_s: what Simulate() does on the host between receiving the objects and the first C-ABI call (workload expansion,
    # queue sorts, snapshot compiler).  Generating the synthetic objects themselves is the caller's input, not part of it.
    t0 = time.perf_counter()
    p = simulator.plan(cluster, apps)
    c = compile_cluster(p.nodes, p.pods, p.ctx)
    host_s = time.perf_counter() - t0
    build_workload.last_objects = (cluster, apps)
    return p, c, host_s


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None
        self.th = None

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.th = threading.Thread(target=self._read, daemon=True)
        self.th.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def host_cores() -> int:
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def cpu_threads(args, c=None, first_sched=0, cap=64) -> int:
    """Host threads for the CPU port: --cpu-threads, or the count that is fastest on a short sample of this workload
    (the per-node loops of one cycle are short, so more threads than that only add fork/join cost)."""
    ncpu = host_cores()
    if args.cpu_threads > 0:
        return max(1, min(64, args.cpu_threads))
    if c is None or ncpu <= 1:
        return 1
    from oracle.binding import Oracle
    best_t, best_v = 1, 0.0
    n = min(1500, c.pods_dims["n_pods"] - first_sched)
    for t in (1, 2, 4, 8, 16, 32, 64):
        if t > ncpu or t > cap:
            break
        o = Oracle(c, threads=t)
        o.schedule(0, first_sched)
        t0 = time.perf_counter()
        o.schedule(first_sched, n)
        v = n / (time.perf_counter() - t0)
        o.close()
        if v > best_v:
            best_t, best_v = t, v
    return best_t


def run_reference(args):
    """The reference's CPU path, restated (oracle/simon_oracle.c) — there is no Go toolchain to build the original.
    Like the GPU arm, a job at N "GPUs" is N independent replicas (distinct seeds): rank 0 runs them CONCURRENTLY on the box's
    host cores (one oracle per replica, each with the thread count that is fastest for it, capped so that the N replicas
    share the cores), the other ranks exit at once."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle.binding import Oracle
    n_rep = max(1, int(os.environ.get("WORLD_SIZE", str(args.gpus))))
    ncpu = host_cores()
    reps = []
    for r in range(n_rep):
        p, c, _ = build_workload(args, 3 + r)
        reps.append(c)
    c0 = reps[0]
    P = c0.pods_dims["n_pods"]
    first0 = int(np.argmax(c0.pods["pod_fixed_node"] == -1))
    per = cpu_threads(args, c0, first0, cap=max(1, ncpu // n_rep))
    sample = min(args.cpu_sample, min(int(c.pods_dims["n_pods"]) - int(np.argmax(c.pods["pod_fixed_node"] == -1)) for c in reps))
    oracles = [Oracle(c, threads=per) for c in reps]
    firsts = [int(np.argmax(c.pods["pod_fixed_node"] == -1)) for c in reps]
    times = []
    for step in range(args.warmup + args.steps):
        for o, f in zip(oracles, firsts):
            o.reset()
            o.schedule(0, f)                       # pre-bound pods: accounting only, not timed
        ths = [threading.Thread(target=o.schedule, args=(f, sample)) for o, f in zip(oracles, firsts)]
        t0 = time.perf_counter()
        for th in ths:
            th.start()
        for th in ths:
            th.join()
        dt = time.perf_counter() - t0
        if step >= args.warmup:
            times.append(dt)
    tot = sum(times)
    value = n_rep * sample * len(times) / tot
    cb = {"value": value, "unit": "decisions/s", "cores": per * n_rep, "kind": "port",
          "sample": f"first {sample} scheduled pods of each of {n_rep} replica pod list(s) ({P} pods) per step, {n_rep} concurrent "
                    f"oracle instance(s) x {per} host threads (oracle/simon_oracle.c; {ncpu} cores visible)",
          "go": go_probe()}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "decisions/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot / len(times), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int64+f64", "data": "synthetic",
            "config": workload_config(args, c0), "cpu_baseline": cb,
            "e2e": {"value": value, "unit": "decisions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir, eng):
    """Placements and per-node totals on the device after the last replay, converted exactly (node indices < 2^24 in
    float32, int64 totals < 2^53 in float64)."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"out_node": eng.results(), **eng.state()}
    for name, a in arrays.items():
        f = a.astype(np.float32 if a.dtype == np.int32 else np.float64)
        if not np.array_equal(f.astype(a.dtype), a):
            raise ValueError(f"{name} is not exact in {f.dtype}")
        np.save(os.path.join(out_dir, f"{name}.npy"), f)


def workload_config(args, c):
    return {"workload": f"C3: {args.nodes} nodes x {c.pods_dims['n_pods']} pods ({args.workloads} workloads x {args.replicas}), "
                        "full predicate set (taints, nodeSelector/affinity, inter-pod (anti)affinity, topology spread), seed 0x51514D4F4E03",
            "nodes": args.nodes, "pods": int(c.pods_dims["n_pods"]), "pod_classes": int(c.pods_dims["n_classes"]),
            "parallelism": "1 scenario per GPU (replicas)", "l2": "flushed between timed steps (256 MiB write)"}


# ---------------------------------------------------------------------------------------------------------------------
# blocks beside the headline
# ---------------------------------------------------------------------------------------------------------------------
def block_c2(args, local, flush, torch):
    """BASELINE config 2: 1k nodes x 10k pods, NodeResourcesFit-only predicates (the default score set stays active)."""
    from simon_b200 import simulator, synth
    from simon_b200.compiler import compile_cluster
    from simon_b200.engine import Engine
    from oracle.binding import Oracle
    cluster, apps = synth.make_c2(n_nodes=1000, n_workloads=100, replicas=100, seed_no=2)
    p = simulator.plan(cluster, apps)
    c = compile_cluster(p.nodes, p.pods, p.ctx)
    D = int((c.pods["pod_fixed_node"] == -1).sum())
    with Engine(c, device=local) as eng:
        for _ in range(3):
            eng.replay(1)
        ms = 0.0
        for _ in range(5):
            flush.zero_()
            torch.cuda.synchronize()
            ms += eng.replay(1)
        eng.reset()
        out = eng.schedule()[0]
    o = Oracle(c)
    t0 = time.perf_counter()
    ref = o.schedule()[0]
    cpu = D / (time.perf_counter() - t0)
    v = D * 5 / (ms * 1e-3)
    peak, _ = peaks()
    return {"workload": "C2: 1000 nodes x 10000 pods (100 deployments x 100), NodeResourcesFit-only predicates", "value": v, "unit": "decisions/s",
            "ms_per_step": ms / 5, "placements_identical_to_oracle": bool(np.array_equal(out, ref)), "cpu_port_1_thread": cpu,
            "roofline_frac": v * ALGO_BYTES_PER_NODE_DECISION_C2 * 1000 / 1e9 / peak}


def block_daemonsets(args, local, flush, torch):
    """The headline cluster with 5 DaemonSets on top (one pinned pod per node each): pods of the reference's
    MakeValidPodsByDaemonset (pkg/utils/utils.go:337-351).  One class per DaemonSet + a per-pod pin column; runs of pinned pods are
    placed in one pass.  Both device paths are timed and must agree pod for pod (the oracle comparison lives in the tests)."""
    from simon_b200 import simulator, synth
    from simon_b200.compiler import compile_cluster
    from simon_b200.engine import Engine
    cluster, apps = synth.make_c3(n_nodes=args.nodes, n_workloads=args.workloads, replicas=args.replicas, n_apps=10, seed_no=3)
    for k in range(5):
        lab = {"ds": f"agent-{k}"}
        cluster.DaemonSets.append({"apiVersion": "apps/v1", "kind": "DaemonSet", "metadata": {"name": f"agent-{k}", "namespace": "kube-system"},
                                   "spec": {"selector": {"matchLabels": lab}, "template": {"metadata": {"labels": lab}, "spec": {
                                       "tolerations": [{"operator": "Exists"}],
                                       "containers": [{"name": "c", "image": f"agent:{k}", "resources": {"requests": {"cpu": "50m", "memory": "64Mi"}},
                                                       "ports": [{"containerPort": 9100 + k, "hostPort": 9100 + k}]}]}}}})
    t0 = time.perf_counter()
    p = simulator.plan(cluster, apps)
    c = compile_cluster(p.nodes, p.pods, p.ctx)
    host_s = time.perf_counter() - t0
    n_ds = int((c.pods["pod_pin_node"] >= 0).sum())
    D = int((c.pods["pod_fixed_node"] == -1).sum())
    res = {}
    outs = {}
    for name, fast in (("run_at_once", True), ("general_path", False)):
        with Engine(c, device=local, pin_fast=fast) as eng:
            for _ in range(2):
                eng.replay(1)
            flush.zero_()
            torch.cuda.synchronize()
            ms = eng.replay(1)
            eng.reset()
            outs[name] = eng.schedule()[0]
        res[name] = {"ms": ms, "pods_per_s": D / (ms * 1e-3)}
    return {"workload": f"C3 cluster ({args.nodes} nodes) + 5 DaemonSets: {D} scheduled pods of which {n_ds} pinned DaemonSet pods",
            "classes": int(c.pods_dims["n_classes"]), "host_compile_s": host_s, **res,
            "paths_identical": bool(np.array_equal(outs["run_at_once"], outs["general_path"])),
            "placed": int((outs["run_at_once"] >= 0).sum()), "unschedulable": int((outs["run_at_once"] == -1).sum())}


def block_batch(args, c, D, P, placed, local, flush, torch):
    """Concurrent what-if replicas of the C3 workload on one GPU: one thread-block cluster each; report the best residency."""
    from simon_b200.engine import Engine
    best = None
    tried = []
    act = np.arange(int(c.n_nodes), dtype=np.uint32)
    for cs, tpb, nb in ((16, 320, 7), (8, 320, 15), (9, 320, 15), (9, 384, 15), (0, 0, 15), (0, 0, 7), (9, 384, 16)):      # (0, 0): the engine's own choice for a batch
        try:
            with Engine(c, device=local, cluster_ctas=cs, threads_per_cta=tpb) as eng:
                eng.run_scenarios([act] * nb)                                   # warm-up
                flush.zero_()
                torch.cuda.synchronize()
                res, _ = eng.run_scenarios([act] * nb)
                ms = eng.last_kernel_ms()
        except Exception as e:       # noqa: BLE001
            tried.append({"cluster_ctas": cs, "threads": tpb, "scenarios": nb, "error": str(e)[:120]})
            continue
        same = all(r["n_scheduled"] == placed - (P - D) or r["n_scheduled"] == placed for r in res)
        rec = {"cluster_ctas": cs, "threads": tpb, "scenarios": nb, "value": nb * D / (ms * 1e-3), "ms": ms, "identical_counts": bool(same)}
        tried.append(rec)
        if same and (best is None or rec["value"] > best["value"]):
            best = rec
    if best is None:
        return {"tried": tried}
    peak, _ = peaks()
    return dict(best, unit="decisions/s", tried=tried,
                roofline_frac_nominal=best["value"] * ALGO_BYTES_PER_NODE_DECISION * args.nodes / 1e9 / peak,
                note="simon_scenarios_run: independent replicas of the same workload placed concurrently on one GPU (the capacity-planning "
                     "batch shape); aggregate, not the headline value.  The snapshot of every scenario is resident in its cluster's shared "
                     "memory, so the nominal roofline fraction counts algorithmic bytes that never touch DRAM")


def block_capacity(args, rank, world, local, dist, torch):
    """BASELINE config 4: the add-node search (pkg/apply/apply.go:203-259) as 256 what-if scenarios sharded over the ranks."""
    from simon_b200 import capacity, synth
    from simon_b200.engine import Engine
    t0 = time.perf_counter()
    cluster, apps, specs = synth.make_c4(n_nodes=2000, n_workloads=50, replicas=100)
    ss = capacity.build_scenarios(cluster, apps, specs, list(range(1, 33)))
    t_build = time.perf_counter() - t0
    reduce_fn = capacity.torch_all_reduce_min(f"cuda:{local}") if world > 1 else None
    eng = Engine(ss.compiled, device=local)
    runner = capacity.gpu_runner(local, engine=eng)
    capacity.search(ss, runner, rank=rank, world=world, all_reduce_min=reduce_fn)       # warm-up: buffers + communicator
    times = []
    best = None
    for _ in range(3):
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        t1 = time.perf_counter()
        best, _local = capacity.search(ss, runner, rank=rank, world=world, all_reduce_min=reduce_fn)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t1)
    kernel_ms = eng.last_kernel_ms()
    eng.close()
    dt = min(times)
    tt = torch.tensor([dt, kernel_ms], dtype=torch.float64, device=f"cuda:{local}")
    if dist is not None:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dt, kernel_ms = float(tt[0].item()), float(tt[1].item())
    dec = capacity.decode_key(best)
    pods_per_scen = int((ss.compiled.pods["pod_fixed_node"] == -1).sum())
    # the same search through the native host side (simon_host_capacity_search: objects as JSON in -> per-scenario results + packed key
    # out; C++ superset expansion + compile + scenario lists + the launch), this rank's shard, wall clock of the whole call
    native = None
    try:
        from simon_b200 import native_host as _nh
        _nh.capacity_search_native(cluster, apps, specs, list(range(1, 33)), device=local, rank=rank, world=world)      # warm-up
        t1 = time.perf_counter()
        nat = _nh.capacity_search_native(cluster, apps, specs, list(range(1, 33)), device=local, rank=rank, world=world)
        nat_s = time.perf_counter() - t1
        key = nat["bestKey"]
        if reduce_fn is not None:
            key = reduce_fn(int(key))
        native = {"call_s_incl_request_encoding": nat_s, "library_timing": nat["timing"], "same_answer": bool(int(key) == int(best))}
    except Exception as e:       # noqa: BLE001
        native = {"error": f"{type(e).__name__}: {e}"[:200]}
    return {"workload": "C4: 2000-node base ~85 % full, 5000 pending pods, 8 node specs x k = 1..32 -> 256 scenarios",
            "scenarios": len(ss.scenarios), "n_gpus": world, "search_s": dt, "kernel_ms_max_rank": kernel_ms, "host_build_s": t_build,
            "best": dec, "best_spec": (ss.scenarios[dec["scenario"]].spec if dec else None),
            "decisions_per_s": len(ss.scenarios) * pods_per_scen / dt, "scheduled_pods_per_scenario": pods_per_scen,
            "native_host": native,
            "collective": "one all_reduce(MIN) of an int64 key (k << 32 | scenario) over NCCL, inside search_s" if world > 1 else "none (single process)",
            "timing": "best of 3 searches, wall clock per rank (includes the scenario-list uploads, the launch, the result download "
                      "and the collective), max over ranks"}


def block_moves(args, rank, world, local, dist, torch):
    """BASELINE config 5: 1,000,000 candidate moves scored on a 10k-node live snapshot."""
    from simon_b200 import moves as M, simulator, synth
    from simon_b200.compiler import compile_cluster
    from simon_b200.engine import Engine
    cluster, apps = synth.make_c3(n_nodes=args.nodes, n_workloads=max(10, args.nodes // 10), replicas=10, n_apps=10, seed_no=3)
    p = simulator.plan(cluster, apps)
    c = compile_cluster(p.nodes, p.pods, p.ctx)
    live = synth.make_c5(c, args.running)
    n_moves = args.moves
    with Engine(live, device=local) as eng:
        out = eng.schedule()[0]                                     # import of the running pods (accounting only)
        mv = M.sample_moves(len(out), live.n_nodes, n_moves, seed=11, placement=out)
        lo, hi = M.shard_bounds(n_moves, rank, world)
        eng.moves_upload(mv[lo:hi], lo)
        eng.moves_replay(3)
        steps = 20
        ms = eng.moves_replay(steps) / steps                        # device-resident: pack + score kernels, CUDA events
        arm, agk = M.torch_collectives(f"cuda:{local}") if world > 1 else (None, None)
        runner = M.gpu_runner(eng)
        M.search(mv, runner, k=16, rank=rank, world=world, all_reduce_max=arm, all_gather_topk=agk)     # warm-up
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        t0 = time.perf_counter()
        best, topk, res = M.search(mv, runner, k=16, rank=rank, world=world, all_reduce_max=arm, all_gather_topk=agk)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        check = None
        if rank == 0 and not args.no_cpu_baseline:
            from oracle.binding import Oracle
            o = Oracle(live)
            o.schedule()
            nchk = min(200000, hi - lo)
            eng.moves_upload(mv[lo:lo + nchk], lo)
            r = eng.moves_run(k=0, want_arrays=True)
            t1 = time.perf_counter()
            g, cd = o.moves_score(mv[lo:lo + nchk], out)
            cpu = nchk / (time.perf_counter() - t1)
            check = {"moves_compared_with_oracle": nchk, "identical": bool(np.array_equal(g, r["gain"]) and np.array_equal(cd, r["code"])),
                     "cpu_port_moves_per_s_1_thread": cpu}
    tt = torch.tensor([ms, dt], dtype=torch.float64, device=f"cuda:{local}")
    if dist is not None:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms, dt = float(tt[0].item()), float(tt[1].item())
    peak, _ = peaks()
    v = n_moves / (ms * 1e-3)
    return {"workload": f"C5: {live.n_nodes} nodes, {live.pods_dims['n_pods']} running pods, {n_moves} candidate moves sampled uniformly",
            "n_gpus": world, "value": v, "unit": "moves/s", "us_per_pass_max_rank": ms * 1e3,
            "roofline": {"bound": "hbm", "achieved": v / world * ALGO_BYTES_PER_MOVE / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": v / world * ALGO_BYTES_PER_MOVE / 1e9 / peak,
                         "note": f"algorithmic bytes = {ALGO_BYTES_PER_MOVE} B/move (move 8, pod 8, class 56, target + source node records 96 each, "
                                 "static verdict 8, outputs 8); per GPU; the node table (~1 MB) is L2-resident, so DRAM traffic is the move list "
                                 "and the outputs"},
            "e2e": {"value": n_moves / dt, "unit": "moves/s", "h2d_bytes": int(8 * (hi - lo)), "path": "simon_moves_upload + simon_moves_run(top-16) "
                    "+ all_reduce(MAX) + all_gather(top-k), wall clock, max over ranks"},
            "best": best, "topk": topk[:4], "check": check}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="gpu", choices=["gpu", "reference"])
    ap.add_argument("--nodes", type=int, default=10000)
    ap.add_argument("--workloads", type=int, default=1000)
    ap.add_argument("--replicas", type=int, default=100)
    ap.add_argument("--running", type=int, default=300000, help="running pods of the C5 live snapshot")
    ap.add_argument("--moves", type=int, default=1000000, help="candidate moves of C5")
    ap.add_argument("--cpu-sample", type=int, default=30000, help="decisions per step of the --impl reference arm")
    ap.add_argument("--cluster-ctas", type=int, default=0)
    ap.add_argument("--threads", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-threads", type=int, default=0, help="host threads of the CPU port (0 = fastest count on this box, capped at 64)")
    ap.add_argument("--no-batch", action="store_true")
    ap.add_argument("--no-blocks", action="store_true", help="headline only: skip the c2 / batch / capacity_search / move_scoring blocks")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "gpu" else args.warmup

    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl gpu needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from simon_b200.engine import Engine
    p, c, host_s = build_workload(args, 3 + rank)          # replicas: distinct seeds per rank
    P = int(c.pods_dims["n_pods"])
    D = int((c.pods["pod_fixed_node"] == -1).sum())        # decisions = pods that go through filter+score (pre-bound pods excluded)
    eng = Engine(c, device=local, cluster_ctas=args.cluster_ctas, threads_per_cta=args.threads)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{local}")

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        eng.replay(1)
    sampler = ClockSampler(local)
    launches0 = eng.launch_count()
    barrier()
    sampler.start()
    t_wall0 = time.perf_counter()
    ms_total = 0.0
    for _ in range(args.steps):
        flush.zero_()
        torch.cuda.synchronize()
        ms_total += eng.replay(1)
    barrier()
    wall = time.perf_counter() - t_wall0
    clocks = sampler.stop()
    launches = eng.launch_count() - launches0
    t = torch.tensor([ms_total], dtype=torch.float64, device=f"cuda:{local}")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * D * args.steps / (ms_max * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng)

    # ---- e2e: host buffers -> C ABI -> host results ----
    import ctypes as C
    from simon_b200.engine import lib
    L = lib()
    h2d = sum(a.nbytes for a in eng._keep)
    out_node = np.empty(P, np.int32)
    n_fail = C.c_uint32(0)
    e2e_times = []
    for step in range(2 + args.steps):
        barrier()
        t0 = time.perf_counter()
        assert L.simon_snapshot_upload(eng.h, C.byref(eng.snap)) == 0
        assert L.simon_pods_upload(eng.h, C.byref(eng.pods)) == 0
        assert L.simon_schedule(eng.h, 0, P, out_node.ctypes.data, None, None, None, 0, C.byref(n_fail)) == 0
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if step >= 2:
            e2e_times.append(dt)
    # ---- the public API itself: Simulate(objects) -> SimulateResult, wall clock (plan + compile + engine creation + uploads +
    #      placement + result objects); one untimed call first (lazy imports), on fresh copies of the objects each time ----
    api_s = None
    api_native = None
    if not args.no_blocks and rank == 0:
        from simon_b200 import simulator as _sim
        from simon_b200.objects import deep_copy as _dc
        cl0, ap0 = build_workload.last_objects
        api_times = []
        for rep in range(3):
            cl = type(cl0)(**{k: _dc(v) for k, v in vars(cl0).items()})
            ap = [type(a)(Name=a.Name, Resource=type(a.Resource)(**{k: _dc(v) for k, v in vars(a.Resource).items()})) for a in ap0]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res_api = _sim.Simulate(cl, ap, _sim.WithDevice(local))
            dt = time.perf_counter() - t0
            if rep:
                api_times.append(dt)
        api_s = min(api_times)
        api_parts = {k: round(v, 4) for k, v in getattr(_sim.Simulate, "last_timing", {}).items()}
        api_placed = sum(len(ns.Pods) for ns in res_api.NodeStatus)
        # ---- the same call through the NATIVE host side (simon_host_simulate: JSON objects in -> placements + failure messages out,
        #      C++ expansion / queue sorts / snapshot compiler / result; what the Go shim calls).  The request is marshalled once,
        #      outside the timed region (the Go caller marshals its typed objects with encoding/json; Python's json.dumps of the
        #      same objects is reported as request_encode_s for scale) ----
        try:
            from simon_b200 import native_host as _nh
            t0 = time.perf_counter()
            req = _nh.request_json(cl0, ap0)
            enc_s = time.perf_counter() - t0
            nat_times = []
            for rep in range(3):
                torch.cuda.synchronize()
                nat = _nh.simulate_native(None, None, device=local, req=req)
                if rep:
                    nat_times.append(_nh.simulate_native.last_call_s)
            nat_s = min(nat_times)
            nat_placed = sum(len(x) for x in nat["nodeStatus"])
            # identical outcome: every pod on the same node as through the Python mirror, same failure messages
            py_node = {}
            for ns in res_api.NodeStatus:
                for r in ns.Pods:
                    py_node[r.key()] = (ns.Node.get("metadata") or {}).get("name")
            tl = nat["templates"]
            same = nat_placed == api_placed
            for ti, name, o, nd in zip(nat["podTemplate"], nat["podName"], nat["podOrdinal"], nat["podNode"]):
                tt = tl[ti]
                k = (tt["kind"], tt["namespace"], name if tt["kind"] == "Pod" else tt["workload"], o)
                if (nat["nodes"][nd] if nd >= 0 else None) != py_node.get(k):
                    same = False
                    break
            same = same and [u["reason"] for u in nat["unscheduledPods"]] == [u.Reason for u in res_api.UnscheduledPods]
            api_native = {"value": D / nat_s, "unit": "decisions/s", "simulate_s": nat_s, "request_bytes": len(req), "request_encode_s": enc_s,
                          "result_decode_s": _nh.simulate_native.last_decode_s,
                          "last_call_parts": nat["timing"], "identical_to_python_simulate": bool(same),
                          "path": "simon_host_simulate(request JSON) -> result JSON, wall clock of the C-ABI call on rank 0 (what a cgo caller "
                                  "waits for; decoding the result is the caller's: result_decode_s is Python's json.loads), best of 2 after one "
                                  "untimed call: JSON parse + workload expansion + Go 1.18 queue sorts + snapshot "
                                  "compiler (C++) + engine creation + uploads + placement + per-node lists and FitError messages"}
        except Exception as e:       # noqa: BLE001
            api_native = {"error": f"{type(e).__name__}: {e}"[:300]}
    te = torch.tensor([sum(e2e_times)], dtype=torch.float64, device=f"cuda:{local}")
    if dist is not None:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * D * len(e2e_times) / float(te.item())
    placed = int((out_node >= 0).sum())
    stats = eng.stats()
    eng.close()

    # ---- the other BASELINE configurations ----
    blocks = {}
    if not args.no_blocks:
        def guarded(name, fn, *a):
            try:
                blocks[name] = fn(*a)
            except Exception as e:       # noqa: BLE001  (a block must never take the headline down with it)
                blocks[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
        if world == 1:
            guarded("c2", block_c2, args, local, flush, torch)
            guarded("daemonsets", block_daemonsets, args, local, flush, torch)
            if not args.no_batch:
                guarded("batch", block_batch, args, c, D, P, placed, local, flush, torch)
        guarded("capacity_search", block_capacity, args, rank, world, local, dist, torch)
        guarded("move_scoring", block_moves, args, rank, world, local, dist, torch)

    if rank == 0:
        peak, peak_src = peaks()
        per_gpu_dps = D * args.steps / (ms_total * 1e-3)
        achieved = per_gpu_dps * ALGO_BYTES_PER_NODE_DECISION * args.nodes / 1e9
        traffic, traffic_src = None, None
        for name in ("r02_ncu_full_summary.json", "r01_ncu_full_summary.json"):
            try:
                prof = json.load(open(os.path.join(ROOT, "profiles", name)))
                traffic = prof["dram_bytes_per_launch"]      # dram__bytes_read.sum + dram__bytes_write.sum of one --set full capture
                traffic_src = f"profiles/{name} (one ncu --set full capture of the same launch shape; not measured in this run)"
                break
            except Exception:
                continue
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": ALGO_BYTES_PER_NODE_DECISION * args.nodes * D,
                "note": f"algorithmic bytes = {ALGO_BYTES_PER_NODE_DECISION} B/node-decision x {args.nodes} nodes x {D} decisions per launch; "
                        "the snapshot is cluster-resident in shared memory, so DRAM traffic << algorithmic bytes and the kernel is bound by the "
                        "latency of its per-decision reductions, not by HBM"}
        cb = None
        if not args.no_cpu_baseline and world == 1:          # the CPU baseline is reported at N = 1 only
            from oracle.binding import Oracle
            first_sched = int(np.argmax(c.pods["pod_fixed_node"] == -1))
            o = Oracle(c, threads=cpu_threads(args, c, first_sched))
            o.schedule(0, first_sched)
            t0 = time.perf_counter()
            ref_nodes, _, _, _ = o.schedule(first_sched, P - first_sched)        # EVERY decision of the timed pod list
            dt = time.perf_counter() - t0
            agree = bool(np.array_equal(ref_nodes, out_node[first_sched:]))
            n_dec = int((c.pods["pod_fixed_node"][first_sched:] == -1).sum())
            cb = {"value": n_dec / dt, "unit": "decisions/s", "cores": o.threads, "kind": "port",
                  "sample": f"all {n_dec} decisions of the same pod list (oracle/simon_oracle.c, per-node loops shared "
                            f"between {o.threads} host threads, the fastest count on this box; {host_cores()} cores visible)",
                  "placements_identical": agree, "decisions_compared": n_dec, "go": go_probe()}
        line = {"metric": METRIC, "value": value, "unit": "decisions/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "int64+f64", "data": "synthetic", "config": workload_config(args, c),
                "roofline": roof, "cpu_baseline": cb,
                "e2e": {"value": e2e_value, "unit": "decisions/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(4 * P + 8),
                        "path": "simon_snapshot_upload + simon_pods_upload + simon_schedule(host out_node), wall clock; the host-side snapshot "
                                "compile (host_compile_s) happens once per cluster and is reported separately"},
                "e2e_api": {"value": (D / api_s) if api_s else None, "unit": "decisions/s", "simulate_s": api_s, "last_call_parts": api_parts if api_s else None,
                            "estimate_from_parts": D / (host_s + float(te.item()) / len(e2e_times)),
                            "path": "simulator.Simulate(cluster objects, app objects) -> SimulateResult, wall clock of the call on rank 0, best of 2 "
                                    "after one untimed call: workload expansion + queue sorts + snapshot compiler (Python, host_compile_s) + "
                                    "engine creation + uploads + placement + per-node result lists; estimate_from_parts = host_compile_s + one e2e pass"},
                "e2e_api_native": api_native if api_s else None,
                "gpu_launches": int(launches), "clocks": clocks, "decisions_per_step": D, "prebound_pods_per_step": P - D, "placed": placed,
                "unschedulable": int((out_node == -1).sum()), "wall_s_timed_region": wall, "host_compile_s": host_s,
                "kernel_stats": {k: stats[k] for k in ("class_switches", "summary_rebuilds", "redone", "single_flip_fast", "merged_decisions", "merged_redone")}}
        line.update(blocks)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
