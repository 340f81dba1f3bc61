"""bench.py --dump-outputs: the arrays of the last timed step, identical from run to run and equal to the oracle's placements."""
import argparse
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZE = ["--nodes", "300", "--workloads", "40", "--replicas", "5"]


def _bench_dump(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1", "--no-blocks",
           "--no-cpu-baseline", "--dump-outputs", str(out_dir)] + SIZE
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


@pytest.mark.gpu
def test_bench_dump_outputs_match_the_oracle(tmp_path):
    import bench
    from util import run_oracle
    a = _bench_dump(tmp_path / "a", steps=1)
    b = _bench_dump(tmp_path / "b", steps=3)
    assert sorted(a) == ["num_pods", "nz_mcpu", "nz_mem", "out_node", "req_eph", "req_mcpu", "req_mem"]
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    _, c, _ = bench.build_workload(argparse.Namespace(nodes=300, workloads=40, replicas=5), 3)
    (ref, _, _, _), st = run_oracle(c)
    np.testing.assert_array_equal(a["out_node"], ref)
    for k, v in st.items():
        np.testing.assert_array_equal(a[k], v, err_msg=k)
