"""bench.py --dump-outputs: what the timed path computed in its last step, as float64 .npy files, so that two builds of
the project can be compared output for output on identical inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sample_rows_are_fixed_and_in_range():
    import bench
    for n in (100, 70_000, 200_000, 100_000_000):
        rows = bench.dump_sample_rows(n)
        assert rows.size == min(n, bench.DUMP_BLOCKS * bench.DUMP_BLOCK_ROWS)
        assert rows[0] >= 0 and rows[-1] < n and np.all(np.diff(rows) > 0)
        assert np.array_equal(rows, bench.dump_sample_rows(n))


def test_reference_arm_refuses_dump_outputs(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path / "out")],
                         cwd=ROOT, capture_output=True, text=True)
    assert out.returncode != 0 and "--dump-outputs" in out.stderr
    assert not (tmp_path / "out").exists()


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def bench_data(workload, n):
    """The points bench.py generates for `workload` at --points n, downloaded from the device."""
    import bench
    from ml_b200 import cabi
    _, _, d, k = bench.WORKLOADS[workload]
    ctx = cabi.Context(1)
    data = cabi.Data.generate_gmm(ctx, n, d, min(k, 64), seed=bench.DATA_SEED)
    x = data.download(0, n)
    data.close()
    ctx.close()
    return x, k


@pytest.mark.gpu
@pytest.mark.parametrize("workload,steps,extra", [("c3", 1, []), ("c5", 3, ["--no-e2e"])])
def test_dump_outputs_repeat_and_hold_the_last_timed_step(tmp_path, workload, steps, extra):
    """Two runs with the same arguments write identical files.  The trace has one entry per timed step and ends at the
    line's last_scalar.  The parameters and the sampled per-point outputs are those of the CPU oracle run from the same
    start (data points 0..K-1) for warmup + steps iterations on the same generated points.  The c3 case times a single
    step with the e2e fit included."""
    n, warmup = 100_000, 1

    def run(tag):
        out = tmp_path / tag
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--points", str(n), "--steps", str(steps),
               "--warmup", str(warmup), "--no-cpu", "--no-clocks", "--dump-outputs", str(out), *extra]
        res = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-2000:]
        line = json.loads(res.stdout.strip().splitlines()[-1])
        return line, {name[:-4]: np.load(out / name) for name in os.listdir(out)}

    line, a = run("a")
    _, b = run("b")
    for name in a:
        assert np.array_equal(a[name], b[name]), name
    trace = "log_likelihood" if workload == "c3" else "inertia"
    per_point = {"responsibilities", "labels"} if workload == "c3" else {"labels"}
    params = {"means", "covariances", "mixing_probabilities"} if workload == "c3" else {"centroids"}
    assert set(a) == {trace, "sample_rows"} | per_point | params
    assert line["steps"] == steps and a[trace].shape == (steps,) and a[trace][-1] == line["last_scalar"]
    assert all(x.dtype == np.float64 for x in a.values()) and sum(x.nbytes for x in a.values()) <= 64 << 20
    rows = a["sample_rows"].astype(np.int64)
    assert rows.size == 65536 and np.all(np.diff(rows) > 0) and rows[-1] < n
    assert all(a[name].shape[0] == rows.size for name in per_point)

    import oracle
    x, k = bench_data(workload, n)
    init = np.ascontiguousarray(x[:k].T)
    if workload == "c3":
        ref = oracle.em_fit(x, k, means_init=oracle.EXPLICIT, explicit_means=init, maximum_steps=warmup + steps,
                            absolute_tolerance=0.0, relative_tolerance=0.0)
        assert ref.iterations == warmup + steps
        assert abs(a[trace][-1] - ref.log_likelihood) <= 1e-9 * abs(ref.log_likelihood)
        assert rel(a["means"], ref.means) <= 1e-9 and rel(a["covariances"], ref.covariances) <= 1e-9
        assert rel(a["mixing_probabilities"], ref.mixing_probabilities) <= 1e-9
        resp = ref.responsibilities[rows]
        assert np.max(np.abs(a["responsibilities"] - resp)) <= 1e-9
        # labels are the most responsible components; rows whose two largest responsibilities tie to rounding may differ
        top2 = np.sort(resp, axis=1)[:, -2:]
        differ = a["labels"] != resp.argmax(axis=1)
        assert np.all(top2[differ, 1] - top2[differ, 0] <= 1e-9)
    else:
        ref = oracle.kmeans_fit(x, k, init=oracle.EXPLICIT, explicit_means=init, maximum_steps=warmup + steps, absolute_tolerance=0.0)
        assert ref.iterations == warmup + steps and not ref.converged
        assert abs(a[trace][-1] - ref.inertia) <= 1e-9 * ref.inertia
        assert rel(a["centroids"], ref.centroids) <= 1e-9
        assert np.array_equal(a["labels"], ref.labels[rows])
