"""K-means distances and inertia on the device: mlb_km_transform, mlb_km_transform_range, mlb_km_score,
mlb_km_score_fitted, ml::Clustering::KMeans::transform / inertia(points) / final_inertia(), and the cppyml
KMeans.transform / KMeans.score.

Every K-means configuration of the kernel matrix (tests/test_gpu_kernel_matrix.py, KM_CASES: the filter path at every DP,
the exact path D > 64, several centroid blocks, chunk 128 and 2048, ragged N) plus K = 1 on both paths, each asserting
the configuration it ran.  km_transform_kernel has one instance; every case runs it.

Bars: a squared distance from transform is bitwise predict's at the predicted label, and within 4 D u (relative) of the
long-double direct difference everywhere; the Euclidean output is sqrt of the squared one, bitwise.  score_fitted is
bitwise the next assign's inertia; score's inertia is within 1e-13 of the exact sum of predict's squared distances.
"""
import math

import numpy as np
import pytest

from tests.test_gpu_kernel_matrix import KM_CASES, N_A, N_B, _km_id, km_problem

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
CASES = KM_CASES + [
    (5, 1, N_A, 128, {}, (8, 32, 32, 1, 4, 0, 0, 128)),
    (5, 1, N_B, 2048, {}, (8, 32, 32, 1, 4, 0, 0, 2048)),
    (100, 1, N_A, 128, {}, (128, 32, 32, 1, 4, 1, 1, 128)),
    (100, 1, N_B, 2048, {}, (128, 32, 32, 1, 4, 1, 1, 2048)),
]
SAMPLE = 400   # rows per case checked against the long-double reference (every row is checked against predict)


@pytest.fixture(scope="module")
def ctx():
    from ml_b200 import cabi
    assert cabi.device_count() >= 1, "no CUDA device: the product has no CPU fallback"
    c = cabi.Context(1)
    yield c
    c.close()


def ref_sq(x, centroids):
    """(m, K) squared distances by direct differences in long double."""
    x = np.asarray(x, dtype=np.longdouble)
    c = np.asarray(centroids, dtype=np.longdouble)
    out = np.zeros((x.shape[0], c.shape[1]), dtype=np.longdouble)
    for l in range(x.shape[1]):
        t = x[:, l, None] - c[None, l, :]
        out += t * t
    return out


def sample_rows(m, seed=0):
    rng = np.random.default_rng(seed)
    rows = np.concatenate([[0, m - 1], rng.choice(m, size=min(m, SAMPLE), replace=False)])
    return np.unique(rows)


def check_accuracy(got_sq, x, centroids, rows):
    want = ref_sq(x[rows], centroids)
    d = x.shape[1]
    err = np.abs(got_sq[rows].astype(np.longdouble) - want)
    assert np.all(err <= 4 * d * U * want), float(np.max(err / np.maximum(want, 1e-300)))
    return float(np.max(err / np.maximum(want, 1e-300)))


def check_against_predict(sq, labels, dist):
    m = len(labels)
    assert np.array_equal(sq[np.arange(m), labels], dist)          # bitwise at the predicted label
    assert np.array_equal(sq.min(axis=1), dist)
    assert np.array_equal(np.argmin(sq, axis=1).astype(np.uint32), labels)   # first minimum = lowest index


@pytest.mark.parametrize("case", CASES, ids=_km_id)
def test_transform_and_score_every_configuration(ctx, monkeypatch, case):
    from ml_b200 import cabi
    d, k, n, chunk, env, expected = case
    x, q, c0, _ = km_problem(d, k, n)
    monkeypatch.setenv("MLB200_CHUNK", str(chunk))
    for key, val in env.items():
        monkeypatch.setenv(key, val)
    dev = cabi.Data.upload(ctx, x)
    km = cabi.Km(dev, k)
    try:
        cfg = km.kernel_config()
        assert tuple(cfg[f] for f in cabi.KM_CONFIG_FIELDS) == expected, cfg
        km.set_centroids(c0)
        # new points
        labels, dist = km.predict(q)
        sq = km.transform(q, squared=True)
        assert sq.shape == (q.shape[0], k) and sq.dtype == np.float64
        check_against_predict(sq, labels, dist)
        assert np.array_equal(km.transform(q), np.sqrt(sq))
        err_q = check_accuracy(sq, q, c0, sample_rows(q.shape[0]))
        sqd, inertia = km.score(q)
        assert np.array_equal(sqd, dist)
        assert abs(inertia - math.fsum(dist)) <= 1e-13 * math.fsum(dist)
        # resident points: the whole range and a ragged one
        labels_x, dist_x = km.predict(x)
        sq_x = km.transform_range(0, n, squared=True)
        check_against_predict(sq_x, labels_x, dist_x)
        assert np.array_equal(km.transform_range(0, n), np.sqrt(sq_x))
        assert np.array_equal(km.transform_range(37, n - 100, squared=True), sq_x[37:n - 63])
        err_x = check_accuracy(sq_x, x, c0, sample_rows(n, 1))
        # the fitted inertia is bitwise the next assignment's
        fitted = km.score_fitted()
        inertia_x, _ = km.assign()
        assert fitted == inertia_x
        print(f"\n[{_km_id(case)}] accuracy {err_q:.1e} / {err_x:.1e} (bar {4 * d * U:.1e})")
    finally:
        km.close()
        dev.close()


# filter path with the one-hot statistics, the exact path, centroid blocks, 16 warps per CTA
STATE_CASES = [c for c in KM_CASES if c[5][7] == 2048 and (c[0], c[1], tuple(c[4].items())) in
               {(3, 31, ()), (65, 3, ()), (8, 150, (("MLB200_KM_BLOCK", "64"),)), (16, 530, ())}]


@pytest.mark.parametrize("case", STATE_CASES, ids=_km_id)
def test_scoring_touches_no_fit_state(ctx, monkeypatch, case):
    """Two objects on the same points driven through the same steps; one also transforms and scores between them.
    Labels, centroids, the next assign (inertia, n_changed), the next update (shift, centroids) and the kernel timer
    stay bitwise what they are without those calls."""
    from ml_b200 import cabi
    d, k, n, chunk, env, _ = case
    x, q, c0, _ = km_problem(d, k, n)
    monkeypatch.setenv("MLB200_CHUNK", str(chunk))
    for key, val in env.items():
        monkeypatch.setenv(key, val)
    dev = cabi.Data.upload(ctx, x)
    a, b = cabi.Km(dev, k), cabi.Km(dev, k)

    def extras():
        a.transform(q)
        a.transform_range(0, n, squared=True)
        a.score(q)
        return a.score_fitted()

    try:
        for km in (a, b):
            km.set_kernel_timing(True)
            km.set_centroids(c0)
        for step in range(3):
            fitted = extras()
            got, want = a.assign(), b.assign()
            assert got == want and fitted == got[0]
            extras()
            assert np.array_equal(a.get_labels(), b.get_labels())
            assert np.array_equal(a.get_centroids(), b.get_centroids())
            assert a.update() == b.update()   # the update still applies the last assignment
            assert np.array_equal(a.get_centroids(), b.get_centroids())
        assert a.kernel_time_ms()[1] == b.kernel_time_ms()[1]
        assert a.launch_count > b.launch_count
    finally:
        a.close()
        b.close()
        dev.close()


def test_score_is_independent_of_batching(ctx):
    """More than one 2^20-point stage: the inertia of one call is the in-order sum of the inertias of its 2048-point
    pieces, bitwise, and the per-point values are those of the pieces."""
    from ml_b200 import cabi
    rng = np.random.default_rng(5)
    d, k = 2, 7
    x = np.ascontiguousarray(rng.standard_normal((4096, d)))
    m = (1 << 20) + 3 * 2048 + 17
    q = np.ascontiguousarray(rng.standard_normal((m, d)) * 3.0)
    dev = cabi.Data.upload(ctx, x)
    km = cabi.Km(dev, k)
    try:
        km.set_centroids(np.ascontiguousarray(x[:k].T))
        sqd, inertia = km.score(q)
        total = 0.0
        for lo in range(0, m, 2048):
            piece_sq, piece = km.score(q[lo:lo + 2048])
            assert np.array_equal(piece_sq, sqd[lo:lo + 2048])
            total += piece
        assert inertia == total
        _, again = km.score(q, want_sqdist=False)
        assert again == inertia
        assert abs(inertia - math.fsum(sqd)) <= 1e-13 * inertia
    finally:
        km.close()
        dev.close()


def test_edge_cases(ctx):
    """m = 0, points 1e6 away from every centroid, duplicate centroids (equal columns; argmin takes the lower index)."""
    from ml_b200 import cabi
    d, k, n, *_ = KM_CASES[0]
    x, q, c0, _ = km_problem(d, k, n)
    dev = cabi.Data.upload(ctx, x)
    km = cabi.Km(dev, k)
    try:
        km.set_centroids(c0)
        empty = np.zeros((0, d))
        assert km.transform(empty).shape == (0, k)
        assert km.score(empty)[1] == 0.0 and km.transform_range(5, 0).shape == (0, k)
        far = np.ascontiguousarray(q + 1e6)
        sq = km.transform(far, squared=True)
        check_against_predict(sq, *km.predict(far))
        check_accuracy(sq, far, c0, np.arange(far.shape[0]))
        dup = c0.copy()
        dup[:, 5] = dup[:, 2]
        dup[:, 9] = dup[:, 2]
        km.set_centroids(dup)
        sq = km.transform(q, squared=True)
        assert np.array_equal(sq[:, 5], sq[:, 2]) and np.array_equal(sq[:, 9], sq[:, 2])
        labels, dist = km.predict(q)
        check_against_predict(sq, labels, dist)
        assert not np.any(labels == 5) and not np.any(labels == 9)
    finally:
        km.close()
        dev.close()


def test_cabi_errors(ctx):
    import ctypes
    from ml_b200 import cabi
    lib = cabi.lib()
    d, k, n, *_ = KM_CASES[0]
    x, q, c0, _ = km_problem(d, k, n)
    dev = cabi.Data.upload(ctx, x)
    km = cabi.Km(dev, k)
    try:
        out = np.empty((k, q.shape[0]))
        inertia = ctypes.c_double()
        p_q, p_out = q.ctypes.data_as(ctypes.c_void_p), out.ctypes.data_as(ctypes.c_void_p)
        # before the centroids are set
        for rc in (lib.mlb_km_transform(km._h, p_q, q.shape[0], d, 0, p_out, q.shape[0]),
                   lib.mlb_km_transform_range(km._h, 0, 10, 0, p_out, 10),
                   lib.mlb_km_score(km._h, p_q, q.shape[0], d, None, ctypes.byref(inertia)),
                   lib.mlb_km_score_fitted(km._h, ctypes.byref(inertia))):
            assert rc == cabi.MLB_ESTATE
        km.set_centroids(c0)
        assert lib.mlb_km_transform(km._h, p_q, q.shape[0], d, 0, p_out, q.shape[0] - 1) == cabi.MLB_EINVAL    # ld_out < m
        assert lib.mlb_km_transform(km._h, p_q, q.shape[0], d - 1, 0, p_out, q.shape[0]) == cabi.MLB_EINVAL    # ld_x < D
        assert lib.mlb_km_transform_range(km._h, 0, 10, 0, p_out, 9) == cabi.MLB_EINVAL
        assert lib.mlb_km_transform_range(km._h, -1, 10, 0, p_out, 10) == cabi.MLB_EINVAL
        assert lib.mlb_km_transform_range(km._h, n - 5, 10, 0, p_out, 10) == cabi.MLB_EINVAL
        assert lib.mlb_km_score(km._h, p_q, q.shape[0], d - 1, None, ctypes.byref(inertia)) == cabi.MLB_EINVAL
        assert lib.mlb_km_score(km._h, p_q, q.shape[0], d, None, None) == cabi.MLB_EINVAL
    finally:
        km.close()
        dev.close()


def test_score_fitted_and_transform_range_do_not_depend_on_the_gpu_count():
    from ml_b200 import cabi
    count = cabi.device_count()
    if count < 2:
        pytest.skip("needs at least 2 GPUs")
    d, k, n, *_ = KM_CASES[0]
    x, _, c0, _ = km_problem(d, k, n)
    results = []
    for g in (1, 2, 4, 8):
        if g > count:
            break
        c = cabi.Context(g)
        dev = cabi.Data.upload(c, x)
        km = cabi.Km(dev, k)
        km.set_centroids(c0)
        results.append((km.score_fitted(), km.transform_range(0, n, squared=True), km.transform_range(n // 3, n // 2)))
        km.close()
        dev.close()
        c.close()
    for got in results[1:]:
        assert got[0] == results[0][0]
        assert np.array_equal(got[1], results[0][1]) and np.array_equal(got[2], results[0][2])


# ---------------------------------------------------------------- the fit (ml::Clustering::KMeans through cppyml)

def _cppyml():
    return __import__("ml_b200").import_cppyml()


def _blobs(n, d, k, seed):
    rng = np.random.default_rng(seed)
    centres = rng.uniform(-5.0, 5.0, size=(k, d))
    x = centres[rng.integers(0, k, size=n)] + rng.standard_normal((n, d))
    return np.ascontiguousarray(x)


def _ref_inertia(x, centroids_kd):
    return float(np.sum(np.min(ref_sq(x, centroids_kd.T), axis=1)))


def test_final_inertia_after_convergence_and_after_the_step_limit():
    c = _cppyml().clustering
    x = _blobs(30000, 6, 8, 11)
    km = c.KMeans(8)
    km.set_seed(3)
    km.set_absolute_tolerance(0.0)   # converges on unchanged labels: the last assignment is at the returned centroids
    assert km.fit(x)
    assert -km.score() == km.inertia
    km2 = c.KMeans(8)
    km2.set_seed(3)
    km2.set_maximum_steps(2)
    km2.fit(x)
    want = _ref_inertia(x, km2.centroids)
    assert abs(-km2.score() - want) <= 1e-12 * want
    assert abs(-km2.score(x) - want) <= 1e-12 * want


@pytest.mark.parametrize("converge", [True, False], ids=["converged", "step-limit"])
@pytest.mark.parametrize("lockstep", ["1", "0"])
def test_multi_start_uses_the_returned_centroids(monkeypatch, lockstep, converge):
    """Three starts, on the lockstep and the sequential path, either converged or all stopped at maximum_steps (then the
    fit returns the last start's centroids)."""
    monkeypatch.setenv("MLPP_KMEANS_LOCKSTEP", lockstep)
    c = _cppyml().clustering
    if converge:
        x, q = _blobs(20000, 5, 6, 21), _blobs(3000, 5, 6, 22)
    else:
        rng = np.random.default_rng(23)   # no cluster structure: the labels still move at the second step
        x, q = np.ascontiguousarray(rng.standard_normal((20000, 5))), np.ascontiguousarray(rng.standard_normal((3000, 5)))
    km = c.KMeans(6)
    km.set_seed(9)
    km.set_number_initialisations(3)
    if not converge:
        km.set_absolute_tolerance(0.0)
        km.set_maximum_steps(2)
    assert km.fit(x) == converge
    cent = km.centroids
    want = np.sqrt(ref_sq(q, cent.T))
    got = km.transform(q)
    assert np.all(np.abs(got - want) <= 4 * 5 * U * want)
    assert abs(-km.score(q) - _ref_inertia(q, cent)) <= 1e-12 * _ref_inertia(q, cent)
    assert abs(-km.score() - _ref_inertia(x, cent)) <= 1e-12 * _ref_inertia(x, cent)
    fitted = km.transform()
    assert fitted.shape == (x.shape[0], 6)
    rows = sample_rows(x.shape[0])
    assert np.all(np.abs(fitted[rows] - np.sqrt(ref_sq(x[rows], cent.T))) <= 4 * 5 * U * np.sqrt(ref_sq(x[rows], cent.T)))


def test_cppyml_surface():
    from sklearn.metrics.pairwise import euclidean_distances
    c = _cppyml().clustering
    x, q = _blobs(20000, 4, 5, 31), _blobs(2500, 4, 5, 32)
    km = c.KMeans(5)
    for call in (km.transform, km.score, km.assign_labels):
        with pytest.raises(ValueError):
            call(q)                # before any fit there are no centroids, so D does not match
    with pytest.raises(RuntimeError):
        km.score()
    km.set_seed(1)
    km.fit(x)
    t = km.transform(q)
    assert t.shape == (q.shape[0], 5) and t.dtype == np.float64
    ref = euclidean_distances(q, km.centroids)
    assert np.max(np.abs(t - ref)) <= 1e-9 * np.max(ref)
    labels, dist = km.assign_labels(q)
    s = km.score(q)
    assert isinstance(s, float) and abs(s + math.fsum(dist)) <= 1e-13 * math.fsum(dist)
    assert km.transform().shape == (x.shape[0], 5)
    assert km.transform(np.zeros((0, 4))).shape == (0, 5)
    assert km.score(np.zeros((0, 4))) == 0.0
    with pytest.raises(ValueError):
        km.transform(np.zeros((3, 5)))
    with pytest.raises(ValueError):
        km.score(np.zeros((3, 5)))
    with pytest.raises(TypeError):
        km.transform(q.astype(np.float32))
    with pytest.raises(TypeError):
        km.score(np.asfortranarray(q))
    km.release_device()
    with pytest.raises(RuntimeError):
        km.transform(q)
    with pytest.raises(RuntimeError):
        km.score()


_RANK_WORKER = """
import os, sys
import numpy as np
import torch
import torch.distributed as dist
sys.path.insert(0, {root!r})
from ml_b200 import import_cppyml
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
cppyml = import_cppyml()
box = [cppyml.distributed.unique_id() if rank == 0 else None]
dist.broadcast_object_list(box, src=0)
cppyml.distributed.init(local, rank, world, box[0])
x, init = np.load({x!r}), np.load({init!r})
lo, hi = cppyml.distributed.shard_range(x.shape[0], world, rank)
km = cppyml.clustering.KMeans(init.shape[0])
km.set_centroids_initialiser(cppyml.clustering.ExplicitCentroids(init))
km.set_absolute_tolerance(0.0)
km.set_maximum_steps(3)
km.fit(np.ascontiguousarray(x[lo:hi]))
np.save(os.path.join({out!r}, f"transform{{rank}}.npy"), km.transform())
np.save(os.path.join({out!r}, f"score{{rank}}.npy"), np.array([km.score()]))
np.save(os.path.join({out!r}, f"centroids{{rank}}.npy"), km.centroids)
dist.barrier()
dist.destroy_process_group()
"""


def test_transform_and_score_under_ml_distributed(ctx, tmp_path):
    """Two ranks under ml::Distributed: KMeans.transform() gives each rank its own rows (its global range), and
    KMeans.score() is the same on both and bitwise that of one process on all points."""
    import os
    import subprocess
    import sys
    from ml_b200 import cabi
    if cabi.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    x = _blobs(30011, 6, 7, 41)
    np.save(tmp_path / "x.npy", x)
    np.save(tmp_path / "init.npy", np.ascontiguousarray(x[:7]))
    script = tmp_path / "worker.py"
    script.write_text(_RANK_WORKER.format(root=root, x=str(tmp_path / "x.npy"), init=str(tmp_path / "init.npy"), out=str(tmp_path)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29657", str(script)]
    run = subprocess.run(cmd, cwd=root, capture_output=True, text=True, timeout=600)
    assert run.returncode == 0, run.stderr[-3000:]
    cent = np.load(tmp_path / "centroids0.npy")
    assert np.array_equal(cent, np.load(tmp_path / "centroids1.npy"))
    dev = cabi.Data.upload(ctx, x)
    km = cabi.Km(dev, 7)
    try:
        km.set_centroids(np.ascontiguousarray(cent.T))
        whole = km.transform_range(0, x.shape[0])
        fitted = km.score_fitted()
    finally:
        km.close()
        dev.close()
    for rank in (0, 1):
        lo, hi = cabi.shard_range(x.shape[0], 2, rank)
        assert np.array_equal(np.load(tmp_path / f"transform{rank}.npy"), whole[lo:hi])
        assert np.load(tmp_path / f"score{rank}.npy")[0] == -fitted
