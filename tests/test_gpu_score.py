"""Scoring: log p(x) under the current parameters (mlb_em_score, mlb_em_score_fitted, ml::EM::log_likelihoods and the
cppyml score_samples / score / bic / aic).

The exact reference is tests/onestep_reference.responsibilities(...)[2] - D log(2 pi) / 2: a long-double log-sum-exp of
log-densities formed with Cholesky solves.  Every kernel instance is reached through the shapes of the kernel matrix
(tests/test_gpu_kernel_matrix.py), with its hard parameters (a weight of 1e-6, condition number 1e3, a mean off the data),
at chunk 128 and 2048 and ragged N, and each case asserts the configuration it ran.

Bars: per point |l_dev - l_ref| <= 1e-11 max(1, |l_ref|); the mean within 1e-12 relative.
"""
import math

import numpy as np
import pytest

from tests import onestep_reference as ref
from tests.test_gpu_kernel_matrix import EM_CASES, _em_id, em_problem

pytestmark = pytest.mark.gpu

POINT_BAR = 1e-11
MEAN_BAR = 1e-12
LOG_2PI = math.log(2.0 * math.pi)


@pytest.fixture(scope="module")
def ctx():
    from ml_b200 import cabi
    assert cabi.device_count() >= 1, "no CUDA device: the product has no CPU fallback"
    c = cabi.Context(1)
    yield c
    c.close()


def ref_scores(x, params):
    means, covs, w = params
    _, _, lse = ref.responsibilities(x, means, covs, w)
    return lse - x.shape[1] * LOG_2PI / 2


def point_err(got, want):
    assert np.all(np.isfinite(got))
    return float(np.max(np.abs(got - want) / np.maximum(1.0, np.abs(want))))


def mean_err(got, want):
    return abs(got - math.fsum(want) / len(want)) / abs(math.fsum(want) / len(want))


@pytest.mark.parametrize("case", EM_CASES, ids=_em_id)
def test_score_every_instance(ctx, monkeypatch, case):
    """score (new points) and score_fitted (resident points) of every fused, split and direct instance."""
    from ml_b200 import cabi
    d, k, n, chunk, force, expected = case
    pb = em_problem(d, k, n)
    monkeypatch.setenv("MLB200_CHUNK", str(chunk))
    dev = cabi.Data.upload(ctx, pb["x"])
    em = cabi.Em(dev, k)
    try:
        cfg = em.kernel_config()
        assert tuple(cfg[f] for f in cabi.EM_CONFIG_FIELDS) == expected, cfg
        if force:
            em.force_path(3)
        em.set_params(*pb["params"])
        _, route = em.conditioning()
        assert route == (3 if (force or expected[0] == 0 or pb["kappa"] > 3e5) else expected[0])
        want_x, want_q = ref_scores(pb["x"], pb["params"]), ref_scores(pb["q"], pb["params"])
        got_q, mean_q = em.score(pb["q"])
        got_x, mean_x = em.score_fitted()
        errs = {"score": point_err(got_q, want_q), "score.mean": mean_err(mean_q, want_q),
                "fitted": point_err(got_x, want_x), "fitted.mean": mean_err(mean_x, want_x)}
        print(f"{_em_id(case)} route {route}: " + " ".join(f"{key} {val:.2e}" for key, val in errs.items()))
        assert errs["score"] <= POINT_BAR and errs["fitted"] <= POINT_BAR, errs
        assert errs["score.mean"] <= MEAN_BAR and errs["fitted.mean"] <= MEAN_BAR, errs
    finally:
        em.close()
        dev.close()


# one shape per path: fused (em_small_kernel, em_kernel), split, and the fused shape forced onto the direct kernels
PATH_SHAPES = [(8, 16, 0), (16, 32, 0), (32, 17, 0), (16, 32, 3)]


def _path_id(shape):
    d, k, force = shape
    return f"D{d}-K{k}" + ("-direct" if force else "")


@pytest.mark.parametrize("shape", PATH_SHAPES, ids=_path_id)
def test_score_fitted_mean_matches_the_next_step(ctx, shape):
    """At theta, score_fitted's mean is the log-likelihood the next step reports (it batches its logs: not bitwise)."""
    from ml_b200 import cabi
    d, k, force = shape
    pb = em_problem(d, k, 20443)
    dev = cabi.Data.upload(ctx, pb["x"])
    em = cabi.Em(dev, k)
    try:
        if force:
            em.force_path(3)
        em.set_params(*pb["params"])
        _, mean = em.score_fitted(want_log_densities=False)
        ll = em.step()
        assert abs(mean - ll) <= 1e-13 * abs(ll), (mean, ll)
    finally:
        em.close()
        dev.close()


def _fit_state(ctx, x, q, k, force, score):
    from ml_b200 import cabi
    dev = cabi.Data.upload(ctx, x)
    em = cabi.Em(dev, k)
    try:
        if force:
            em.force_path(3)
        em.set_params(*em_problem(x.shape[1], k, x.shape[0])["params"])
        em.run_steps(3)
        path = em.last_path
        if score:
            em.score(q)
            em.score_fitted()
            em.score_fitted(want_log_densities=False)
        resp, labels = em.emit()
        params = em.get_params()
        ll = em.step()
        return resp, labels, params, ll, path, em.last_path, em.get_params()
    finally:
        em.close()
        dev.close()


@pytest.mark.parametrize("shape", PATH_SHAPES, ids=_path_id)
def test_scoring_leaves_the_fit_state_alone(ctx, shape):
    """Fit, score, emit: responsibilities, labels, the next step and its path are bitwise those of the same fit unscored."""
    d, k, force = shape
    pb = em_problem(d, k, 20443)
    plain = _fit_state(ctx, pb["x"], pb["q"], k, force, False)
    scored = _fit_state(ctx, pb["x"], pb["q"], k, force, True)
    assert plain[4] == scored[4] == (3 if force else (1 if d <= 16 else 2))
    assert np.array_equal(plain[0], scored[0]) and np.array_equal(plain[1], scored[1])
    for a, b in zip(plain[2], scored[2]):
        assert np.array_equal(a, b)
    assert plain[3] == scored[3] and plain[5] == scored[5]
    for a, b in zip(plain[6], scored[6]):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("shape", PATH_SHAPES, ids=_path_id)
def test_per_point_values_do_not_depend_on_the_batch(ctx, monkeypatch, shape):
    """Alone, permuted, in slices, in a batch that crosses a staging boundary, resident: the same bits per point."""
    from ml_b200 import cabi
    d, k, force = shape
    pb = em_problem(d, k, 20443)
    monkeypatch.setenv("MLB200_CHUNK", "2048")
    rng = np.random.default_rng(7)
    big = pb["q"][rng.integers(0, len(pb["q"]), size=(1 << 20) + 17)]
    big[-len(pb["q"]):] = pb["q"]
    dev = cabi.Data.upload(ctx, pb["x"])
    em = cabi.Em(dev, k)
    try:
        if force:
            em.force_path(3)
        em.set_params(*pb["params"])
        base, mean = em.score(pb["q"])
        perm = rng.permutation(len(pb["q"]))
        assert np.array_equal(em.score(pb["q"][perm])[0], base[perm])
        for lo, hi in [(0, 1), (5, 6), (17, 400), (400, len(pb["q"]))]:
            assert np.array_equal(em.score(np.ascontiguousarray(pb["q"][lo:hi]))[0], base[lo:hi])
        got_big, mean_big = em.score(big)
        assert np.array_equal(got_big[-len(pb["q"]):], base)
        assert em.score(big)[1] == mean_big and em.score(pb["q"])[1] == mean
        # the resident points scored as new points, and the other way round
        fitted, fmean = em.score_fitted()
        assert np.array_equal(em.score(pb["x"])[0], fitted)
        assert em.score_fitted()[1] == fmean
    finally:
        em.close()
        dev.close()


@pytest.mark.parametrize("d,k", [(8, 4), (16, 6), (24, 5)])
def test_far_components_and_far_points(ctx, d, k):
    """A component at kappa > 3e5 sends scoring to the direct kernels, as predict; points 1e3 standard deviations out
    stay finite and meet the bar."""
    from ml_b200 import cabi
    rng = np.random.default_rng(d + k)
    x = rng.standard_normal((9000, d))
    means = np.ascontiguousarray(x[rng.choice(len(x), size=k, replace=False)].T)
    means[:, 0] = 30.0                               # far from the data centre ...
    covs = np.stack([np.eye(d) for _ in range(k)])
    covs[0] = np.eye(d) * 1e-3                       # ... and tight: kappa = 9e5 d
    w = np.full(k, 1.0 / k)
    far = x[:200] + 1e3 * rng.choice([-1.0, 1.0], size=(200, d))   # ~1e3 sigma out of every unit component
    dev = cabi.Data.upload(ctx, x)
    em = cabi.Em(dev, k)
    try:
        em.set_params(means, covs, w)
        kap, route = em.conditioning()
        assert kap > 3e5 and route == 3
        for pts in (x[:3000], far):
            got, mean = em.score(np.ascontiguousarray(pts))
            want = ref_scores(pts, (means, covs, w))
            assert point_err(got, want) <= POINT_BAR and mean_err(mean, want) <= MEAN_BAR
        got, mean = em.score_fitted()
        want = ref_scores(x, (means, covs, w))
        assert point_err(got, want) <= POINT_BAR and mean_err(mean, want) <= MEAN_BAR
    finally:
        em.close()
        dev.close()


def test_cppyml_matches_sklearn():
    """The mouse fit of test_em_mouse_matches_sklearn, its parameters loaded into a GaussianMixture."""
    from sklearn.mixture import GaussianMixture
    from ml_b200 import import_cppyml
    from tests.datasets import mouse_numpy
    clustering = import_cppyml().clustering
    data = mouse_numpy()
    em = clustering.EM(3)
    em.set_seed(42)
    em.set_means_initialiser(clustering.KPP())
    em.set_absolute_tolerance(1e-10)
    em.set_relative_tolerance(0)
    em.set_maximum_steps(1000)
    assert em.fit(data)
    gm = GaussianMixture(n_components=3, covariance_type="full")
    gm.weights_ = np.asarray(em.mixing_probabilities)
    gm.means_ = np.ascontiguousarray(np.asarray(em.means).T)
    gm.covariances_ = np.stack([em.covariance(c) for c in range(3)])
    gm.precisions_cholesky_ = np.stack([np.linalg.inv(np.linalg.cholesky(c)).T for c in gm.covariances_])
    for arg in (None, data):
        assert em.score_samples(arg).shape == (len(data),)
        assert np.max(np.abs(em.score_samples(arg) - gm.score_samples(data))) <= 1e-10
        assert abs(em.score(arg) - gm.score(data)) <= 1e-10
        assert abs(em.bic(arg) - gm.bic(data)) <= 1e-10 * max(1.0, abs(gm.bic(data)))
        assert abs(em.aic(arg) - gm.aic(data)) <= 1e-10 * max(1.0, abs(gm.aic(data)))
    # the fit's own log-likelihood belongs to the parameters before the last M-step; score() to the returned ones
    assert abs(em.score() - em.log_likelihood) <= 1e-8


def test_score_fitted_is_bitwise_invariant_in_the_gpu_count():
    from ml_b200 import cabi
    have = cabi.device_count()
    if have < 2:
        pytest.skip(f"needs at least 2 GPUs, have {have}")
    pb = em_problem(16, 32, 20443)
    x = np.ascontiguousarray(np.tile(pb["x"], (40, 1)))     # 817720 points: every GPU holds some chunks
    results = {}
    for g in [c for c in (1, 2, 4, 8) if c <= have]:
        c = cabi.Context(g)
        try:
            dev = cabi.Data.upload(c, x)
            em = cabi.Em(dev, 32)
            em.set_params(*pb["params"])
            results[g] = em.score_fitted()
            em.close()
            dev.close()
        finally:
            c.close()
    for g, (vals, mean) in results.items():
        print(f"G={g}: mean {mean!r}")
        assert np.array_equal(vals, results[1][0]) and mean == results[1][1], g


def test_errors(ctx):
    from ml_b200 import cabi, import_cppyml
    pb = em_problem(8, 16, 20443)
    dev = cabi.Data.upload(ctx, pb["x"])
    em = cabi.Em(dev, 16)
    try:
        with pytest.raises(cabi.MlbError) as e:
            em.score_fitted()
        assert e.value.code == cabi.MLB_ESTATE
        with pytest.raises(cabi.MlbError) as e:
            em.score(pb["q"])
        assert e.value.code == cabi.MLB_ESTATE
        em.set_params(*pb["params"])
        q = np.ascontiguousarray(pb["q"])
        rc = cabi.lib().mlb_em_score(em._h, q.ctypes.data_as(cabi._vp), len(q), 7, None, None)
        assert rc == cabi.MLB_EINVAL
        assert math.isnan(em.score(np.empty((0, 8)))[1])
    finally:
        em.close()
        dev.close()
    clustering = import_cppyml().clustering
    model = clustering.EM(3)
    data = np.ascontiguousarray(pb["x"][:2000])
    with pytest.raises(RuntimeError):
        model.score()                                    # no fit yet
    model.fit(data)
    with pytest.raises(TypeError):
        model.score_samples(data.astype(np.float32))
    with pytest.raises(TypeError):
        model.score_samples(np.asfortranarray(data))
    with pytest.raises(ValueError):
        model.score(np.ascontiguousarray(data[:, :5]))
    model.release_device()
    with pytest.raises(RuntimeError):
        model.score_samples()
    with pytest.raises(RuntimeError):
        model.bic(data)
    exact = clustering.EM(3)
    exact.fit(np.ascontiguousarray(data[:3]))
    with pytest.raises(RuntimeError):
        exact.score()
