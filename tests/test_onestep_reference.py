"""Pins of the one-step reference (tests/onestep_reference.py) on the CPU, and the check that the kernel matrix
(tests/test_gpu_kernel_matrix.py) covers every kernel instance of the dispatch code.  No GPU needed."""
import numpy as np
import pytest

import oracle
from tests import onestep_reference as ref


def rel_err(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def blobs(n, d, seed):
    rng = np.random.default_rng(seed)
    centres = rng.uniform(-3.0, 3.0, size=(5, d))
    return np.ascontiguousarray(centres[rng.integers(0, 5, size=n)] + rng.standard_normal((n, d)))


# ---------------------------------------------------------------- against the oracle

@pytest.mark.parametrize("n,d,k", [(500, 1, 2), (2000, 3, 5), (1500, 8, 4), (3000, 16, 7)])
def test_em_step_matches_oracle_first_step(n, d, k):
    """One step from the oracle's own start (explicit means, equal weights, the sample covariance everywhere)."""
    x = blobs(n, d, 10 + d)
    means = np.ascontiguousarray(x[:: n // k][:k].T)
    fit = oracle.em_fit(x, k, means_init=oracle.EXPLICIT, explicit_means=means, maximum_steps=1)
    cov = ref.sample_covariance(x)
    assert rel_err(cov, np.atleast_2d(np.cov(x.T))) <= 1e-13
    st = ref.em_step(x, means, np.stack([cov] * k), np.full(k, 1.0 / k))
    assert abs(st["log_likelihood"] - fit.log_likelihood) <= 1e-12 * abs(fit.log_likelihood)
    assert np.max(np.abs(st["responsibilities"] - fit.responsibilities)) <= 1e-12
    assert rel_err(st["means"], fit.means) <= 1e-12
    assert rel_err(st["weights"], fit.mixing_probabilities) <= 1e-12
    for c in range(k):
        assert rel_err(st["covariances"][c], fit.covariances[c]) <= 1e-12


@pytest.mark.parametrize("n,d,k", [(1000, 2, 3), (4000, 8, 40), (2500, 33, 9)])
def test_km_step_matches_oracle_first_step(n, d, k):
    """One assignment + update (KMeans.cpp:167-192), with a centroid no point reaches (its cluster goes to the origin)."""
    x = blobs(n, d, 20 + d)
    c0 = np.ascontiguousarray(x[:: n // k][:k].T)
    c0[:, 1] = 1e3
    fit = oracle.kmeans_fit(x, k, init=oracle.EXPLICIT, explicit_means=c0, maximum_steps=1)
    st = ref.km_step(x, c0, np.zeros(n, dtype=np.uint32))
    assert np.array_equal(st["labels"], fit.labels)
    assert abs(st["inertia"] - fit.inertia) <= 1e-13 * fit.inertia
    assert st["counts"][1] == 0 and np.all(st["centroids"][:, 1] == 0.0)
    assert rel_err(st["centroids"], fit.centroids) <= 1e-13
    assert st["changed"] == np.count_nonzero(fit.labels)


def test_km_assign_settles_near_ties_with_the_oracle():
    """Points on the bisector of two centroids: the label and distance are the reference's scan (strict <)."""
    rng = np.random.default_rng(3)
    c = np.array([[0.0, 1.0], [0.0, 0.0]])          # (D, K): (0, 0) and (1, 0)
    x = np.stack([np.full(50, 0.5), rng.normal(size=50)], axis=1)
    labels, dist, ties = ref.km_assign(x, c)
    assert len(ties) == 50
    for i in range(50):
        assert (labels[i], dist[i]) == oracle.kmeans_assign_label(c, x[i])
    fl, fd = oracle.kmeans_assign_fused(c, x)
    assert np.array_equal(fl, labels)
    assert np.max(np.abs(fd - dist) / dist) <= 1e-15


# ---------------------------------------------------------------- against long double throughout

def _chol_ld(a):
    d = a.shape[0]
    low = np.zeros((d, d), dtype=np.longdouble)
    for j in range(d):
        s = a[j, j] - np.sum(low[j, :j] ** 2)
        low[j, j] = np.sqrt(s)
        for i in range(j + 1, d):
            low[i, j] = (a[i, j] - np.sum(low[i, :j] * low[j, :j])) / low[j, j]
    return low


def _em_step_ld(x, means, covs, weights):
    """The formulas of ref.em_step evaluated in long double throughout (Cholesky, solves, exp / log, sums)."""
    x = x.astype(np.longdouble)
    n, d = x.shape
    k = means.shape[1]
    lg = np.empty((n, k), dtype=np.longdouble)
    for c in range(k):
        low = _chol_ld(covs[c].astype(np.longdouble))
        diff = x - means[:, c].astype(np.longdouble)
        y = np.empty_like(diff)
        for a in range(d):                                   # forward substitution, all points at once
            y[:, a] = (diff[:, a] - y[:, :a] @ low[a, :a]) / low[a, a]
        lg[:, c] = np.log(np.longdouble(weights[c])) - np.sum(np.log(np.diag(low))) - 0.5 * np.sum(y * y, axis=1)
    m = lg.max(axis=1)
    e = np.exp(lg - m[:, None])
    s = e.sum(axis=1)
    resp = e / s[:, None]
    ll = np.sum(m + np.log(s)) / n - d * np.log(2 * np.pi * np.longdouble(1)) / 2
    nk = resp.sum(axis=0)
    new_means = (resp.T @ x) / nk[:, None]
    new_covs = []
    for c in range(k):
        cd = x - new_means[c]
        new_covs.append((cd * resp[:, c:c + 1]).T @ cd / nk[c] + np.longdouble(1e-15) * np.eye(d))
    return ll, resp, new_means.T, np.stack(new_covs), nk / n


@pytest.mark.parametrize("n,d,k", [(2000, 1, 3), (1200, 4, 5), (2000, 8, 6)])
def test_em_step_within_1e14_of_long_double(n, d, k):
    """The reference is at least 100x tighter than the 1e-11 bars it is used with."""
    rng = np.random.default_rng(d)
    x = blobs(n, d, 30 + d)
    means = np.ascontiguousarray(x[rng.choice(n, size=k, replace=False)].T)
    covs = []
    for _ in range(k):
        a = rng.standard_normal((d, d))
        covs.append(a @ a.T / d + 0.5 * np.eye(d))
    covs = np.stack(covs)
    w = rng.dirichlet(np.full(k, 2.0))
    st = ref.em_step(x, means, covs, w)
    ll, resp, nm, nc, nw = _em_step_ld(x, means, covs, w)
    assert abs(st["log_likelihood"] - float(ll)) <= 1e-14 * abs(float(ll))
    assert np.max(np.abs(st["responsibilities"] - resp.astype(np.float64))) <= 1e-14
    assert rel_err(st["means"], nm.astype(np.float64)) <= 1e-14
    assert rel_err(st["weights"], nw.astype(np.float64)) <= 1e-14
    for c in range(k):
        assert rel_err(st["covariances"][c], nc[c].astype(np.float64)) <= 1e-14


def test_km_step_within_1e14_of_long_double():
    x = blobs(2000, 5, 40)
    c0 = np.ascontiguousarray(x[:: 250][:8].T)
    st = ref.km_step(x, c0, np.zeros(2000, dtype=np.uint32))
    xl = x.astype(np.longdouble)
    d2 = np.stack([np.sum((xl - c0[:, c].astype(np.longdouble)) ** 2, axis=1) for c in range(8)], axis=1)
    assert np.array_equal(st["labels"], np.argmin(d2, axis=1))
    assert abs(st["inertia"] - float(np.sum(np.min(d2, axis=1)))) <= 1e-14 * st["inertia"]
    want = np.stack([xl[st["labels"] == c].mean(axis=0) for c in range(8)], axis=1)
    assert rel_err(st["centroids"], want.astype(np.float64)) <= 1e-14


# ---------------------------------------------------------------- coverage of the kernel matrix
# Every instance the dispatch code can launch.  Mirrors em_kernel_for and the split / direct selection in mlb_em_create
# (ml_b200/csrc/em.cu), and km_kernel_for, km_warps_per_cta, the statistics selection in mlb_km_create and
# km_stats_use_sorted (ml_b200/csrc/kmeans.cu).  A new instance there belongs here and in the matrix.
FUSED = {(dp, kp, mode) for dp in (4, 8, 16) for kp in (8, 16, 32) for mode in (0, 1, 2)}
SPLIT = {(nt, mw) for nt in (2, 4, 8) for mw in (3, 4, 5)}
DIRECT_NB = {1, 2, 0}                                  # em_direct_e_kernel<NB>: 1, 2, and 0 for every wider D
KM_ASSIGN = {(dp, nw, compact) for dp, nws in ((4, (4, 8, 16)), (8, (4, 8, 16)), (16, (4, 8, 16)), (32, (4, 8, 16)), (64, (4, 8)))
             for nw in nws for compact in (False, True)}
KM_STATS = ({("small", dp) for dp in (4, 8, 16, 32)} | {("sorted", dp, blocked) for dp in (4, 8, 16, 32, 64, 128) for blocked in (False,)}
            | {("sorted", 8, True), ("owner", 8, True), ("owner", 16, False)} | {("exact", False), ("exact", True)})


def test_kernel_matrix_covers_every_instance():
    from tests.test_gpu_kernel_matrix import EM_CASES, KM_CASES
    fused, split, direct = set(), set(), set()
    for _, _, _, _, force, (path, dp, kp, nt, mw, _, nb, _) in EM_CASES:
        if force == 3:
            direct.add(nb if nb in (1, 2) else 0)
        elif path == 1:
            fused |= {(dp, kp, mode) for mode in (0, 1, 2)}   # step, mstep_from_*, emit / predict
        elif path == 2:
            split.add((nt, mw))
        else:
            direct.add(nb if nb in (1, 2) else 0)
    assign, stats = set(), set()
    for _, _, _, _, env, (dp, kp, kb, nblocks, nw, exact, kind, _) in KM_CASES:
        if exact:
            stats |= {("exact", False), ("exact", True)}    # assign (full statistics) and predict (compact)
        else:
            assign |= {(dp, nw, False), (dp, nw, True)}     # assign + update, and predict
        name = ("small", "sorted", "owner")[kind]
        stats.add((name, dp) if kind == 0 else (name, dp, nblocks > 1))
    assert FUSED <= fused, FUSED - fused
    assert SPLIT <= split, SPLIT - split
    assert DIRECT_NB <= direct, DIRECT_NB - direct
    assert KM_ASSIGN <= assign, KM_ASSIGN - assign
    assert KM_STATS <= stats, KM_STATS - stats
