"""One EM step and one K-means step restated plainly in NumPy, as the reference states them (ML/EM.cpp:190-263,
ML/KMeans.cpp:153-192), for comparing ONE kernel pass from chosen parameters (tests/test_gpu_kernel_matrix.py).

None of the kernels' tricks: no feature expansion, no shift by the data mean, no approximate exponential.  Log-densities
come from direct differences x - mu through a Cholesky solve per component (float64 BLAS), the per-point log-sum-exp
uses the exact maximum, and every sum over points is accumulated in np.longdouble: blocks of `_BLOCK` points are summed
by float64 BLAS (at most 64 terms: a few ulp) and the block sums in long double, so the sums over N points carry no
error that grows with N.  tests/test_onestep_reference.py pins these functions against the CPU oracle and against an
evaluation in long double throughout.

Conventions follow ml::EM: means (D, K), covariances (K, D, D), weights (K,), data (N, D) one point per row,
responsibilities (N, K).
"""
import math

import numpy as np
from scipy.linalg import cho_factor, solve_triangular

_BLOCK = 64
_EPSILON = 1e-15                       # EM.cpp:259: added to the diagonal of every new covariance
LOG_2PI = math.log(2.0 * math.pi)


def _block_sum(a):
    """Sum over axis 0 of a float64 array: float64 within blocks of _BLOCK rows, long double across blocks."""
    a = np.asarray(a, dtype=np.float64)
    n = a.shape[0]
    acc = np.zeros(a.shape[1:], dtype=np.longdouble)
    for b in range(0, n, _BLOCK):
        acc += a[b:b + _BLOCK].sum(axis=0)
    return acc


def _block_gram(w, c):
    """sum_i w_i c_i c_i^T for w (N,), c (N, D): float64 products of _BLOCK points per BLAS call, long double across."""
    n, d = c.shape
    acc = np.zeros((d, d), dtype=np.longdouble)
    for b in range(0, n, _BLOCK):
        cb = c[b:b + _BLOCK]
        acc += (cb * w[b:b + _BLOCK, None]).T @ cb
    return acc


def _block_weighted_sum(r, x):
    """r^T x for r (N, K), x (N, D): (K, D) in long double across blocks."""
    acc = np.zeros((r.shape[1], x.shape[1]), dtype=np.longdouble)
    for b in range(0, x.shape[0], _BLOCK):
        acc += r[b:b + _BLOCK].T @ x[b:b + _BLOCK]
    return acc


def log_densities(x, means, covs, weights):
    """(N, K): log(w_k) - log(sqrt|Sigma_k|) - (x - mu_k)^T Sigma_k^-1 (x - mu_k) / 2, the log of what EM.cpp:205-209
    stores per point and component (the constant D log(2 pi) / 2 left out, as there)."""
    x = np.asarray(x, dtype=np.float64)
    n, d = x.shape
    k = means.shape[1]
    out = np.empty((n, k))
    for c in range(k):
        low, _ = cho_factor(covs[c], lower=True)
        low = np.tril(low)
        y = solve_triangular(low, (x - means[:, c]).T, lower=True)
        q = np.einsum("ij,ij->j", y, y)
        log_sqrt_det = float(np.sum(np.log(np.diag(low))))
        out[:, c] = math.log(weights[c]) - log_sqrt_det - 0.5 * q if weights[c] > 0 else -np.inf
    return out


def responsibilities(x, means, covs, weights):
    """(log-likelihood of the E-step, responsibilities (N, K), per-point log-sum-exp (N,))."""
    lg = log_densities(x, means, covs, weights)
    m = lg.max(axis=1)
    e = np.exp(lg - m[:, None])
    s = e.sum(axis=1)
    resp = e / s[:, None]
    lse = m + np.log(s)
    ll = math.fsum(lse) / x.shape[0] - x.shape[1] * LOG_2PI / 2
    return ll, resp, lse


def em_mstep(x, resp):
    """EM::maximisation_step (EM.cpp:221-263) from responsibilities (N, K): new means (D, K), covariances (K, D, D) about
    the new means plus 1e-15 I, weights (K,)."""
    x = np.asarray(x, dtype=np.float64)
    resp = np.asarray(resp, dtype=np.float64)
    n, d = x.shape
    k = resp.shape[1]
    nk = _block_sum(resp)                                   # (K,) long double
    sums = _block_weighted_sum(resp, x)                     # (K, D) long double
    means = (sums / nk[:, None]).astype(np.float64)         # (K, D)
    covs = np.empty((k, d, d))
    for c in range(k):
        g = _block_gram(resp[:, c], x - means[c]) / nk[c]
        covs[c] = g.astype(np.float64) + _EPSILON * np.eye(d)
    weights = (nk / n).astype(np.float64)
    return np.ascontiguousarray(means.T), covs, weights


def em_step(x, means, covs, weights):
    """One EM iteration (EM.cpp:143-147) from (means (D, K), covs (K, D, D), weights (K,)): a dict with the E-step's
    log-likelihood (mean per point minus D log(2 pi) / 2, EM.cpp:211), responsibilities, labels (first maximum,
    EM.cpp:289-304), the top-two gap of each row, and the M-step's means, covariances, weights."""
    ll, resp, _ = responsibilities(x, means, covs, weights)
    new_means, new_covs, new_weights = em_mstep(x, resp)
    top2 = np.sort(resp, axis=1)[:, -2:] if resp.shape[1] > 1 else np.concatenate([np.zeros((resp.shape[0], 1)), resp], axis=1)
    return {"log_likelihood": ll, "responsibilities": resp, "labels": np.argmax(resp, axis=1).astype(np.uint32),
            "top2_gap": top2[:, 1] - top2[:, 0], "means": new_means, "covariances": new_covs, "weights": new_weights}


def sample_covariance(x):
    """EM::calculate_sample_covariance (EM.cpp:265-272): unbiased, about the mean, sums in long double."""
    x = np.asarray(x, dtype=np.float64)
    n = x.shape[0]
    mean = (_block_sum(x) / n).astype(np.float64)
    return (_block_gram(np.ones(n), x - mean) / (n - 1)).astype(np.float64)


def kappa(x, means, covs):
    """max_k (mu_k - c)^T Sigma_k^-1 (mu_k - c), c the data mean: the conditioning the library routes on (mlb200.h)."""
    x = np.asarray(x, dtype=np.float64)
    c = (_block_sum(x) / x.shape[0]).astype(np.float64)
    best = 0.0
    for k in range(means.shape[1]):
        low = np.tril(cho_factor(covs[k], lower=True)[0])
        y = solve_triangular(low, means[:, k] - c, lower=True)
        best = max(best, float(y @ y))
    return best


# ---------------------------------------------------------------- K-means

def squared_distances(x, centroids):
    """(N, K) squared distances (x - c).squaredNorm() by direct differences in float64 (not bitwise the reference's
    fused chain: see km_step for how near-ties are settled)."""
    x = np.asarray(x, dtype=np.float64)
    k = centroids.shape[1]
    out = np.empty((x.shape[0], k))
    for c in range(k):
        diff = x - centroids[:, c]
        out[:, c] = np.einsum("ij,ij->i", diff, diff)
    return out


def km_assign(x, centroids, tie_rel=1e-12):
    """KMeans::assign_label (KMeans.cpp:153-165) for every row: (labels, squared distances, indices settled by the
    oracle).  Wherever the best two float64 distances lie within `tie_rel` (relative) of each other the label and the
    distance come from oracle.kmeans_assign_label, which evaluates the reference's arithmetic bit for bit; elsewhere
    the label is the argmin (unambiguous) and the distance the float64 one (within a few ulp of the reference's)."""
    import oracle
    x = np.ascontiguousarray(x, dtype=np.float64)
    d2 = squared_distances(x, centroids)
    labels = np.argmin(d2, axis=1).astype(np.uint32)
    if d2.shape[1] > 1:
        part = np.partition(d2, 1, axis=1)
        close = (part[:, 1] - part[:, 0]) <= tie_rel * np.maximum(part[:, 1], 1e-300)
    else:
        close = np.zeros(x.shape[0], dtype=bool)
    ties = np.flatnonzero(close)
    dist = d2[np.arange(x.shape[0]), labels]
    for i in ties:
        labels[i], dist[i] = oracle.kmeans_assign_label(centroids, x[i])
    return labels, dist, ties


def km_update(x, labels, k):
    """KMeans::update_step (KMeans.cpp:180-192): per-cluster means (D, K) in long double; an empty cluster goes to the
    origin."""
    x = np.asarray(x, dtype=np.float64)
    d = x.shape[1]
    sums = np.zeros((k, d), dtype=np.longdouble)
    counts = np.bincount(labels, minlength=k)
    order = np.argsort(labels, kind="stable")
    bounds = np.concatenate([[0], np.cumsum(counts)])
    xs = x[order]
    for c in range(k):
        if counts[c]:
            sums[c] = _block_sum(xs[bounds[c]:bounds[c + 1]])
    cent = np.zeros((k, d))
    nz = counts > 0
    cent[nz] = (sums[nz] / counts[nz, None]).astype(np.float64)
    return np.ascontiguousarray(cent.T), counts


def km_step(x, centroids, prev_labels):
    """One assignment + update (KMeans.cpp:167-192) from centroids (D, K): a dict with labels, per-point squared
    distances, inertia (sum in long double), the number of labels that differ from `prev_labels`, the new centroids
    (D, K), the squared Frobenius shift of the centroids, and the indices whose label the oracle settled."""
    k = centroids.shape[1]
    labels, dist, ties = km_assign(x, centroids)
    inertia = math.fsum(dist)
    changed = int(np.count_nonzero(labels != np.asarray(prev_labels)))
    new_c, counts = km_update(x, labels, k)
    shift = math.fsum(((new_c - centroids) ** 2).ravel())
    return {"labels": labels, "distances": dist, "inertia": inertia, "changed": changed, "centroids": new_c,
            "shift": shift, "counts": counts, "ties": ties}
