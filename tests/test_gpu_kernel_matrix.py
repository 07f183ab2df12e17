"""Every EM and K-means kernel instantiation against a one-step reference (tests/onestep_reference.py).

The kernels are templates, and which instance runs is decided inside the library from (D, K, chunk).  Each case below
names the configuration it expects (Em.kernel_config() / Km.kernel_config()) and asserts it, so a change of the selection
rules fails here instead of quietly moving coverage elsewhere; tests/test_onestep_reference.py checks on the CPU that
the expected configurations cover every instance of the dispatch code.

Each case takes ONE kernel pass from parameters it chooses (unequal weights, one at 1e-6; correlated covariances with
condition number 1e3, different per component; means at data points and one off the data), so any K up to the path's
limit can be reached without the constraints a converging fit puts on the data.  Every case runs at chunk 128 (what
Layout::make picks below ~0.9M points) and at chunk 2048 (what production runs at N = 1e8 use), set through MLB200_CHUNK
before the upload; N leaves a ragged last chunk (n_chunks * chunk - 37 points), a sub-tile remainder that is not a
multiple of 16, and at chunk 2048 either 10 chunks or 5 (three of the 8 virtual shards empty).

Bars: 1e-11 relative for the log-likelihood, means and weights, 1e-11 for each covariance relative to its largest entry,
1e-12 absolute for responsibilities: 100x inside the project's 1e-9 parity bar.  Each case prints its largest errors
(run with -s) so the margin under each bar can be read from the log.
"""
import functools

import numpy as np
import pytest

import oracle
from tests import onestep_reference as ref

pytestmark = pytest.mark.gpu

BAR = 1e-11          # log-likelihood, means, weights, covariances (relative)
RESP_BAR = 1e-12     # responsibilities (absolute)
KM_BAR = 1e-13       # inertia and centroids (relative)
N_A = 10 * 2048 - 37     # 20443: 10 chunks of 2048 (160 of 128), the last one ragged; N % 16 = 11
N_B = 5 * 2048 - 37      # 10203: 5 chunks of 2048, so virtual shards 5..7 hold none
N_PREDICT = 3000

# (D, K, N, expected (path, DP, KP, NT, MW, direct_DP, direct_NB)); path 1 fused em_kernel / em_small_kernel<DP, KP>,
# 2 split em_split_e_kernel<NT> + em_split_m_kernel<NT, MW>, 0 direct kernels only (D > 64 or K > 256).
EM_SHAPES = [
    (3, 7, N_A, (1, 4, 8, 1, 0, 8, 1)),
    (4, 16, N_B, (1, 4, 16, 2, 0, 8, 1)),
    (2, 29, N_A, (1, 4, 32, 4, 0, 8, 1)),
    (1, 32, N_B, (1, 4, 32, 4, 0, 8, 1)),
    (5, 8, N_A, (1, 8, 8, 1, 0, 8, 1)),
    (7, 9, N_B, (1, 8, 16, 2, 0, 8, 1)),
    (8, 32, N_A, (1, 8, 32, 4, 0, 8, 1)),
    (6, 17, N_B, (1, 8, 32, 4, 0, 8, 1)),
    (9, 1, N_A, (1, 16, 8, 1, 0, 16, 2)),
    (16, 16, N_B, (1, 16, 16, 2, 0, 16, 2)),
    (12, 11, N_A, (1, 16, 16, 2, 0, 16, 2)),
    (16, 32, N_B, (1, 16, 32, 4, 0, 16, 2)),
    (13, 25, N_A, (1, 16, 32, 4, 0, 16, 2)),
    (30, 5, N_B, (2, 32, 16, 2, 3, 32, 4)),
    (17, 16, N_A, (2, 20, 16, 2, 4, 24, 3)),
    (27, 3, N_B, (2, 28, 16, 2, 5, 32, 4)),
    (32, 17, N_A, (2, 32, 32, 4, 3, 32, 4)),
    (20, 24, N_B, (2, 20, 32, 4, 4, 24, 3)),
    (28, 32, N_A, (2, 28, 32, 4, 5, 32, 4)),
    (8, 40, N_B, (2, 8, 64, 8, 3, 8, 1)),
    (64, 64, N_A, (2, 64, 64, 8, 4, 64, 8)),
    (16, 256, N_A, (2, 16, 256, 8, 5, 16, 2)),
    (52, 70, N_B, (2, 52, 128, 8, 5, 56, 7)),
    (8, 256, N_B, (2, 8, 256, 8, 3, 8, 1)),
    (8, 257, N_A, (0, 0, 0, 0, 0, 8, 1)),
    (65, 3, N_B, (0, 0, 0, 0, 0, 72, 9)),
    (128, 2, N_A, (0, 0, 0, 0, 0, 128, 16)),
    (96, 9, N_B, (0, 0, 0, 0, 0, 96, 12)),
]

# (D, K, N, chunk, force_path, expected config incl. chunk): every shape at chunk 128 and 2048 on its own path, and at
# chunk 128 forced onto the direct kernels; one shape also at 4096, the largest chunk MLB200_CHUNK accepts.
EM_CASES = []
for _d, _k, _n, _cfg in EM_SHAPES:
    for _chunk in (128, 2048):
        EM_CASES.append((_d, _k, _n, _chunk, 0, _cfg + (_chunk,)))
    EM_CASES.append((_d, _k, _n, 128, 3, _cfg + (128,)))
EM_CASES.append((16, 32, N_B, 4096, 0, (1, 16, 32, 4, 0, 16, 2, 4096)))


def _em_id(case):
    d, k, n, chunk, force, _ = case
    return f"D{d}-K{k}-N{n}-c{chunk}" + ("-direct" if force else "")


# (D, K, N, chunk, env, expected (DP, KP, KB, nblocks, nw, exact, stats, chunk)); stats 0 one-hot km_stats_small_kernel,
# 1 counting sort km_stats_sorted_kernel, 2 owner warps km_stats_kernel.  nw = warps per CTA of km_assign_kernel.
KM_SHAPES = [
    (3, 31, N_A, {}, (4, 32, 32, 1, 4, 0, 0)),
    (4, 1200, N_A, {}, (4, 1216, 1216, 1, 8, 0, 1)),
    (3, 2430, N_A, {}, (4, 2432, 2432, 1, 16, 0, 1)),
    (8, 32, N_B, {}, (8, 32, 32, 1, 4, 0, 0)),
    (7, 600, N_A, {}, (8, 608, 608, 1, 8, 0, 1)),
    (8, 1240, N_A, {}, (8, 1248, 1248, 1, 16, 0, 1)),
    (5, 100, N_B, {}, (8, 128, 128, 1, 4, 0, 1)),
    (16, 20, N_A, {}, (16, 32, 32, 1, 4, 0, 0)),
    (15, 280, N_B, {}, (16, 288, 288, 1, 8, 0, 1)),
    (16, 530, N_A, {}, (16, 544, 544, 1, 16, 0, 1)),
    (9, 63, N_B, {}, (16, 64, 64, 1, 4, 0, 1)),
    (32, 31, N_A, {}, (32, 32, 32, 1, 4, 0, 0)),
    (30, 90, N_B, {}, (32, 96, 96, 1, 8, 0, 1)),
    (32, 150, N_A, {}, (32, 160, 160, 1, 16, 0, 1)),
    (17, 64, N_B, {}, (32, 64, 64, 1, 4, 0, 1)),
    (64, 50, N_A, {}, (64, 64, 64, 1, 4, 0, 1)),
    (40, 96, N_B, {}, (64, 96, 96, 1, 8, 0, 1)),
    (65, 3, N_A, {}, (128, 32, 32, 1, 4, 1, 1)),
    (100, 40, N_B, {}, (128, 64, 64, 1, 4, 1, 1)),
    (8, 150, N_A, {"MLB200_KM_BLOCK": "64"}, (8, 192, 64, 3, 4, 0, 1)),
    (8, 150, N_B, {"MLB200_KM_BLOCK": "64", "MLB200_KM_STATS": "owner"}, (8, 192, 64, 3, 4, 0, 2)),
    (16, 100, N_A, {"MLB200_KM_STATS": "owner"}, (16, 128, 128, 1, 4, 0, 2)),
]
KM_CASES = []
for _d, _k, _n, _env, _cfg in KM_SHAPES:
    for _chunk in (128, 2048):
        KM_CASES.append((_d, _k, _n, _chunk, _env, _cfg + (_chunk,)))
KM_CASES.append((32, 150, N_B, 4096, {}, (32, 160, 160, 1, 16, 0, 1, 4096)))
KM_CASES.append((8, 150, N_B, 4096, {"MLB200_KM_BLOCK": "64"}, (8, 192, 64, 3, 4, 0, 1, 4096)))


def _km_id(case):
    d, k, n, chunk, env, _ = case
    tags = "".join(f"-{key.split('_')[-1].lower()}{val}" for key, val in env.items())
    return f"D{d}-K{k}-N{n}-c{chunk}{tags}"


@pytest.fixture(scope="module")
def ctx():
    from ml_b200 import cabi
    assert cabi.device_count() >= 1, "no CUDA device: the product has no CPU fallback"
    c = cabi.Context(1)
    yield c
    c.close()


def rel_err(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def cov_err(got, want):
    """Largest error of any covariance relative to that covariance's own largest entry."""
    return max(rel_err(g, w) for g, w in zip(got, want))


# ---------------------------------------------------------------- problems

def em_data(n, d, seed):
    rng = np.random.default_rng(seed)
    centres = rng.uniform(-2.0, 2.0, size=(6, d))
    x = centres[rng.integers(0, 6, size=n + N_PREDICT)] + rng.standard_normal((n + N_PREDICT, d))
    return np.ascontiguousarray(x[:n]), np.ascontiguousarray(x[n:])


def random_covariance(rng, d, cond=1e3):
    """A correlated covariance with condition number `cond` (a random rotation of geometric eigenvalues)."""
    if d == 1:
        return np.array([[rng.uniform(0.3, 3.0)]])
    q, _ = np.linalg.qr(rng.standard_normal((d, d)))
    ev = np.geomspace(0.3, 0.3 * cond, d) * rng.uniform(0.5, 2.0)
    c = (q * ev) @ q.T
    return (c + c.T) / 2


def em_params(x, k, seed):
    """(means (D, K), covariances (K, D, D), weights (K,)): means at data points and the last one off the data,
    Dirichlet weights with one component at 1e-6."""
    rng = np.random.default_rng(seed)
    n, d = x.shape
    means = np.ascontiguousarray(x[rng.choice(n, size=k, replace=False)].T)
    if k > 1:
        means[:, k - 1] = x.mean(axis=0) + 0.75
    covs = np.stack([random_covariance(rng, d) for _ in range(k)])
    w = rng.dirichlet(np.full(k, 2.0))
    if k > 2:
        w[k // 2] = 0.0
        w *= (1.0 - 1e-6) / w.sum()
        w[k // 2] = 1e-6
    return means, covs, w


@functools.lru_cache(maxsize=2)
def em_problem(d, k, n):
    """Data, chosen parameters and the reference's answers for one shape (shared by the chunk sizes and paths)."""
    seed = 1000 * d + k
    x, q = em_data(n, d, seed)
    means, covs, w = em_params(x, k, seed + 1)
    step = ref.em_step(x, means, covs, w)
    rng = np.random.default_rng(seed + 2)
    soft = rng.dirichlet(np.full(k, 0.5), size=n)
    hard = rng.permutation(np.arange(n) % k).astype(np.uint32)
    onehot = np.zeros((n, k))
    onehot[np.arange(n), hard] = 1.0
    _, q_resp, _ = ref.responsibilities(q, means, covs, w)
    return {
        "x": x, "q": q, "params": (means, covs, w), "step": step, "q_resp": q_resp,
        "soft": soft, "soft_m": ref.em_mstep(x, soft), "hard": hard, "hard_m": ref.em_mstep(x, onehot),
        "sample_cov": ref.sample_covariance(x), "kappa": ref.kappa(x, means, covs),
    }


def check_params(em, want, label, errs, collapsed=None, centre=None):
    """`collapsed`: components whose responsibilities sit on fewer points than dimensions.  The feature-space M-step
    forms their covariance as S2 / N_k - (mu - c)(mu - c)^T about the data mean c, so it is accurate to u |mu - c|^2
    absolute, not relative to its own (tiny) entries: for them the error is measured against max(|Sigma|, |mu - c|^2)
    and reported separately (DESIGN §2, finding of this matrix)."""
    means, covs, w = em.get_params()
    errs[label + ".means"] = rel_err(means, want[0])
    errs[label + ".weights"] = rel_err(w, want[2])
    if collapsed is None or not np.any(collapsed):
        errs[label + ".covs"] = cov_err(covs, want[1])
        return
    ok = [c for c in range(len(covs)) if not collapsed[c]]
    errs[label + ".covs"] = cov_err(covs[ok], want[1][ok]) if ok else 0.0
    errs[label + ".covs_collapsed"] = max(
        float(np.max(np.abs(covs[c] - want[1][c])) / max(np.max(np.abs(want[1][c])), float(np.sum((want[0][:, c] - centre) ** 2))))
        for c in np.flatnonzero(collapsed))


def run_em_case(ctx, monkeypatch, d, k, n, chunk, force, expected, env=None):
    from ml_b200 import cabi
    pb = em_problem(d, k, n)
    monkeypatch.setenv("MLB200_CHUNK", str(chunk))     # read by Layout::make inside the upload
    for key, val in (env or {}).items():
        monkeypatch.setenv(key, val)
    dev = cabi.Data.upload(ctx, pb["x"])
    em = cabi.Em(dev, k)
    try:
        cfg = em.kernel_config()
        assert tuple(cfg[f] for f in cabi.EM_CONFIG_FIELDS) == expected, cfg
        if force:
            em.force_path(3)
        means, covs, w = pb["params"]
        em.set_params(means, covs, w)
        kap, next_path = em.conditioning()
        errs = {"kappa": abs(kap - pb["kappa"]) / pb["kappa"]}
        want_path = 3 if (force or expected[0] == 0 or pb["kappa"] > 3e5) else expected[0]
        assert next_path == want_path
        st = pb["step"]
        ll = em.step()
        assert em.last_path == want_path
        errs["ll"] = abs(ll - st["log_likelihood"]) / abs(st["log_likelihood"])
        r = st["responsibilities"]
        collapsed = None
        if want_path != 3:
            collapsed = r.sum(axis=0) ** 2 < d * np.maximum((r ** 2).sum(axis=0), 1e-300)
        check_params(em, (st["means"], st["covariances"], st["weights"]), "step", errs, collapsed, pb["x"].mean(axis=0))
        resp, labels = em.emit()
        errs["emit.resp"] = float(np.max(np.abs(resp - st["responsibilities"])))
        clear = st["top2_gap"] > 1e-12
        assert np.array_equal(labels[clear], st["labels"][clear])
        em.set_params(means, covs, w)
        p_resp, p_labels = em.predict(pb["q"])
        errs["predict.resp"] = float(np.max(np.abs(p_resp - pb["q_resp"])))
        top2 = np.sort(pb["q_resp"], axis=1)[:, -2:] if k > 1 else None
        p_clear = (top2[:, 1] - top2[:, 0] > 1e-12) if k > 1 else np.ones(len(p_labels), dtype=bool)
        assert np.array_equal(p_labels[p_clear], np.argmax(pb["q_resp"], axis=1)[p_clear])
        em.mstep_from_responsibilities(pb["soft"])
        check_params(em, pb["soft_m"], "mstep_soft", errs)
        em.mstep_from_labels(pb["hard"])
        check_params(em, pb["hard_m"], "mstep_labels", errs)
        errs["sample_cov"] = rel_err(em.sample_covariance(), pb["sample_cov"])
    finally:
        em.close()
        dev.close()
    print(f"\n[em D={d} K={k} N={n} chunk={chunk} path={want_path}] " + " ".join(f"{key}={v:.1e}" for key, v in errs.items()))
    bars = {"kappa": 1e-9, "emit.resp": RESP_BAR, "predict.resp": RESP_BAR, "sample_cov": 1e-12}
    bad = {key: v for key, v in errs.items() if not v <= bars.get(key, BAR)}
    assert not bad, bad
    return errs


@pytest.mark.parametrize("d,k,n,chunk,force,expected", EM_CASES, ids=[_em_id(c) for c in EM_CASES])
def test_em_one_step(ctx, monkeypatch, d, k, n, chunk, force, expected):
    run_em_case(ctx, monkeypatch, d, k, n, chunk, force, expected)


# ---------------------------------------------------------------- kappa at the routing threshold (DESIGN §4.8)

def kappa_problem(target, n=N_A, d=8, k=4, seed=77):
    """95 % of the points in a unit blob at the origin, 5 % in a tight cluster 10 away, whose component is given the
    covariance s^2 I that puts its kappa exactly at `target`."""
    rng = np.random.default_rng(seed)
    m = n // 20
    far = np.zeros(d)
    far[0] = 10.0
    x = rng.standard_normal((n, d))
    x[:m] = far + 0.02 * rng.standard_normal((m, d))
    x = np.ascontiguousarray(x[rng.permutation(n)])
    means = np.ascontiguousarray(x[rng.choice(n, size=k, replace=False)].T)
    means[:, 0] = far
    covs = np.stack([random_covariance(rng, d, cond=10.0) for _ in range(k)])
    c = x.mean(axis=0)
    covs[0] = np.eye(d) * (float((far - c) @ (far - c)) / target)
    w = np.array([0.05, 0.45, 0.3, 0.2])
    return x, (means, covs, w)


@pytest.mark.parametrize("target,want_path", [(2.9e5, 1), (3.1e5, 3)])
def test_em_kappa_at_routing_threshold(ctx, target, want_path):
    from ml_b200 import cabi
    x, (means, covs, w) = kappa_problem(target)
    assert abs(ref.kappa(x, means, covs) / target - 1) < 1e-12
    st = ref.em_step(x, means, covs, w)
    dev = cabi.Data.upload(ctx, x)
    em = cabi.Em(dev, 4)
    try:
        em.set_params(means, covs, w)
        kap, next_path = em.conditioning()
        assert abs(kap / target - 1) <= 1e-9 and next_path == want_path
        ll = em.step()
        assert em.last_path == want_path
        errs = {"ll": abs(ll - st["log_likelihood"]) / abs(st["log_likelihood"])}
        check_params(em, (st["means"], st["covariances"], st["weights"]), "step", errs)
        resp, _ = em.emit()
        errs["emit.resp"] = float(np.max(np.abs(resp - st["responsibilities"])))
    finally:
        em.close()
        dev.close()
    print(f"\n[em kappa={target:.1e} path={want_path}] " + " ".join(f"{key}={v:.1e}" for key, v in errs.items()))
    # DESIGN §4.8 expected 1.5e-11 at the threshold; the tight component's covariance measures 1.0e-10 at kappa = 2.9e5
    # on the feature path (the rest of the step within 3e-14), so the bar is 2e-10 there: still 5x inside 1e-9.
    assert max(errs.values()) <= (2e-10 if want_path != 3 else 1e-10), errs


# ---------------------------------------------------------------- duplicate components

@pytest.mark.parametrize("d,k,n,force", [(8, 16, N_B, 0), (5, 32, N_B, 0), (20, 24, N_B, 0), (8, 40, N_B, 0), (8, 16, N_B, 3)])
def test_em_duplicate_components_tie_to_lower_index(ctx, d, k, n, force):
    """Components (0, KP - 1) and (7, 8) identical: their responsibility columns are bitwise equal, and no label is
    the higher index of a pair (first maximum wins, EM.cpp:289-304)."""
    from ml_b200 import cabi
    x, q = em_data(n, d, 5 + d)
    means, covs, w = em_params(x, k, 6 + d)
    kp = {16: 16, 32: 32, 24: 32, 40: 64}[k]
    hi = min(kp, k) - 1
    pairs = [(0, hi), (7, 8)]
    for a, b in pairs:
        means[:, b], covs[b], w[b] = means[:, a], covs[a], w[a]
    # give the duplicated components most of the data, so that they are the maximum of many rows
    w[[0, hi, 7, 8]] *= 50.0
    w /= w.sum()
    dev = cabi.Data.upload(ctx, x)
    em = cabi.Em(dev, k)
    try:
        if force:
            em.force_path(3)
        em.set_params(means, covs, w)
        em.step()
        resp, labels = em.emit()
        em.set_params(means, covs, w)
        p_resp, p_labels = em.predict(q)
    finally:
        em.close()
        dev.close()
    for a, b in pairs:
        assert np.array_equal(resp[:, a], resp[:, b]) and np.array_equal(p_resp[:, a], p_resp[:, b]), (a, b)
        assert not np.any(labels == b) and not np.any(p_labels == b), (a, b)
        assert np.any(labels == a)


# ---------------------------------------------------------------- K-means

def km_centroids(x, k, seed):
    """K - 1 centroids at data points and one far outside the data, which no point reaches (its cluster empties and
    goes to the origin on the update)."""
    rng = np.random.default_rng(seed)
    c = np.ascontiguousarray(x[rng.choice(x.shape[0], size=k, replace=False)].T)
    c[:, k // 3] = 1e3
    return c


@functools.lru_cache(maxsize=2)
def km_problem(d, k, n):
    seed = 2000 * d + k
    x, q = em_data(n, d, seed)
    c0 = km_centroids(x, k, seed + 1)
    return x, q, c0, ref.km_step(x, c0, np.zeros(n, dtype=np.uint32))


def check_predict(km, centroids, q, label):
    """Labels and squared distances of Km.predict (the COMPACT kernel) bitwise those of the reference's scan with the
    device's fused distance chain, on a sample of 1000 points plus every point the float64 reference calls a near-tie."""
    labels, dist = km.predict(q)
    want_l, want_d = oracle.kmeans_assign_fused(centroids, q)
    assert np.array_equal(labels, want_l), label
    _, _, ties = ref.km_assign(q, centroids)
    sample = np.union1d(np.arange(min(1000, len(q))), ties)
    assert np.array_equal(dist[sample], want_d[sample]), label
    # and within 1e-13 of the reference's own unfused sum (oracle.kmeans_assign_label) on a few points
    for i in sample[:50]:
        lab, sq = oracle.kmeans_assign_label(centroids, q[i])
        assert lab == labels[i] and abs(dist[i] - sq) <= 1e-13 * sq
    return len(ties)


@pytest.mark.parametrize("d,k,n,chunk,env,expected", KM_CASES, ids=[_km_id(c) for c in KM_CASES])
def test_kmeans_one_step(ctx, monkeypatch, d, k, n, chunk, env, expected):
    from ml_b200 import cabi
    x, q, c0, st = km_problem(d, k, n)
    monkeypatch.setenv("MLB200_CHUNK", str(chunk))
    for key, val in env.items():
        monkeypatch.setenv(key, val)
    dev = cabi.Data.upload(ctx, x)
    km = cabi.Km(dev, k)
    errs = {}
    try:
        cfg = km.kernel_config()
        assert tuple(cfg[f] for f in cabi.KM_CONFIG_FIELDS) == expected, cfg
        km.set_centroids(c0)
        inertia, changed = km.assign()
        labels = km.get_labels()
        assert np.array_equal(labels, st["labels"])
        assert changed == st["changed"]
        errs["inertia"] = abs(inertia - st["inertia"]) / st["inertia"]
        shift = km.update()
        c1 = km.get_centroids()
        assert st["counts"][k // 3] == 0 and np.all(c1[:, k // 3] == 0.0)
        errs["centroids"] = rel_err(c1, st["centroids"])
        errs["shift"] = abs(shift - st["shift"]) / st["shift"]
        # the second assignment from the device's own centroids: the changed count against the first labels
        st2 = ref.km_step(x, c1, labels)
        inertia2, changed2 = km.assign()
        assert np.array_equal(km.get_labels(), st2["labels"])
        assert changed2 == st2["changed"]
        errs["inertia2"] = abs(inertia2 - st2["inertia"]) / st2["inertia"]
        ties = check_predict(km, c1, q, "predict")
    finally:
        km.close()
        dev.close()
    print(f"\n[km D={d} K={k} N={n} chunk={chunk} {env}] ties={ties} " + " ".join(f"{key}={v:.1e}" for key, v in errs.items()))
    bad = {key: v for key, v in errs.items() if not v <= (1e-12 if key == "shift" else KM_BAR)}
    assert not bad, bad


@pytest.mark.parametrize("chunk", [128, 2048])
def test_kmeans_two_sets(ctx, monkeypatch, chunk):
    """Two K-means starts in lockstep (mlb_kms): per set, what one Km pass gives."""
    from ml_b200 import cabi
    d, k, n = 16, 40, N_B
    monkeypatch.setenv("MLB200_CHUNK", str(chunk))
    x, q = em_data(n, d, 99)
    starts = [km_centroids(x, k, 100), km_centroids(x, k, 101)]
    steps = [ref.km_step(x, c, np.zeros(n, dtype=np.uint32)) for c in starts]
    dev = cabi.Data.upload(ctx, x)
    assert cabi.Kms.supported(dev, k, 2)
    kms = cabi.Kms(dev, k, 2)
    try:
        for s, c in enumerate(starts):
            kms.set_centroids(s, c)
        inertia, changed = kms.assign()
        shift = kms.update()
        for s, st in enumerate(steps):
            assert np.array_equal(kms.get_labels(s), st["labels"]) and changed[s] == st["changed"]
            assert abs(inertia[s] - st["inertia"]) <= KM_BAR * st["inertia"]
            assert rel_err(kms.get_centroids(s), st["centroids"]) <= KM_BAR
            assert abs(shift[s] - st["shift"]) <= 1e-12 * st["shift"]
    finally:
        kms.close()
        dev.close()
