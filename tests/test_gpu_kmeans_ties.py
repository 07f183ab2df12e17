"""Near-ties in the K-means assignment: points placed so that the filter's ambiguity bound decides.

The DMMA filter of km_assign_kernel scores every centroid with an expanded quadratic form and keeps a label only when
`second_lo > best_hi + tau`, tau = 8 (d + 4) u (|z| + cmax)^2 (kmeans.cu); every other point goes to the exact scan.  A
bound that is too small silently changes labels near a bisector.  For a centroid pair (a, b) the points are
m + t f + s e: m the pair's midpoint, e the unit vector from a to b, f perpendicular to e, s in {0, +-1, +-2, +-8, +-64}
ulp of |m| and +-1e-12, +-1e-9 times the gap.  Two scales: the pair 1e-3 apart among centroids spread over 1e3 (|z| and
cmax large against the gap), and the pair 1e3 apart with everything else within 1e-3 of the origin.  Pairs at (0, 1)
(one n-tile), (6, 9) (two n-tiles), (31, 32) (two 32-groups), (K - 2, K - 1) next to the padding, (31, 32) across a
centroid block (MLB200_KM_BLOCK=32: km_combine_kernel's strict < decides), a three-way tie and duplicates at (3, 40).

Every label, through the fit's assignment, Km.predict (the COMPACT kernel) and a two-set Kms, and every predicted
squared distance must be bitwise those of the reference's scan (strict <, lowest index) evaluated with the device's
fused distance chain (oracle.kmeans_assign_fused)."""
import numpy as np
import pytest

import oracle

pytestmark = pytest.mark.gpu

K = 45
DIMS = [1, 3, 4, 7, 8, 16, 31, 32, 64, 65, 100]
PLACEMENTS = ["tile", "ntiles", "groups", "padding", "block", "three", "duplicate"]
SCALES = ["small_gap", "large_gap"]


@pytest.fixture(scope="module")
def ctx():
    from ml_b200 import cabi
    assert cabi.device_count() >= 1, "no CUDA device: the product has no CPU fallback"
    c = cabi.Context(1)
    yield c
    c.close()


def _unit(v):
    return v / np.linalg.norm(v)


def tie_problem(d, placement, scale, seed):
    """(centroids (D, K), points (N, D)) for one scenario."""
    rng = np.random.default_rng(seed)
    spread, gap = (1e3, 1e-3) if scale == "small_gap" else (1e-3, 1e3)
    c = rng.uniform(-spread, spread, size=(K, d))
    centre = rng.uniform(-spread, spread, size=d)
    pair = {"tile": (0, 1), "ntiles": (6, 9), "groups": (31, 32), "padding": (K - 2, K - 1), "block": (31, 32),
            "three": (10, 20), "duplicate": (3, 40)}[placement]
    e = _unit(rng.standard_normal(d))
    a, b = pair
    c[a] = centre - 0.5 * gap * e
    c[b] = centre + 0.5 * gap * e
    if placement == "duplicate":
        c[b] = c[a]
    m = 0.5 * (c[a] + c[b])
    if placement == "three" and d >= 2:
        # a third centroid at the same distance from m as a and b
        f = _unit(rng.standard_normal(d) - (rng.standard_normal(d) @ e) * e)
        f = _unit(f - (f @ e) * e)
        c[30] = m + 0.5 * gap * f
    ulp = np.spacing(np.linalg.norm(m))
    offsets = [0.0] + [sg * v for v in (ulp, 2 * ulp, 8 * ulp, 64 * ulp, 1e-12 * gap, 1e-9 * gap) for sg in (1.0, -1.0)]
    ts = [0.0] if d == 1 else [0.0, 0.3 * gap, 3.0 * gap]
    pts = []
    for t in ts:
        f = np.zeros(d) if d == 1 else _unit((lambda r: r - (r @ e) * e)(rng.standard_normal(d)))
        for s in offsets:
            pts.append(m + t * f + s * e)
            if placement == "duplicate":
                pts.append(c[a] + t * f + s * e)
    pts = np.array(pts)
    # some ordinary points around the centroids so that the fit's chunks hold more than the ties
    filler = c[rng.integers(0, K, size=600)] + rng.standard_normal((600, d)) * (0.1 * gap)
    x = np.concatenate([pts, filler, pts])
    return np.ascontiguousarray(c.T), np.ascontiguousarray(x), len(pts)


@pytest.mark.parametrize("scale", SCALES)
@pytest.mark.parametrize("placement", PLACEMENTS)
@pytest.mark.parametrize("d", DIMS)
def test_kmeans_near_ties_match_the_scan(ctx, monkeypatch, d, placement, scale):
    from ml_b200 import cabi
    if placement == "block":
        monkeypatch.setenv("MLB200_KM_BLOCK", "32")
    seed = 100 * d + 10 * PLACEMENTS.index(placement) + SCALES.index(scale)
    cent, x, _ = tie_problem(d, placement, scale, seed)
    want_l, want_d = oracle.kmeans_assign_fused(cent, x)
    dev = cabi.Data.upload(ctx, x)
    km = cabi.Km(dev, K)
    try:
        cfg = km.kernel_config()
        assert (cfg["nblocks"] > 1) == (placement == "block")
        km.set_centroids(cent)
        km.assign()
        fit_l = km.get_labels()
        pred_l, pred_d = km.predict(x)
    finally:
        km.close()
        dev.close()
    bad_fit = np.flatnonzero(fit_l != want_l)
    bad_pred = np.flatnonzero((pred_l != want_l) | (pred_d != want_d))
    assert bad_fit.size == 0, (bad_fit[:10], fit_l[bad_fit[:10]], want_l[bad_fit[:10]])
    assert bad_pred.size == 0, (bad_pred[:10], pred_l[bad_pred[:10]], want_l[bad_pred[:10]])
    if placement == "duplicate":
        assert not np.any(fit_l == 40)


@pytest.mark.parametrize("d", [3, 16, 64])
def test_kmeans_near_ties_two_sets(ctx, d):
    """The same points through a two-set Kms: each set's labels those of the scan."""
    from ml_b200 import cabi
    c0, x, _ = tie_problem(d, "groups", "small_gap", 7 * d)
    c1, x1, _ = tie_problem(d, "ntiles", "small_gap", 7 * d)
    x = np.ascontiguousarray(np.concatenate([x, x1]))
    dev = cabi.Data.upload(ctx, x)
    assert cabi.Kms.supported(dev, K, 2)
    kms = cabi.Kms(dev, K, 2)
    try:
        kms.set_centroids(0, c0)
        kms.set_centroids(1, c1)
        kms.assign()
        for s, c in enumerate((c0, c1)):
            assert np.array_equal(kms.get_labels(s), oracle.kmeans_assign_fused(c, x)[0]), s
    finally:
        kms.close()
        dev.close()
