"""Host <-> device copies of the C-ABI with pageable and strided host memory: large copies are cut into pieces that
several host threads pack through pinned bounce buffers (ml_b200/csrc/context.cu, staged_h2d / staged_d2h); the
reference passes Eigen::Ref matrices, whose outer stride may exceed the row count (EM.cpp:91, KMeans.cpp:25)."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cabi():
    from ml_b200 import cabi as module
    assert module.device_count() >= 1
    return module


@pytest.fixture(scope="module")
def ctx(cabi):
    c = cabi.Context(1)
    yield c
    c.close()


def _upload_strided(cabi, ctx, padded, n, d):
    h = ctypes.c_void_p()
    cabi.check(cabi.lib().mlb_data_upload(ctx._h, padded.ctypes.data_as(ctypes.c_void_p), n, n, d, padded.shape[1], ctypes.byref(h)))
    return cabi.Data(ctx, h)


@pytest.mark.parametrize("n,d,pad", [(1000, 3, 2), (700_001, 5, 3), (3_000_001, 2, 1), (2_500_000, 8, 0), (1_300_000, 7, 9)])
def test_upload_round_trip_contiguous_and_strided(cabi, ctx, n, d, pad):
    """Outer stride ld = d + pad: every size class (direct small copy, one thread, several threads) returns the points."""
    rng = np.random.default_rng(n + d)
    padded = np.ascontiguousarray(rng.normal(size=(n, d + pad)))
    points = np.ascontiguousarray(padded[:, :d])
    dev = _upload_strided(cabi, ctx, padded, n, d)
    assert np.array_equal(dev.download(0, n), points)
    assert np.array_equal(dev.download(n // 3, n // 2), points[n // 3: n // 3 + n // 2])
    dev.close()


def test_strided_responsibilities_and_queries(cabi, ctx):
    """mlb_em_mstep_from_responsibilities with ld > n (rows of n doubles, 6.4 MB in all) and mlb_em_predict /
    mlb_km_predict with ld_x > d give what the dense calls give."""
    from tests.datasets import synthetic_gmm
    n, d, k = 200_000, 4, 4
    data, labels, _ = synthetic_gmm(n, d, k, seed=4, spread=6.0)
    dev = cabi.Data.upload(ctx, data)
    resp = np.zeros((n, k), order="F")
    resp[np.arange(n), labels] = 0.75
    resp[np.arange(n), (labels + 1) % k] = 0.25
    dense = cabi.Em(dev, k)
    dense.mstep_from_responsibilities(resp)
    wide = np.zeros((n + 13, k), order="F")
    wide[:n] = resp
    strided = cabi.Em(dev, k)
    cabi.check(cabi.lib().mlb_em_mstep_from_responsibilities(strided._h, wide.ctypes.data_as(ctypes.c_void_p), n + 13))
    for a, b in zip(dense.get_params(), strided.get_params()):
        assert np.array_equal(a, b)

    m = 300_000
    queries = np.ascontiguousarray(np.random.default_rng(8).normal(size=(m, d + 3)) * 5.0)
    q_dense = np.ascontiguousarray(queries[:, :d])
    want_resp, want_labels = dense.predict(q_dense)
    got_resp = np.empty((m, k), order="F")
    got_labels = np.empty(m, dtype=np.uint32)
    cabi.check(cabi.lib().mlb_em_predict(dense._h, queries.ctypes.data_as(ctypes.c_void_p), m, d + 3, got_resp.ctypes.data_as(ctypes.c_void_p), m,
                                        got_labels.ctypes.data_as(ctypes.c_void_p)))
    assert np.array_equal(got_resp, want_resp) and np.array_equal(got_labels, want_labels)

    km = cabi.Km(dev, k)
    km.set_centroids(data[:k].T)
    want_l, want_d = km.predict(q_dense)
    got_l, got_d = np.empty(m, dtype=np.uint32), np.empty(m)
    cabi.check(cabi.lib().mlb_km_predict(km._h, queries.ctypes.data_as(ctypes.c_void_p), m, d + 3, got_l.ctypes.data_as(ctypes.c_void_p),
                                        got_d.ctypes.data_as(ctypes.c_void_p)))
    assert np.array_equal(got_l, want_l) and np.array_equal(got_d, want_d)
    km.close(), dense.close(), strided.close(), dev.close()


def test_pinned_host_memory_takes_the_direct_path(cabi, ctx):
    """Pinned buffers (what bench.py's end-to-end leg uses) round-trip as well."""
    import torch
    n, d = 1_500_000, 6
    host = torch.empty((n, d), dtype=torch.float64, pin_memory=True)
    view = host.numpy()
    view[:] = np.random.default_rng(2).normal(size=(n, d))
    dev = cabi.Data.upload(ctx, view)
    out = torch.empty((n, d), dtype=torch.float64, pin_memory=True)
    cabi.check(cabi.lib().mlb_data_download(dev._h, 0, n, ctypes.c_void_p(out.data_ptr())))
    assert np.array_equal(out.numpy(), view)
    dev.close()


@pytest.mark.parametrize("n,d,offset", [(3_000_000, 8, 0), (2_500_001, 16, 3), (1_100_000, 5, 1)])
def test_upload_round_trip_from_unaligned_start(cabi, ctx, n, d, offset):
    """Large contiguous pageable uploads through the bounce buffers: the points come back bit for bit, also from a buffer
    that does not start on a page boundary, and again on a second upload that reuses the bounce buffers."""
    rng = np.random.default_rng(n)
    backing = rng.normal(size=n * d + 8)
    points = backing[offset: offset + n * d].reshape(n, d)       # 8 * offset bytes into the allocation
    for _ in range(2):
        dev = cabi.Data.upload(ctx, points)
        assert np.array_equal(dev.download(0, n), points)
        dev.close()
    dev = cabi.Data.upload(ctx, points)
    assert np.array_equal(dev.download(n - 1000, 1000), points[-1000:])
    dev.close()
