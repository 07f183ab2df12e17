"""CPU-side checks of the K-means distance and inertia entry points (no GPU needed): null handles and bad arguments are
MLB_EINVAL before any device work, a machine without a device fails loudly, and the cppyml methods exist with the
error behaviour of assign_labels."""
import ctypes

import numpy as np
import pytest


@pytest.fixture(scope="module", autouse=True)
def built():
    import __graft_entry__
    __graft_entry__.build()


def test_null_handles_are_rejected():
    from ml_b200 import cabi
    lib = cabi.lib()
    x = np.zeros((4, 3))
    out = np.zeros((4, 2))
    inertia = ctypes.c_double()
    p_x, p_out = x.ctypes.data_as(ctypes.c_void_p), out.ctypes.data_as(ctypes.c_void_p)
    assert lib.mlb_km_transform(None, p_x, 4, 3, 0, p_out, 4) == cabi.MLB_EINVAL
    assert b"mlb_km_transform" in lib.mlb_last_error()
    assert lib.mlb_km_transform_range(None, 0, 4, 1, p_out, 4) == cabi.MLB_EINVAL
    assert b"mlb_km_transform_range" in lib.mlb_last_error()
    assert lib.mlb_km_score(None, p_x, 4, 3, None, ctypes.byref(inertia)) == cabi.MLB_EINVAL
    assert b"mlb_km_score" in lib.mlb_last_error()
    assert lib.mlb_km_score_fitted(None, ctypes.byref(inertia)) == cabi.MLB_EINVAL
    assert b"mlb_km_score_fitted" in lib.mlb_last_error()
    # null outputs and bad shapes, with a null model as well: rejected before anything reaches a device
    assert lib.mlb_km_transform(None, p_x, 4, 3, 0, None, 4) == cabi.MLB_EINVAL
    assert lib.mlb_km_transform(None, p_x, -1, 3, 0, p_out, 4) == cabi.MLB_EINVAL
    assert lib.mlb_km_transform_range(None, -1, 4, 0, p_out, 4) == cabi.MLB_EINVAL
    assert lib.mlb_km_score(None, p_x, 4, 3, None, None) == cabi.MLB_EINVAL
    assert lib.mlb_km_score_fitted(None, None) == cabi.MLB_EINVAL


def test_no_device_means_a_loud_failure():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from ml_b200 import cabi
    with pytest.raises(cabi.MlbError) as err:
        cabi.Context(1)
    assert err.value.code == cabi.MLB_ECUDA
    km = __import__("ml_b200").import_cppyml().clustering.KMeans(2)
    with pytest.raises(RuntimeError):
        km.fit(np.random.default_rng(0).normal(size=(50, 2)))
    with pytest.raises(RuntimeError):
        km.transform()


def test_cppyml_methods_and_errors_without_device_state():
    c = __import__("ml_b200").import_cppyml().clustering
    km = c.KMeans(3)
    assert callable(km.transform) and callable(km.score)
    assert "sklearn" in km.transform.__doc__ and "sklearn" in km.score.__doc__
    x = np.array([[0.5, 0.1], [0.3, 0.2], [0.1, -0.4]])
    assert km.fit(x) is True            # N == K: the exact fit, nothing is resident
    assert km.inertia == 0.0
    for call in (km.transform, km.score):
        with pytest.raises(ValueError):
            call(np.zeros((4, 5)))      # wrong D
        with pytest.raises(TypeError):
            call(np.zeros((4, 2), dtype=np.float32))
        with pytest.raises(TypeError):
            call(np.asfortranarray(np.zeros((4, 2))))
        with pytest.raises(RuntimeError):
            call(np.zeros((4, 2)))      # no fitted device state, as assign_labels
        with pytest.raises(RuntimeError):
            call()
    with pytest.raises(RuntimeError):
        km.assign_labels(np.zeros((4, 2)))
