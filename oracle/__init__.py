"""ctypes loader for the CPU oracle (TEST INFRASTRUCTURE ONLY).

`oracle/mlpp_oracle.cpp` restates the reference's clustering hot path on the CPU.  Only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s `cpu_baseline` / `--impl reference` legs may import this
module; the product (`ml_b200/`) never does.

All matrices follow the reference's convention: column-major D x N data (a point per column), which
is the same memory as a C-contiguous numpy array of shape (N, D).
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libmlpp_oracle.so")
# The reference's own translation units compiled against the Eigen stand-in (oracle/Makefile target `ref`); built in the
# builder container where /root/reference is mounted, then shipped as a prebuilt file.
_REF_LIB_PATH = os.path.join(_HERE, "_ref", "libmlpp_ref.so")

FORGY, RANDOM_PARTITION, KPP, EXPLICIT = 0, 1, 2, 3

_dp = ctypes.POINTER(ctypes.c_double)
_up = ctypes.POINTER(ctypes.c_uint)


class _EmOptions(ctypes.Structure):
    _fields_ = [
        ("seed", ctypes.c_uint),
        ("set_seed", ctypes.c_int),
        ("absolute_tolerance", ctypes.c_double),
        ("relative_tolerance", ctypes.c_double),
        ("maximum_steps", ctypes.c_uint),
        ("means_init_kind", ctypes.c_int),
        ("resp_init_centroid_kind", ctypes.c_int),
        ("maximise_first", ctypes.c_int),
        ("explicit_means", _dp),
    ]


class _EmResult(ctypes.Structure):
    _fields_ = [
        ("means", _dp),
        ("covariances", _dp),
        ("mixing_probabilities", _dp),
        ("responsibilities", _dp),
        ("labels", _up),
        ("inverse_covariances", _dp),
        ("sqrt_covariance_determinants", _dp),
        ("step_seconds", _dp),
        ("log_likelihood", ctypes.c_double),
        ("converged", ctypes.c_int),
        ("iterations", ctypes.c_uint),
    ]


class _KmOptions(ctypes.Structure):
    _fields_ = [
        ("seed", ctypes.c_uint),
        ("set_seed", ctypes.c_int),
        ("absolute_tolerance", ctypes.c_double),
        ("maximum_steps", ctypes.c_uint),
        ("number_initialisations", ctypes.c_uint),
        ("init_kind", ctypes.c_int),
        ("explicit_means", _dp),
    ]


class _KmResult(ctypes.Structure):
    _fields_ = [
        ("centroids", _dp),
        ("labels", _up),
        ("step_seconds", _dp),
        ("inertia", ctypes.c_double),
        ("converged", ctypes.c_int),
        ("iterations", ctypes.c_uint),
    ]


def build(force=False):
    """Compiles the oracle with the recipe in oracle/Makefile."""
    src = os.path.join(_HERE, "mlpp_oracle.cpp")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-B", "libmlpp_oracle.so"], stdout=subprocess.DEVNULL)
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = ctypes.CDLL(_LIB_PATH)
        _lib.mlpp_oracle_em_fit.restype = ctypes.c_int
        _lib.mlpp_oracle_em_fit.argtypes = [_dp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_uint,
                                            ctypes.POINTER(_EmOptions), ctypes.POINTER(_EmResult)]
        _lib.mlpp_oracle_kmeans_fit.restype = ctypes.c_int
        _lib.mlpp_oracle_kmeans_fit.argtypes = [_dp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_uint,
                                                ctypes.POINTER(_KmOptions), ctypes.POINTER(_KmResult)]
        _lib.mlpp_oracle_em_assign_responsibilities.restype = None
        _lib.mlpp_oracle_em_assign_responsibilities.argtypes = [_dp, ctypes.c_int64, ctypes.c_uint, _dp, _dp, _dp, _dp, _dp]
        _lib.mlpp_oracle_kmeans_assign_label.restype = ctypes.c_uint
        _lib.mlpp_oracle_kmeans_assign_label.argtypes = [_dp, ctypes.c_int64, ctypes.c_uint, _dp, _dp]
        _lib.mlpp_oracle_kmeans_assign_fused.restype = None
        _lib.mlpp_oracle_kmeans_assign_fused.argtypes = [_dp, ctypes.c_int64, ctypes.c_int64, ctypes.c_uint, _dp, _up, _dp]
        _lib.mlpp_oracle_centroids_init.restype = None
        _lib.mlpp_oracle_centroids_init.argtypes = [ctypes.c_int, _dp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64,
                                                    ctypes.c_uint, ctypes.c_uint, ctypes.c_int, _dp]
        _lib.mlpp_oracle_xAx_symmetric.restype = ctypes.c_double
        _lib.mlpp_oracle_xAx_symmetric.argtypes = [_dp, ctypes.c_int64, _dp]
        _lib.mlpp_oracle_xxT.restype = None
        _lib.mlpp_oracle_xxT.argtypes = [_dp, ctypes.c_int64, _dp]
        _lib.mlpp_oracle_add_a_xxT.restype = None
        _lib.mlpp_oracle_add_a_xxT.argtypes = [_dp, ctypes.c_int64, _dp, ctypes.c_double]
        _lib.mlpp_oracle_testdata_two_gaussians.restype = None
        _lib.mlpp_oracle_testdata_two_gaussians.argtypes = [_dp, _up]
        _lib.mlpp_oracle_testdata_mouse.restype = None
        _lib.mlpp_oracle_testdata_mouse.argtypes = [_dp, _up, ctypes.c_uint]
    return _lib


_ref = None


def ref_available():
    """True when oracle/_ref/libmlpp_ref.so (the reference's own sources, see oracle/Makefile) exists."""
    return os.path.exists(_REF_LIB_PATH)


def ref_lib():
    global _ref
    if _ref is None:
        if not ref_available():
            raise RuntimeError("oracle/_ref/libmlpp_ref.so is not built (run `make -C oracle ref` where /root/reference is mounted)")
        _ref = ctypes.CDLL(_REF_LIB_PATH)
        _ref.mlpp_ref_em_fit.restype = ctypes.c_int
        _ref.mlpp_ref_em_fit.argtypes = [_dp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_uint, ctypes.POINTER(_EmOptions),
                                         ctypes.POINTER(_EmResult), ctypes.c_int, _dp, ctypes.c_int64, _dp]
        _ref.mlpp_ref_kmeans_fit.restype = ctypes.c_int
        _ref.mlpp_ref_kmeans_fit.argtypes = [_dp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_uint, ctypes.POINTER(_KmOptions),
                                             ctypes.POINTER(_KmResult), ctypes.c_int, _dp, ctypes.c_int64, _up, _dp]
        _ref.mlpp_ref_centroids_init.restype = None
        _ref.mlpp_ref_centroids_init.argtypes = [ctypes.c_int, _dp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_uint,
                                                 ctypes.c_uint, ctypes.c_int, _dp]
        _ref.mlpp_ref_xAx_symmetric.restype = ctypes.c_double
        _ref.mlpp_ref_xAx_symmetric.argtypes = [_dp, ctypes.c_int64, _dp]
        _ref.mlpp_ref_xxT.restype = None
        _ref.mlpp_ref_xxT.argtypes = [_dp, ctypes.c_int64, _dp]
        _ref.mlpp_ref_add_a_xxT.restype = None
        _ref.mlpp_ref_add_a_xxT.argtypes = [_dp, ctypes.c_int64, _dp, ctypes.c_double]
    return _ref


def _ptr(a):
    return a.ctypes.data_as(_dp)


def _check_data(data):
    data = np.ascontiguousarray(data, dtype=np.float64)
    if data.ndim != 2:
        raise ValueError("data must be (N, D)")
    return data


class EmFit:
    """Result of `em_fit`.  `means` is (D, K) like ml::EM::means(); `covariances` is (K, D, D);
    `responsibilities` is (N, K)."""


def em_fit(data, k, *, seed=None, absolute_tolerance=1e-8, relative_tolerance=1e-8, maximum_steps=1000,
           means_init=FORGY, resp_init_centroids=FORGY, maximise_first=False, explicit_means=None,
           want_responsibilities=True, impl="oracle", count_iterations=True, queries=None):
    """ml::EM::fit (ML/EM.cpp:91-174) on `data` of shape (N, D), one point per row.

    impl="oracle" runs the restatement (mlpp_oracle.cpp); impl="reference" runs the reference's own ml::EM from
    oracle/_ref (no per-step clock: `fit_seconds` is the whole fit; no inverse covariances; `queries` (Q, D) are passed
    to EM::assign_responsibilities after the fit and come back as `query_responsibilities` (Q, K))."""
    data = _check_data(data)
    n, d = data.shape
    opt = _EmOptions()
    opt.seed = 0 if seed is None else int(seed)
    opt.set_seed = 0 if seed is None else 1
    opt.absolute_tolerance = absolute_tolerance
    opt.relative_tolerance = relative_tolerance
    opt.maximum_steps = maximum_steps
    opt.means_init_kind = means_init
    opt.resp_init_centroid_kind = resp_init_centroids
    opt.maximise_first = int(bool(maximise_first))
    em_means = None
    if explicit_means is not None:
        # (D, K) as ml::EM::means(): stored column-major, i.e. the memory of a C-contiguous (K, D) array.
        em_means = np.ascontiguousarray(np.asarray(explicit_means, dtype=np.float64).T)
        assert em_means.shape == (k, d)
        opt.explicit_means = _ptr(em_means)
    means = np.zeros((k, d))
    covs = np.zeros((k, d, d))
    inv = np.zeros((k, d, d))
    sqrt_det = np.zeros(k)
    mix = np.zeros(k)
    resp = np.zeros((k, n)) if want_responsibilities else None
    labels = np.zeros(n, dtype=np.uint32)
    step_seconds = np.full(maximum_steps, np.nan)
    res = _EmResult()
    res.means = _ptr(means)
    res.covariances = _ptr(covs)
    res.inverse_covariances = _ptr(inv)
    res.sqrt_covariance_determinants = _ptr(sqrt_det)
    res.mixing_probabilities = _ptr(mix)
    res.responsibilities = _ptr(resp) if resp is not None else None
    res.labels = labels.ctypes.data_as(_up)
    res.step_seconds = _ptr(step_seconds)
    query_out = None
    if impl == "reference":
        q = None if queries is None else np.ascontiguousarray(queries, dtype=np.float64)
        query_out = None if q is None else np.zeros((q.shape[0], k))
        rc = ref_lib().mlpp_ref_em_fit(_ptr(data), d, n, d, k, ctypes.byref(opt), ctypes.byref(res), int(bool(count_iterations)),
                                       None if q is None else _ptr(q), 0 if q is None else q.shape[0],
                                       None if q is None else _ptr(query_out))
    else:
        rc = lib().mlpp_oracle_em_fit(_ptr(data), d, n, d, k, ctypes.byref(opt), ctypes.byref(res))
    if rc != 0:
        raise ValueError("EM: invalid arguments")
    out = EmFit()
    out.query_responsibilities = query_out
    out.fit_seconds = float(step_seconds[0]) if impl == "reference" else float(np.nansum(step_seconds))
    out.means = means.T.copy()
    out.covariances = covs.transpose(0, 2, 1).copy()  # each block is column-major D x D (symmetric anyway)
    out.inverse_covariances = inv.transpose(0, 2, 1).copy()
    out.sqrt_covariance_determinants = sqrt_det
    out.mixing_probabilities = mix
    out.responsibilities = resp.T.copy() if resp is not None else None
    out.labels = labels
    out.log_likelihood = res.log_likelihood
    out.converged = bool(res.converged)
    out.iterations = int(res.iterations)
    out.step_seconds = step_seconds[: out.iterations] if impl != "reference" else None
    return out


def em_assign_responsibilities(fit, x):
    """EM::assign_responsibilities (ML/EM.cpp:176-188) with the post-fit parameters of `fit`."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    d, k = fit.means.shape
    means = np.ascontiguousarray(fit.means.T)
    inv = np.ascontiguousarray(fit.inverse_covariances.transpose(0, 2, 1))
    u = np.zeros(k)
    lib().mlpp_oracle_em_assign_responsibilities(_ptr(x), d, k, _ptr(means), _ptr(inv),
                                                 _ptr(np.ascontiguousarray(fit.mixing_probabilities)),
                                                 _ptr(np.ascontiguousarray(fit.sqrt_covariance_determinants)), _ptr(u))
    return u


class KMeansFit:
    """Result of `kmeans_fit`.  `centroids` is (D, K) like KMeans::centroids()."""


def kmeans_fit(data, k, *, seed=None, absolute_tolerance=1e-8, maximum_steps=1000, number_initialisations=1,
               init=FORGY, explicit_means=None, impl="oracle", count_iterations=True, queries=None):
    """ml::Clustering::KMeans::fit (ML/KMeans.cpp:25-114) on `data` of shape (N, D).  impl as in em_fit; with
    impl="reference" `queries` (Q, D) go to KMeans::assign_label and come back as `query_labels`, `query_distances`."""
    data = _check_data(data)
    n, d = data.shape
    opt = _KmOptions()
    opt.seed = 0 if seed is None else int(seed)
    opt.set_seed = 0 if seed is None else 1
    opt.absolute_tolerance = absolute_tolerance
    opt.maximum_steps = maximum_steps
    opt.number_initialisations = number_initialisations
    opt.init_kind = init
    km_means = None
    if explicit_means is not None:
        km_means = np.ascontiguousarray(np.asarray(explicit_means, dtype=np.float64).T)
        assert km_means.shape == (k, d)
        opt.explicit_means = _ptr(km_means)
    centroids = np.zeros((k, d))
    labels = np.zeros(n, dtype=np.uint32)
    step_seconds = np.full(maximum_steps, np.nan)
    res = _KmResult()
    res.centroids = _ptr(centroids)
    res.labels = labels.ctypes.data_as(_up)
    res.step_seconds = _ptr(step_seconds)
    q_labels = q_sq = None
    if impl == "reference":
        q = None if queries is None else np.ascontiguousarray(queries, dtype=np.float64)
        if q is not None:
            q_labels, q_sq = np.zeros(q.shape[0], dtype=np.uint32), np.zeros(q.shape[0])
        rc = ref_lib().mlpp_ref_kmeans_fit(_ptr(data), d, n, d, k, ctypes.byref(opt), ctypes.byref(res), int(bool(count_iterations)),
                                           None if q is None else _ptr(q), 0 if q is None else q.shape[0],
                                           None if q is None else q_labels.ctypes.data_as(_up), None if q is None else _ptr(q_sq))
    else:
        rc = lib().mlpp_oracle_kmeans_fit(_ptr(data), d, n, d, k, ctypes.byref(opt), ctypes.byref(res))
    if rc != 0:
        raise ValueError("KMeans: invalid arguments")
    out = KMeansFit()
    out.query_labels, out.query_distances = q_labels, q_sq
    out.fit_seconds = float(step_seconds[0]) if impl == "reference" else float(np.nansum(step_seconds))
    out.centroids = centroids.T.copy()
    out.labels = labels
    out.inertia = res.inertia
    out.converged = bool(res.converged)
    out.iterations = int(res.iterations)
    out.step_seconds = step_seconds[np.isfinite(step_seconds)] if impl != "reference" else None
    return out


def kmeans_assign_label(centroids, x):
    """KMeans::assign_label (ML/KMeans.cpp:153-165); `centroids` is (D, K)."""
    c = np.ascontiguousarray(np.asarray(centroids, dtype=np.float64).T)
    k, d = c.shape
    x = np.ascontiguousarray(x, dtype=np.float64)
    sq = ctypes.c_double()
    label = lib().mlpp_oracle_kmeans_assign_label(_ptr(x), d, k, _ptr(c), ctypes.byref(sq))
    return int(label), sq.value


def kmeans_assign_fused(centroids, x):
    """KMeans::assign_label (strict <, lowest index wins) for the rows of `x` (m, D), each squared distance summed as a
    chain of fused multiply-adds over the dimensions in order, as the device's exact refinement evaluates it; `centroids`
    is (D, K).  Returns (labels (m,) uint32, squared distances (m,))."""
    c = np.ascontiguousarray(np.asarray(centroids, dtype=np.float64).T)
    k, d = c.shape
    x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, d)
    labels = np.zeros(x.shape[0], dtype=np.uint32)
    sq = np.zeros(x.shape[0])
    lib().mlpp_oracle_kmeans_assign_fused(_ptr(x), d, x.shape[0], k, _ptr(c), labels.ctypes.data_as(_up), _ptr(sq))
    return labels, sq


def centroids_init(kind, data, k, seed=None, impl="oracle"):
    """Forgy / RandomPartition / KPP (ML/Clustering.cpp:16-59).  Returns (D, K)."""
    data = _check_data(data)
    n, d = data.shape
    c = np.zeros((k, d))
    (ref_lib().mlpp_ref_centroids_init if impl == "reference" else lib().mlpp_oracle_centroids_init)(kind, _ptr(data), d, n, d, k, 0 if seed is None else int(seed),
                                     0 if seed is None else 1, _ptr(c))
    return c.T.copy()


def xAx_symmetric(A, x, impl="oracle"):
    A = np.asfortranarray(A, dtype=np.float64)
    x = np.ascontiguousarray(x, dtype=np.float64)
    return (ref_lib().mlpp_ref_xAx_symmetric if impl == "reference" else lib().mlpp_oracle_xAx_symmetric)(A.ctypes.data_as(_dp), A.shape[0], _ptr(x))


def xxT(x, impl="oracle"):
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.zeros((x.size, x.size), order="F")
    (ref_lib().mlpp_ref_xxT if impl == "reference" else lib().mlpp_oracle_xxT)(_ptr(x), x.size, out.ctypes.data_as(_dp))
    return np.array(out)


def add_a_xxT(x, dest, a, impl="oracle"):
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.asfortranarray(dest, dtype=np.float64).copy(order="F")
    (ref_lib().mlpp_ref_add_a_xxT if impl == "reference" else lib().mlpp_oracle_add_a_xxT)(_ptr(x), x.size, out.ctypes.data_as(_dp), a)
    return np.array(out)


def testdata_two_gaussians():
    """The 400-point D=3 data of Tests/test_EM.cpp:10-34.  Returns ((400, 3) data, ground-truth labels)."""
    data = np.zeros((400, 3))
    truth = np.zeros(400, dtype=np.uint32)
    lib().mlpp_oracle_testdata_two_gaussians(_ptr(data), truth.ctypes.data_as(_up))
    return data, truth


def testdata_mouse(n):
    """The "mouse" data of Benchmarks/bm_EM.cpp:11-34.  Returns ((n, 2) data, class labels)."""
    data = np.zeros((n, 2))
    classes = np.zeros(n, dtype=np.uint32)
    lib().mlpp_oracle_testdata_mouse(_ptr(data), classes.ctypes.data_as(_up), n)
    return data, classes
