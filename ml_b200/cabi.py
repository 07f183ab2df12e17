"""ctypes binding of the C-ABI in include/mlb200.h (libmlb200.so).

This is the Python face of the same boundary the C++ host classes (ml_b200/host) call.  It never
imports the CPU oracle and has no fallback: loading fails loudly if the CUDA library is missing,
and every compute entry point fails with MLB_ECUDA when there is no device.

Matrices follow the reference's convention: column-major D x N data, which is the memory of a
C-contiguous numpy array of shape (N, D); means are (D, K) in the reference and cross this module
as C-contiguous (K, D) arrays (the same memory).
"""
import ctypes
import os
import weakref

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# MLB200_LIB: developer override used to time experimental builds of the same library (never a fallback).
LIB_PATH = os.environ.get("MLB200_LIB") or os.path.join(_HERE, "lib", "libmlb200.so")

MLB_OK, MLB_EINVAL, MLB_ECUDA, MLB_ENCCL, MLB_ENOMEM, MLB_ESTATE = range(6)

_c_dp = ctypes.POINTER(ctypes.c_double)
_c_up = ctypes.POINTER(ctypes.c_uint)
_c_i64p = ctypes.POINTER(ctypes.c_int64)
_c_ip = ctypes.POINTER(ctypes.c_int)
_vp = ctypes.c_void_p

# name -> (restype, argtypes).  tests/test_cabi_symbols.py checks this table against the header.
SIGNATURES = {
    "mlb_version": (ctypes.c_int, []),
    "mlb_last_error": (ctypes.c_char_p, []),
    "mlb_device_count": (ctypes.c_int, [_c_ip]),
    "mlb_selftest_exp": (ctypes.c_int, [_vp, ctypes.c_int64, _vp]),
    "mlb_selftest_fp64_peak": (ctypes.c_int, [ctypes.c_int, _c_dp, _c_dp]),
    "mlb_ctx_create": (ctypes.c_int, [_c_ip, ctypes.c_int, ctypes.POINTER(_vp)]),
    "mlb_nccl_unique_id": (ctypes.c_int, [_vp]),
    "mlb_ctx_create_rank": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, ctypes.POINTER(_vp)]),
    "mlb_ctx_destroy": (ctypes.c_int, [_vp]),
    "mlb_ctx_world": (ctypes.c_int, [_vp, _c_ip, _c_ip, _c_ip]),
    "mlb_ctx_sum_int64": (ctypes.c_int, [_vp, ctypes.c_int64, _c_i64p]),
    "mlb_ctx_synchronize": (ctypes.c_int, [_vp]),
    "mlb_ctx_timer_start": (ctypes.c_int, [_vp]),
    "mlb_ctx_timer_stop": (ctypes.c_int, [_vp, _c_dp]),
    "mlb_shard_range": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int, ctypes.c_int, _c_i64p, _c_i64p]),
    "mlb_data_upload": (ctypes.c_int, [_vp, _vp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int, ctypes.c_int64, ctypes.POINTER(_vp)]),
    "mlb_data_wrap_device": (ctypes.c_int, [_vp, _vp, ctypes.c_int64, ctypes.c_int, ctypes.POINTER(_vp)]),
    "mlb_data_generate_gmm": (ctypes.c_int, [_vp, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_uint64, ctypes.c_double, _vp,
                                             ctypes.POINTER(_vp)]),
    "mlb_data_download": (ctypes.c_int, [_vp, ctypes.c_int64, ctypes.c_int64, _vp]),
    "mlb_data_shape": (ctypes.c_int, [_vp, _c_i64p, _c_i64p, _c_ip]),
    "mlb_data_free": (ctypes.c_int, [_vp]),
    "mlb_standardise_features": (ctypes.c_int, [_vp, _vp, ctypes.c_int64, ctypes.c_int, ctypes.c_int64, _vp, ctypes.c_int64]),
    "mlb_data_kpp_update": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp]),
    "mlb_data_launch_count": (ctypes.c_int, [_vp, _c_i64p]),
    "mlb_em_create": (ctypes.c_int, [_vp, _vp, ctypes.c_int, ctypes.POINTER(_vp)]),
    "mlb_em_destroy": (ctypes.c_int, [_vp]),
    "mlb_em_sample_covariance": (ctypes.c_int, [_vp, _vp]),
    "mlb_em_set_params": (ctypes.c_int, [_vp, _vp, _vp, _vp]),
    "mlb_em_mstep_from_responsibilities": (ctypes.c_int, [_vp, _vp, ctypes.c_int64]),
    "mlb_em_mstep_from_labels": (ctypes.c_int, [_vp, _vp]),
    "mlb_em_step": (ctypes.c_int, [_vp, _c_dp]),
    "mlb_em_run_steps": (ctypes.c_int, [_vp, ctypes.c_int, _vp]),
    "mlb_em_get_params": (ctypes.c_int, [_vp, _vp, _vp, _vp]),
    "mlb_em_get_precisions": (ctypes.c_int, [_vp, _vp, _vp]),
    "mlb_em_emit": (ctypes.c_int, [_vp, _vp, ctypes.c_int64, _vp]),
    "mlb_em_emit_range": (ctypes.c_int, [_vp, ctypes.c_int64, ctypes.c_int64, _vp, ctypes.c_int64, _vp]),
    "mlb_em_predict": (ctypes.c_int, [_vp, _vp, ctypes.c_int64, ctypes.c_int64, _vp, ctypes.c_int64, _vp]),
    "mlb_em_set_kernel_timing": (ctypes.c_int, [_vp, ctypes.c_int]),
    "mlb_em_kernel_time_ms": (ctypes.c_int, [_vp, _c_dp, _c_i64p]),
    "mlb_em_last_path": (ctypes.c_int, [_vp, _c_ip]),
    "mlb_em_direct_steps": (ctypes.c_int, [_vp, _c_i64p]),
    "mlb_em_force_path": (ctypes.c_int, [_vp, ctypes.c_int]),
    "mlb_em_conditioning": (ctypes.c_int, [_vp, _c_dp, _c_ip]),
    "mlb_em_launch_count": (ctypes.c_int, [_vp, _c_i64p]),
    "mlb_em_kernel_config": (ctypes.c_int, [_vp, _c_ip]),
    "mlb_km_create": (ctypes.c_int, [_vp, _vp, ctypes.c_int, ctypes.POINTER(_vp)]),
    "mlb_km_destroy": (ctypes.c_int, [_vp]),
    "mlb_km_set_centroids": (ctypes.c_int, [_vp, _vp]),
    "mlb_km_get_centroids": (ctypes.c_int, [_vp, _vp]),
    "mlb_km_assign": (ctypes.c_int, [_vp, _c_dp, _c_i64p]),
    "mlb_km_update": (ctypes.c_int, [_vp, _c_dp]),
    "mlb_km_predict": (ctypes.c_int, [_vp, _vp, ctypes.c_int64, ctypes.c_int64, _vp, _vp]),
    "mlb_km_get_labels": (ctypes.c_int, [_vp, _vp]),
    "mlb_km_launch_count": (ctypes.c_int, [_vp, _c_i64p]),
    "mlb_km_kernel_config": (ctypes.c_int, [_vp, _c_ip]),
    "mlb_km_set_kernel_timing": (ctypes.c_int, [_vp, ctypes.c_int]),
    "mlb_km_kernel_time_ms": (ctypes.c_int, [_vp, _c_dp, _c_i64p]),
    "mlb_kms_supported": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int]),
    "mlb_kms_create": (ctypes.c_int, [_vp, _vp, ctypes.c_int, ctypes.c_int, ctypes.POINTER(_vp)]),
    "mlb_kms_destroy": (ctypes.c_int, [_vp]),
    "mlb_kms_set_centroids": (ctypes.c_int, [_vp, ctypes.c_int, _vp]),
    "mlb_kms_get_centroids": (ctypes.c_int, [_vp, ctypes.c_int, _vp]),
    "mlb_kms_assign": (ctypes.c_int, [_vp, ctypes.c_uint, _c_dp, _c_i64p]),
    "mlb_kms_update": (ctypes.c_int, [_vp, ctypes.c_uint, _c_dp]),
    "mlb_kms_get_labels": (ctypes.c_int, [_vp, ctypes.c_int, _vp]),
    "mlb_kms_launch_count": (ctypes.c_int, [_vp, _c_i64p]),
}

_lib = None


class MlbError(RuntimeError):
    def __init__(self, code, text):
        super().__init__(f"libmlb200 error {code}: {text}")
        self.code = code


def lib():
    """Loads libmlb200.so (built by __graft_entry__.build() / `make -C ml_b200/csrc`)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `make -C ml_b200/csrc` (there is no CPU fallback)")
        handle = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = handle
    return _lib


def check(rc):
    if rc != MLB_OK:
        raise MlbError(rc, lib().mlb_last_error().decode("utf-8", "replace"))


def _ptr(a):
    return None if a is None else a.ctypes.data_as(_vp)


def _kernel_config(fn, handle, names):
    out = (ctypes.c_int * 8)()
    check(fn(handle, out))
    return dict(zip(names, out))


EM_CONFIG_FIELDS = ("path", "DP", "KP", "NT", "MW", "direct_DP", "direct_NB", "chunk")
KM_CONFIG_FIELDS = ("DP", "KP", "KB", "nblocks", "nw", "exact", "stats", "chunk")


def device_count():
    n = ctypes.c_int()
    check(lib().mlb_device_count(ctypes.byref(n)))
    return n.value


def selftest_exp(x):
    """The kernels' FP64 exp for arguments <= 0, evaluated on device 0 (diagnostic)."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.empty_like(x)
    check(lib().mlb_selftest_exp(x.ctypes.data, x.size, out.ctypes.data))
    return out


def fp64_peak(device=0):
    """(DMMA, DFMA) TFLOP/s of `device`, measured now (diagnostic; bench.py's roofline denominator)."""
    a, b = ctypes.c_double(), ctypes.c_double()
    check(lib().mlb_selftest_fp64_peak(device, ctypes.byref(a), ctypes.byref(b)))
    return a.value, b.value


def standardise_features(ctx, features):
    """cppyml.utils.standardise_features (cppyml/cppyml/utils.py:8-28) on the device: (N, D) -> standardised copy."""
    x = np.ascontiguousarray(features, dtype=np.float64)
    assert x.ndim == 2
    out = np.empty_like(x)
    if x.size:
        check(lib().mlb_standardise_features(ctx._h, _ptr(x), x.shape[0], x.shape[1], x.shape[1], _ptr(out), x.shape[1]))
    return out


def shard_range(n_total, world, rank):
    b, e = ctypes.c_int64(), ctypes.c_int64()
    check(lib().mlb_shard_range(n_total, world, rank, ctypes.byref(b), ctypes.byref(e)))
    return b.value, e.value


def nccl_unique_id():
    buf = (ctypes.c_ubyte * 128)()
    check(lib().mlb_nccl_unique_id(ctypes.cast(buf, _vp)))
    return bytes(buf)


class Context:
    """A set of GPUs: `Context(n_devices=G)` drives G local GPUs from this process;
    `Context.for_rank(device, rank, world, unique_id)` is one rank of a torchrun-style job."""

    def __init__(self, n_devices=1, devices=None, _handle=None):
        self._h = _vp()
        self._children = weakref.WeakSet()   # Data / Em / Km objects living on this context: closed before it is
        if _handle is not None:
            self._h = _handle
            return
        arr = None
        if devices is not None:
            arr = (ctypes.c_int * len(devices))(*devices)
            n_devices = len(devices)
        check(lib().mlb_ctx_create(arr, n_devices, ctypes.byref(self._h)))

    @classmethod
    def for_rank(cls, device, rank, world, unique_id):
        h = _vp()
        buf = (ctypes.c_ubyte * 128).from_buffer_copy(unique_id) if unique_id is not None else None
        check(lib().mlb_ctx_create_rank(device, rank, world, ctypes.cast(buf, _vp) if buf is not None else None, ctypes.byref(h)))
        return cls(_handle=h)

    @property
    def world(self):
        w, n, f = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        check(lib().mlb_ctx_world(self._h, ctypes.byref(w), ctypes.byref(n), ctypes.byref(f)))
        return w.value

    def synchronize(self):
        check(lib().mlb_ctx_synchronize(self._h))

    def timer_start(self):
        check(lib().mlb_ctx_timer_start(self._h))

    def timer_stop(self):
        ms = ctypes.c_double()
        check(lib().mlb_ctx_timer_stop(self._h, ctypes.byref(ms)))
        return ms.value

    def close(self):
        if self._h:
            # objects that outlived their scope (a test that failed before its own close()) must go first: their handles
            # point into this context
            for kind in (Em, Km, Data):
                for child in list(self._children):
                    if isinstance(child, kind):
                        child.close()
            lib().mlb_ctx_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Data:
    """The point matrix resident in HBM."""

    def __init__(self, ctx, handle, keep=None):
        self.ctx = ctx
        self._h = handle
        self._keep = keep
        ctx._children.add(self)

    @classmethod
    def upload(cls, ctx, points, n_total=None):
        """`points`: C-contiguous float64 (n, D), i.e. column-major D x n.  Rank contexts pass their own rows."""
        if points.dtype != np.float64 or points.ndim != 2 or not points.flags.c_contiguous:
            raise TypeError("points must be a C-contiguous float64 array of shape (N, D)")
        n, d = points.shape
        h = _vp()
        check(lib().mlb_data_upload(ctx._h, _ptr(points), n, n if n_total is None else n_total, d, d, ctypes.byref(h)))
        return cls(ctx, h)

    @classmethod
    def wrap_device(cls, ctx, device_ptr, n, d, keep=None):
        h = _vp()
        check(lib().mlb_data_wrap_device(ctx._h, _vp(device_ptr), n, d, ctypes.byref(h)))
        return cls(ctx, h, keep)

    @classmethod
    def generate_gmm(cls, ctx, n_total, d, k_true, seed=1, spread=10.0):
        h = _vp()
        true_means = np.zeros((k_true, d))
        check(lib().mlb_data_generate_gmm(ctx._h, n_total, d, k_true, seed, spread, _ptr(true_means), ctypes.byref(h)))
        out = cls(ctx, h)
        out.true_means = true_means
        return out

    @property
    def shape(self):
        n, nl, d = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int()
        check(lib().mlb_data_shape(self._h, ctypes.byref(n), ctypes.byref(nl), ctypes.byref(d)))
        return n.value, nl.value, d.value

    def download(self, begin, count):
        _, _, d = self.shape
        out = np.empty((count, d))
        check(lib().mlb_data_download(self._h, begin, count, _ptr(out)))
        return out

    def kpp_update(self, centroid, first, want_nearest=True):
        """The distance pass of KPP::init (Clustering.cpp:42-51) for the newest centroid; returns the per-point
        squared distance to the nearest centroid chosen so far (all held points), or None."""
        c = np.ascontiguousarray(centroid, dtype=np.float64)
        _, n_local, d = self.shape
        assert c.shape == (d,)
        out = np.empty(n_local) if want_nearest else None
        check(lib().mlb_data_kpp_update(self._h, _ptr(c), int(bool(first)), _ptr(out)))
        return out

    @property
    def launch_count(self):
        c = ctypes.c_int64()
        check(lib().mlb_data_launch_count(self._h, ctypes.byref(c)))
        return c.value

    def close(self):
        if self._h:
            lib().mlb_data_free(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Em:
    """Device state of one ml::EM fit (ML/EM.hpp:168-187)."""

    def __init__(self, data, k):
        self.data = data
        self.k = k
        self.n_total, self.n_local, self.d = data.shape
        self._h = _vp()
        check(lib().mlb_em_create(data.ctx._h, data._h, k, ctypes.byref(self._h)))
        data.ctx._children.add(self)

    def sample_covariance(self):
        cov = np.empty((self.d, self.d))
        check(lib().mlb_em_sample_covariance(self._h, _ptr(cov)))
        return cov

    def set_params(self, means_dk, covariances, weights):
        """means_dk: (D, K) like ml::EM::means(); covariances: (K, D, D); weights: (K,)."""
        means = np.ascontiguousarray(np.asarray(means_dk, dtype=np.float64).T)
        covs = np.ascontiguousarray(np.asarray(covariances, dtype=np.float64).transpose(0, 2, 1))
        w = np.ascontiguousarray(weights, dtype=np.float64)
        assert means.shape == (self.k, self.d) and covs.shape == (self.k, self.d, self.d) and w.shape == (self.k,)
        check(lib().mlb_em_set_params(self._h, _ptr(means), _ptr(covs), _ptr(w)))

    def mstep_from_responsibilities(self, resp_nk):
        """resp_nk: (n, K) responsibilities as ml::EM::responsibilities() (column-major N x K)."""
        r = np.asfortranarray(resp_nk, dtype=np.float64)
        check(lib().mlb_em_mstep_from_responsibilities(self._h, _ptr(r), r.shape[0]))

    def mstep_from_labels(self, labels):
        """The M-step of one-hot responsibilities (ClosestCentroid start, Clustering.cpp:72-89) from the labels."""
        lab = np.ascontiguousarray(labels, dtype=np.uint32)
        assert lab.shape == (self.n_local,)
        check(lib().mlb_em_mstep_from_labels(self._h, _ptr(lab)))

    def predict(self, points, want_responsibilities=True, want_labels=True):
        """EM::assign_responsibilities (EM.cpp:176-188) for the rows of `points` (m, D) with the current parameters."""
        pts = np.ascontiguousarray(points, dtype=np.float64)
        assert pts.ndim == 2 and pts.shape[1] == self.d
        m = pts.shape[0]
        resp = np.empty((m, self.k), order="F") if want_responsibilities else None
        labels = np.empty(m, dtype=np.uint32) if want_labels else None
        check(lib().mlb_em_predict(self._h, _ptr(pts), m, self.d, _ptr(resp), max(m, 1), _ptr(labels)))
        return resp, labels

    def step(self):
        ll = ctypes.c_double()
        check(lib().mlb_em_step(self._h, ctypes.byref(ll)))
        return ll.value

    def run_steps(self, steps, want_ll=True):
        lls = np.empty(steps) if want_ll else None
        check(lib().mlb_em_run_steps(self._h, steps, _ptr(lls)))
        return lls

    def get_params(self):
        means = np.empty((self.k, self.d))
        covs = np.empty((self.k, self.d, self.d))
        w = np.empty(self.k)
        check(lib().mlb_em_get_params(self._h, _ptr(means), _ptr(covs), _ptr(w)))
        return means.T.copy(), covs.transpose(0, 2, 1).copy(), w

    def get_precisions(self):
        inv = np.empty((self.k, self.d, self.d))
        sd = np.empty(self.k)
        check(lib().mlb_em_get_precisions(self._h, _ptr(inv), _ptr(sd)))
        return inv.transpose(0, 2, 1).copy(), sd

    def emit(self, want_responsibilities=True, want_labels=True, rows=None, labels_out=None):
        """`labels_out`: an optional caller-owned uint32 array of n_local entries to receive the labels (e.g. pinned
        host memory, which the library copies into directly instead of through its bounce buffers)."""
        n = self.n_local if rows is None else rows
        resp = np.empty((n, self.k), order="F") if want_responsibilities else None
        labels = None
        if want_labels:
            labels = np.empty(n, dtype=np.uint32) if labels_out is None else labels_out
            assert labels.dtype == np.uint32 and labels.shape == (n,) and labels.flags.c_contiguous
        check(lib().mlb_em_emit(self._h, _ptr(resp), n, _ptr(labels)))
        return resp, labels

    def emit_range(self, begin, count, want_labels=True):
        """Responsibilities (count, K) and labels of the global point range [begin, begin + count) at the parameters the
        last step's E-step used."""
        resp = np.empty((count, self.k), order="F")
        labels = np.empty(count, dtype=np.uint32) if want_labels else None
        check(lib().mlb_em_emit_range(self._h, begin, count, _ptr(resp), max(count, 1), _ptr(labels)))
        return resp, labels

    def set_kernel_timing(self, enabled):
        check(lib().mlb_em_set_kernel_timing(self._h, int(enabled)))

    def kernel_time_ms(self):
        """(summed duration in ms, launches) of the fused kernel since timing was enabled."""
        ms, n = ctypes.c_double(), ctypes.c_int64()
        check(lib().mlb_em_kernel_time_ms(self._h, ctypes.byref(ms), ctypes.byref(n)))
        return ms.value, n.value

    @property
    def last_path(self):
        p = ctypes.c_int()
        check(lib().mlb_em_last_path(self._h, ctypes.byref(p)))
        return p.value

    @property
    def direct_steps(self):
        n = ctypes.c_int64()
        check(lib().mlb_em_direct_steps(self._h, ctypes.byref(n)))
        return n.value

    def force_path(self, path):
        """3: always the direct-difference kernels; 0: automatic routing."""
        check(lib().mlb_em_force_path(self._h, path))

    def conditioning(self):
        """(kappa of the current parameters, path of the next step)."""
        kappa, path = ctypes.c_double(), ctypes.c_int()
        check(lib().mlb_em_conditioning(self._h, ctypes.byref(kappa), ctypes.byref(path)))
        return kappa.value, path.value

    @property
    def launch_count(self):
        c = ctypes.c_int64()
        check(lib().mlb_em_launch_count(self._h, ctypes.byref(c)))
        return c.value

    def kernel_config(self):
        """The kernels chosen for this shape (diagnostic): path (1 fused, 2 split, 0 direct only), DP, KP, NT, MW (split M
        kernel, else 0), direct_DP, direct_NB, chunk (points per chunk of the data layout)."""
        return _kernel_config(lib().mlb_em_kernel_config, self._h, EM_CONFIG_FIELDS)

    def close(self):
        if self._h:
            lib().mlb_em_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Km:
    """Device state of one ml::Clustering::KMeans fit (ML/KMeans.hpp:103-116)."""

    def __init__(self, data, k):
        self.data = data
        self.k = k
        self.n_total, self.n_local, self.d = data.shape
        self._h = _vp()
        check(lib().mlb_km_create(data.ctx._h, data._h, k, ctypes.byref(self._h)))
        data.ctx._children.add(self)

    def set_centroids(self, centroids_dk):
        c = np.ascontiguousarray(np.asarray(centroids_dk, dtype=np.float64).T)
        assert c.shape == (self.k, self.d)
        check(lib().mlb_km_set_centroids(self._h, _ptr(c)))

    def get_centroids(self):
        c = np.empty((self.k, self.d))
        check(lib().mlb_km_get_centroids(self._h, _ptr(c)))
        return c.T.copy()

    def assign(self):
        inertia, changed = ctypes.c_double(), ctypes.c_int64()
        check(lib().mlb_km_assign(self._h, ctypes.byref(inertia), ctypes.byref(changed)))
        return inertia.value, changed.value

    def update(self):
        shift = ctypes.c_double()
        check(lib().mlb_km_update(self._h, ctypes.byref(shift)))
        return shift.value

    def predict(self, points):
        """KMeans::assign_label (KMeans.cpp:153-165) for the rows of `points` (m, D): (labels, squared distances)."""
        pts = np.ascontiguousarray(points, dtype=np.float64)
        assert pts.ndim == 2 and pts.shape[1] == self.d
        m = pts.shape[0]
        labels = np.empty(m, dtype=np.uint32)
        dist = np.empty(m)
        check(lib().mlb_km_predict(self._h, _ptr(pts), m, self.d, _ptr(labels), _ptr(dist)))
        return labels, dist

    def get_labels(self, labels_out=None):
        labels = np.empty(self.n_local, dtype=np.uint32) if labels_out is None else labels_out
        assert labels.dtype == np.uint32 and labels.shape == (self.n_local,) and labels.flags.c_contiguous
        check(lib().mlb_km_get_labels(self._h, _ptr(labels)))
        return labels

    def set_kernel_timing(self, enabled):
        check(lib().mlb_km_set_kernel_timing(self._h, int(enabled)))

    def kernel_time_ms(self):
        ms, n = ctypes.c_double(), ctypes.c_int64()
        check(lib().mlb_km_kernel_time_ms(self._h, ctypes.byref(ms), ctypes.byref(n)))
        return ms.value, n.value

    @property
    def launch_count(self):
        c = ctypes.c_int64()
        check(lib().mlb_km_launch_count(self._h, ctypes.byref(c)))
        return c.value

    def kernel_config(self):
        """The kernels chosen for this shape (diagnostic): DP, KP, KB, nblocks, nw (warps per assignment CTA), exact (D > 64
        scan), stats (0 one-hot, 1 counting sort, 2 owner warps), chunk."""
        return _kernel_config(lib().mlb_km_kernel_config, self._h, KM_CONFIG_FIELDS)

    def close(self):
        if self._h:
            lib().mlb_km_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Kms:
    """Up to four K-means starts advanced in lockstep on one resident data set (mlb_kms, KMeans.cpp:29-47).  `active` is a
    bit mask of the starts a call advances (default: all)."""

    def __init__(self, data, k, n_sets):
        self.data, self.k, self.n_sets = data, k, n_sets
        self.n_total, self.n_local, self.d = data.shape
        self._h = _vp()
        check(lib().mlb_kms_create(data.ctx._h, data._h, k, n_sets, ctypes.byref(self._h)))
        data.ctx._children.add(self)

    @staticmethod
    def supported(data, k, n_sets):
        return bool(lib().mlb_kms_supported(data._h, k, n_sets))

    def _mask(self, active):
        return (1 << self.n_sets) - 1 if active is None else int(active)

    def set_centroids(self, s, centroids_dk):
        c = np.ascontiguousarray(np.asarray(centroids_dk, dtype=np.float64).T)
        assert c.shape == (self.k, self.d)
        check(lib().mlb_kms_set_centroids(self._h, s, _ptr(c)))

    def get_centroids(self, s):
        c = np.empty((self.k, self.d))
        check(lib().mlb_kms_get_centroids(self._h, s, _ptr(c)))
        return c.T.copy()

    def assign(self, active=None):
        """(inertia[n_sets], changed[n_sets]); entries of starts outside `active` stay 0."""
        inertia = np.zeros(4)
        changed = np.zeros(4, dtype=np.int64)
        check(lib().mlb_kms_assign(self._h, self._mask(active), inertia.ctypes.data_as(_c_dp), changed.ctypes.data_as(_c_i64p)))
        return inertia[: self.n_sets], changed[: self.n_sets]

    def update(self, active=None):
        shift = np.zeros(4)
        check(lib().mlb_kms_update(self._h, self._mask(active), shift.ctypes.data_as(_c_dp)))
        return shift[: self.n_sets]

    def get_labels(self, s):
        labels = np.empty(self.n_local, dtype=np.uint32)
        check(lib().mlb_kms_get_labels(self._h, s, _ptr(labels)))
        return labels

    @property
    def launch_count(self):
        c = ctypes.c_int64()
        check(lib().mlb_kms_launch_count(self._h, ctypes.byref(c)))
        return c.value

    def close(self):
        if self._h:
            lib().mlb_kms_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
