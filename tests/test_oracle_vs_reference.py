"""The CPU restatement (oracle/mlpp_oracle.cpp) against the reference's OWN code.

oracle/_ref/libmlpp_ref.so is built by oracle/Makefile from the reference's four clustering translation units where they
lie under /root/reference (ML/EM.cpp, ML/KMeans.cpp, ML/Clustering.cpp, ML/LinearAlgebra.cpp), with the first-party
Eigen stand-in of oracle/eigen_standin/ in place of the Eigen 3 headers the image lacks.  Control flow, loop structure,
PRNG use and scalar arithmetic are therefore the reference's; only the evaluation order INSIDE Eigen's dense products,
reductions and LLT is the stand-in's (sequential).  The restatement makes the same choice, so the two agree operation
for operation: compiled with -ffp-contract=off they are bit-identical (test_bitwise_without_fma_contraction); with the
reference's release flags the compiler fuses a*b+c differently in the two sources, which moves results by an ulp, so
the default builds are compared at 1e-13 relative with identical iteration counts, convergence flags and labels.

Every reference-side result is a named case of CASES.  Where oracle/_ref is built, a case runs there, and the stored
record tests/golden/reference_cases.npz must agree with it too.  Elsewhere the record stands in for the library, so the
comparisons also run in a checkout without the reference.  tests/golden/make_reference_cases.py writes the record; its
`source` entry says whether the reference's own code or the oracle wrote it (the oracle, when the library was not
built).  The record keeps RESPONSIBILITY_ROWS evenly spread rows of each responsibility matrix and everything else
whole."""
import functools
import os
import types

import numpy as np
import pytest

import oracle
from tests.datasets import mouse_numpy, synthetic_gmm

RECORD_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_cases.npz")
RESPONSIBILITY_ROWS = 256
INITS = [oracle.FORGY, oracle.RANDOM_PARTITION, oracle.KPP]
EM_SYNTHETIC = [(3000, 2, 3, 1), (2000, 8, 5, 2), (1500, 13, 4, 3), (1500, 14, 4, 4), (1500, 15, 3, 5), (1200, 20, 4, 6), (900, 33, 3, 7)]
KM_MULTI_START = [(3, 2), (5, 3), (4, 100), (6, 100)]
KM_SYNTHETIC = [(4000, 2, 3, 1), (3000, 8, 16, 2), (2000, 32, 40, 3), (1000, 1, 4, 4)]
INIT_SEEDS = (None, 0, 12345)
LINALG_DIMS = [1, 2, 5, 10, 11, 13, 14, 15, 24, 40]


# ------------------------------------------------------------------------------------------------ the cases

def _em(data_fn, k, queries=0, **kw):
    """A case of oracle.em_fit; `queries` first points go through EM::assign_responsibilities after the fit."""
    def run(impl):
        data = data_fn()
        q = data[:queries] if queries else None
        fit = oracle.em_fit(data, k, impl=impl, queries=q, **kw)
        out = dict(converged=fit.converged, iterations=fit.iterations, log_likelihood=fit.log_likelihood, means=fit.means,
                   covariances=fit.covariances, mixing_probabilities=fit.mixing_probabilities,
                   responsibilities=fit.responsibilities, labels=fit.labels)
        if q is not None:
            out["query_responsibilities"] = (fit.query_responsibilities if impl == "reference" else
                                             np.array([oracle.em_assign_responsibilities(fit, x) for x in q]))
        return out
    return run


def _kmeans(data_fn, k, queries=0, **kw):
    """A case of oracle.kmeans_fit; `queries` first points go through KMeans::assign_label after the fit."""
    def run(impl):
        data = data_fn()
        q = data[:queries] if queries else None
        fit = oracle.kmeans_fit(data, k, impl=impl, queries=q, **kw)
        out = dict(converged=fit.converged, inertia=fit.inertia, centroids=fit.centroids, labels=fit.labels)
        if kw.get("number_initialisations", 1) == 1:
            out["iterations"] = fit.iterations   # not observable from outside for a multi-start fit
        if q is not None:
            if impl == "reference":
                out["query_labels"], out["query_distances"] = fit.query_labels, fit.query_distances
            else:
                pairs = [oracle.kmeans_assign_label(fit.centroids, x) for x in q]
                out["query_labels"] = np.array([p[0] for p in pairs], dtype=np.uint32)
                out["query_distances"] = np.array([p[1] for p in pairs])
        return out
    return run


def _em_errors(impl):
    data = np.random.default_rng(0).normal(size=(5, 3))
    out = {}
    for name, k in (("k6_raises", 6), ("k0_raises", 0)):   # fewer points than components (EM.cpp:99-101), no components (EM.cpp:34-36)
        try:
            oracle.em_fit(data, k, impl=impl)
            out[name] = False
        except ValueError:
            out[name] = True
    return out


def _initialiser(kind, seed, impl):
    data, _, _ = synthetic_gmm(700, 5, 6, seed=21)
    return {"centroids": oracle.centroids_init(kind, data, 6, seed=seed, impl=impl)}


def _linalg_inputs(dim):
    rng = np.random.default_rng(dim)
    a = rng.normal(size=(dim, dim))
    return a + a.T, rng.normal(size=dim)


def _linalg(dim, impl):
    a, x = _linalg_inputs(dim)
    return {"xAx": oracle.xAx_symmetric(a, x, impl=impl), "xxT": oracle.xxT(x, impl=impl), "add_a_xxT": oracle.add_a_xxT(x, a, 0.37, impl=impl)}


def _two_gaussians():
    return oracle.testdata_two_gaussians()[0]


def _mouse(n):
    return oracle.testdata_mouse(n)[0]


def _synthetic(n, d, k, seed, spread):
    return synthetic_gmm(n, d, k, seed=seed, spread=spread)[0]


def _explicit_means_case():
    data = _synthetic(2500, 6, 4, 11, 5.0)
    return data, np.ascontiguousarray(data[::600][:4].T)


CASES = {}   # name -> run(impl) -> dict of the reference-side results
for _init in INITS:
    for _mf in (False, True):
        CASES[f"em_test_data_{_init}_{int(_mf)}"] = _em(_two_gaussians, 2, queries=16, seed=42, means_init=_init, resp_init_centroids=_init,
                                                        maximise_first=_mf, maximum_steps=100)
    for _inits in (1, 3):
        CASES[f"km_test_data_{_init}_{_inits}"] = _kmeans(_two_gaussians, 2, queries=32, seed=42, init=_init, number_initialisations=_inits,
                                                          maximum_steps=100)
    for _seed in INIT_SEEDS:
        CASES[f"initialiser_{_init}_{_seed}"] = functools.partial(_initialiser, _init, _seed)
CASES["em_mouse"] = _em(functools.partial(_mouse, 10000), 3, seed=42, means_init=oracle.KPP, absolute_tolerance=1e-14, relative_tolerance=1e-14)
for _n, _d, _k, _seed in EM_SYNTHETIC:
    CASES[f"em_synthetic_{_n}_{_d}_{_k}_{_seed}"] = _em(functools.partial(_synthetic, _n, _d, _k, _seed, 6.0), _k, seed=7, means_init=oracle.FORGY,
                                                        maximum_steps=40)
CASES["em_explicit_means"] = lambda impl: _em(lambda: _explicit_means_case()[0], 4, means_init=oracle.EXPLICIT,
                                              explicit_means=_explicit_means_case()[1], maximum_steps=60)(impl)
CASES["em_exact_fit"] = _em(lambda: np.random.default_rng(0).normal(size=(5, 3)), 5)
CASES["em_argument_errors"] = _em_errors
for _inits, _steps in KM_MULTI_START:
    CASES[f"km_multi_start_{_inits}_{_steps}"] = _kmeans(functools.partial(_mouse, 4000), 3, seed=77, init=oracle.KPP, absolute_tolerance=1e-14,
                                                         number_initialisations=_inits, maximum_steps=_steps)
for _n, _d, _k, _seed in KM_SYNTHETIC:
    CASES[f"km_synthetic_{_n}_{_d}_{_k}_{_seed}"] = _kmeans(functools.partial(_synthetic, _n, _d, min(_k, 12), _seed, 5.0), _k, seed=3,
                                                            init=oracle.KPP, maximum_steps=200)
CASES["km_mouse"] = _kmeans(mouse_numpy, 3, seed=1, init=oracle.FORGY, absolute_tolerance=1e-14)
for _dim in LINALG_DIMS:
    CASES[f"linalg_{_dim}"] = functools.partial(_linalg, _dim)


# ------------------------------------------------------------------------------------------------ the record

def record_entries(name, result):
    """What the record keeps of one case's results, keyed `name/field`: responsibility matrices cut to
    RESPONSIBILITY_ROWS rows (their indices under `name/responsibility_rows`), everything else whole."""
    out = {}
    for field, value in result.items():
        value = np.asarray(value)
        if field == "responsibilities":
            rows = np.unique(np.linspace(0, value.shape[0] - 1, min(value.shape[0], RESPONSIBILITY_ROWS)).astype(np.int64))
            out[f"{name}/responsibility_rows"] = rows
            value = value[rows]
        out[f"{name}/{field}"] = value
    return out


@functools.lru_cache(maxsize=None)
def _record():
    with np.load(RECORD_PATH) as z:
        return {key: z[key] for key in z.files}


def reference(name):
    """The reference-side results of case `name` as attributes: computed by oracle/_ref when it is built (the record must
    then agree with them), else read from the record."""
    prefix = name + "/"
    stored = {key: value for key, value in _record().items() if key.startswith(prefix)}
    assert stored, f"case {name} is not in {RECORD_PATH}; rerun tests/golden/make_reference_cases.py"
    if oracle.ref_available():
        live = CASES[name]("reference")
        expected = record_entries(name, live)
        assert sorted(stored) == sorted(expected), name
        for key, want in expected.items():
            if want.dtype.kind in "biuU":
                assert np.array_equal(stored[key], want), key
            else:
                assert np.array_equal(stored[key], want) or close(stored[key], want, False), key
        return types.SimpleNamespace(**live)
    return types.SimpleNamespace(**{key[len(prefix):]: (value.item() if value.ndim == 0 else value) for key, value in stored.items()})


# ------------------------------------------------------------------------------------------------ the comparisons

def close(x, y, exact):
    x, y = np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)
    if exact:
        return np.array_equal(x, y, equal_nan=True)
    return bool(np.all(np.abs(x - y) <= 1e-13 * max(1e-300, float(np.max(np.abs(y))))))


def responsibilities(a, b):
    """a's responsibilities on the rows b holds (all of them, unless b comes from the record)."""
    rows = getattr(b, "responsibility_rows", None)
    return a.responsibilities if rows is None else a.responsibilities[rows]


def same_em(a, b, exact=False):
    assert a.converged == b.converged
    assert a.iterations == b.iterations
    assert close(a.log_likelihood, b.log_likelihood, exact) or (np.isinf(a.log_likelihood) and a.log_likelihood == b.log_likelihood)
    assert close(a.means, b.means, exact)
    assert close(a.covariances, b.covariances, exact)
    assert close(a.mixing_probabilities, b.mixing_probabilities, exact)
    assert close(responsibilities(a, b), b.responsibilities, exact)
    if a.converged:
        assert np.array_equal(a.labels, b.labels)


def same_kmeans(a, b, exact=False):
    assert a.converged == b.converged
    assert a.iterations == b.iterations
    assert close(a.inertia, b.inertia, exact)
    assert close(a.centroids, b.centroids, exact)
    assert np.array_equal(a.labels, b.labels)


@pytest.mark.parametrize("init", INITS)
@pytest.mark.parametrize("maximise_first", [False, True])
def test_em_on_the_reference_test_data(init, maximise_first):
    """Tests/test_EM.cpp:36-87: the 400-point two-Gaussian data, every initialiser, both start modes."""
    data, _ = oracle.testdata_two_gaussians()
    kw = dict(seed=42, means_init=init, resp_init_centroids=init, maximise_first=maximise_first, maximum_steps=100)
    a = oracle.em_fit(data, 2, **kw)
    b = reference(f"em_test_data_{init}_{int(maximise_first)}")
    same_em(a, b)
    # EM::assign_responsibilities of the reference (EM.cpp:176-188) against the oracle's, from the post-fit parameters
    for i in range(16):
        assert close(oracle.em_assign_responsibilities(a, data[i]), b.query_responsibilities[i], False)


def test_em_mouse_benchmark_configuration():
    """BASELINE config 1 (Benchmarks/bm_EM.cpp:9-48): mouse data, N = 10k, K = 3, KPP, tolerances 1e-14."""
    data, _ = oracle.testdata_mouse(10000)
    kw = dict(seed=42, means_init=oracle.KPP, absolute_tolerance=1e-14, relative_tolerance=1e-14)
    same_em(oracle.em_fit(data, 3, **kw), reference("em_mouse"))


@pytest.mark.parametrize("n,d,k,seed", EM_SYNTHETIC)
def test_em_on_synthetic_mixtures(n, d, k, seed):
    """Dimensions on both sides of the reference's hand-written / Eigen switches (LinearAlgebra.cpp:17, 59: 15 and 14)
    and of Eigen's blocked LLT (n >= 32 in the real library; unblocked in both stand-ins)."""
    data = _synthetic(n, d, k, seed, 6.0)
    kw = dict(seed=7, means_init=oracle.FORGY, maximum_steps=40)
    same_em(oracle.em_fit(data, k, **kw), reference(f"em_synthetic_{n}_{d}_{k}_{seed}"))


def test_em_explicit_means_plugin():
    """A user-supplied CentroidsInitialiser (Clustering.hpp:58-72) is how the parity tests fix the initial means."""
    data, init = _explicit_means_case()
    kw = dict(means_init=oracle.EXPLICIT, explicit_means=init, maximum_steps=60)
    same_em(oracle.em_fit(data, 4, **kw), reference("em_explicit_means"))


def test_em_exact_fit_and_argument_errors():
    data = np.random.default_rng(0).normal(size=(5, 3))
    a, b = oracle.em_fit(data, 5), reference("em_exact_fit")
    assert a.converged and b.converged and np.isinf(a.log_likelihood) and np.isinf(b.log_likelihood)
    assert np.array_equal(a.means, b.means) and np.array_equal(a.labels, b.labels) and np.array_equal(responsibilities(a, b), b.responsibilities)
    errors = reference("em_argument_errors")
    assert errors.k6_raises and errors.k0_raises
    with pytest.raises(ValueError):
        oracle.em_fit(data, 6)          # fewer points than components (EM.cpp:99-101)
    with pytest.raises(ValueError):
        oracle.em_fit(data, 0)          # no components (EM.cpp:34-36)


@pytest.mark.parametrize("init", INITS)
@pytest.mark.parametrize("inits", [1, 3])
def test_kmeans_on_the_reference_test_data(init, inits):
    """Tests/test_KMeans.cpp:40-73 plus the multi-start selection of KMeans.cpp:29-47."""
    data, _ = oracle.testdata_two_gaussians()
    kw = dict(seed=42, init=init, number_initialisations=inits, maximum_steps=100)
    a = oracle.kmeans_fit(data, 2, **kw)
    b = reference(f"km_test_data_{init}_{inits}")
    if inits > 1:
        b.iterations = a.iterations   # not observable from outside for a multi-start fit
    same_kmeans(a, b)
    for i in range(32):
        label, sq = oracle.kmeans_assign_label(a.centroids, data[i])
        assert label == b.query_labels[i] and close(sq, b.query_distances[i], False)


@pytest.mark.parametrize("inits,max_steps", KM_MULTI_START)
def test_kmeans_multi_start_with_and_without_convergence(inits, max_steps):
    """KMeans.cpp:29-47 when some or all starts run out of steps: the best CONVERGED start wins; when none converged the
    object is left in the last start's state (labels of its last assignment, centroids of its last update).  The device
    path's lockstep multi-start (ml_b200/host/src/KMeans.cpp, fit_lockstep) is tested against the port on exactly these
    cases (tests/test_gpu_kmeans_sets.py), so the port is pinned to the reference's own code on them here."""
    data, _ = oracle.testdata_mouse(4000)
    kw = dict(seed=77, init=oracle.KPP, absolute_tolerance=1e-14, number_initialisations=inits, maximum_steps=max_steps)
    a = oracle.kmeans_fit(data, 3, **kw)
    b = reference(f"km_multi_start_{inits}_{max_steps}")
    b.iterations = a.iterations   # not observable from outside for a multi-start fit
    same_kmeans(a, b)


@pytest.mark.parametrize("n,d,k,seed", KM_SYNTHETIC)
def test_kmeans_on_synthetic_mixtures(n, d, k, seed):
    data = _synthetic(n, d, min(k, 12), seed, 5.0)
    kw = dict(seed=3, init=oracle.KPP, maximum_steps=200)
    same_kmeans(oracle.kmeans_fit(data, k, **kw), reference(f"km_synthetic_{n}_{d}_{k}_{seed}"))


def test_kmeans_mouse():
    data = mouse_numpy()
    kw = dict(seed=1, init=oracle.FORGY, absolute_tolerance=1e-14)
    same_kmeans(oracle.kmeans_fit(data, 3, **kw), reference("km_mouse"))


@pytest.mark.parametrize("kind", INITS)
def test_initialisers_draw_the_same_prng_stream(kind):
    data, _, _ = synthetic_gmm(700, 5, 6, seed=21)
    for seed in INIT_SEEDS:
        assert close(oracle.centroids_init(kind, data, 6, seed=seed), reference(f"initialiser_{kind}_{seed}").centroids, False)


@pytest.mark.parametrize("dim", LINALG_DIMS)
def test_linear_algebra_helpers(dim):
    """LinearAlgebra.cpp:8-73 on both sides of its size switches (15, 11, 14)."""
    a, x = _linalg_inputs(dim)
    b = reference(f"linalg_{dim}")
    assert abs(oracle.xAx_symmetric(a, x) - b.xAx) <= 1e-13 * np.abs(a).sum() * np.abs(x).max() ** 2
    assert close(oracle.xxT(x), b.xxT, False)
    assert close(oracle.add_a_xxT(x, a, 0.37), b.add_a_xxT, False)


def test_bitwise_without_fma_contraction(tmp_path):
    """Both sources compiled with -ffp-contract=off: every arithmetic operation is then the one written in the source,
    and the restatement must reproduce the reference's own code BIT FOR BIT (EM and K-means, several shapes)."""
    import ctypes
    import os
    import subprocess
    reference = "/root/reference/ML"
    if not os.path.exists(os.path.join(reference, "EM.cpp")):
        pytest.skip("the reference checkout is not mounted here")
    here = os.path.dirname(os.path.abspath(oracle.__file__))
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    flags = ["-O2", "-march=x86-64-v3", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared", "-w"]
    o_path, r_path = str(tmp_path / "oracle_nofma.so"), str(tmp_path / "ref_nofma.so")
    subprocess.check_call([cxx, *flags, "-o", o_path, os.path.join(here, "mlpp_oracle.cpp")])
    subprocess.check_call([cxx, *flags, "-I", os.path.join(here, "eigen_standin"), "-I", reference, "-o", r_path,
                           *[os.path.join(reference, f) for f in ("EM.cpp", "KMeans.cpp", "Clustering.cpp", "LinearAlgebra.cpp")],
                           os.path.join(here, "ref_shim.cpp")])
    saved = (oracle._lib, oracle._ref, oracle._LIB_PATH, oracle._REF_LIB_PATH, oracle.build)
    try:
        oracle._lib = oracle._ref = None
        oracle._LIB_PATH, oracle._REF_LIB_PATH = o_path, r_path
        oracle.build = lambda force=False: o_path
        mouse, _ = oracle.testdata_mouse(10000)
        kw = dict(seed=42, means_init=oracle.KPP, absolute_tolerance=1e-14, relative_tolerance=1e-14)
        same_em(oracle.em_fit(mouse, 3, **kw), oracle.em_fit(mouse, 3, impl="reference", **kw), exact=True)
        for n, d, k, seed in [(2000, 8, 5, 2), (1500, 14, 4, 4), (1500, 15, 3, 5), (1200, 20, 4, 6)]:
            data, _, _ = synthetic_gmm(n, d, k, seed=seed, spread=6.0)
            kw = dict(seed=7, means_init=oracle.FORGY, maximum_steps=40)
            same_em(oracle.em_fit(data, k, **kw), oracle.em_fit(data, k, impl="reference", **kw), exact=True)
            kw = dict(seed=3, init=oracle.KPP, maximum_steps=200)
            same_kmeans(oracle.kmeans_fit(data, k + 3, **kw), oracle.kmeans_fit(data, k + 3, impl="reference", **kw), exact=True)
    finally:
        oracle._lib, oracle._ref, oracle._LIB_PATH, oracle._REF_LIB_PATH, oracle.build = saved
