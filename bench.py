#!/usr/bin/env python
"""Benchmark of the clustering hot path (BASELINE.json): Gaussian-mixture EM iterations on B200.

    python bench.py --gpus N --steps K --warmup W            # this repository's CUDA path
    python bench.py --impl reference --steps K --warmup W     # the reference algorithm on the host CPU
    python bench.py ... --dump-outputs DIR                     # also write what the last timed step computed to DIR/*.npy

Default workload: BASELINE configuration 3, the north-star target: ml::EM full-covariance GMM, N = 100M, D = 16, K = 32.
N is FIXED: --gpus G shards the same 100M points over G GPUs ("scaling": "strong"), one process per GPU under torchrun.
Other workloads (`--workload`): c1 (mouse data, whole fits), c2 (N=10M, D=8, K=16), c4 (N=20M, D=64, K=64), c5 (K-means,
N=100M, D=32, K=256).  A "step" is one iteration (E-step + M-step + statistics exchange + parameter refresh) over the
whole data set; metric = point-component pairs per second.

One JSON line on stdout (rank 0):
  value        K steps with the points resident in HBM, CUDA events on the library's stream, max over ranks;
  e2e          the same metric for a whole `cppyml.clustering.EM(k).fit(X)` (KMeans for c5) on a plain, PAGEABLE numpy array:
               upload, initialisation, K iterations with the convergence scalar read back each iteration, parameters
               read back through the Python properties; wall clock, max over ranks;
  roofline     the dominant kernel's algorithmic flops / its CUDA-event time against the FP64 pipe peak measured live;
  cpu_baseline the CPU oracle (a port of the reference's single-threaded loops) on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# name -> (kind, TOTAL points, D, K): the BASELINE.json configurations as quoted.
WORKLOADS = {
    "c1": ("em", 10_000, 2, 3),
    "c2": ("em", 10_000_000, 8, 16),
    "c3": ("em", 100_000_000, 16, 32),
    "c4": ("em", 20_000_000, 64, 64),
    "c5": ("km", 100_000_000, 32, 256),
}
METRIC = "em_point_components_per_second"
METRIC_KM = "kmeans_point_centroids_per_second"
UNIT = "Gpoint*comp/s"
DATA_SEED = 20261018
# Fallback roofline denominator when the live measurement is unavailable: profiles/fp64_peaks_r01.json (DMMA chain).
FP64_PEAK_TFLOPS_FALLBACK = 37.0
# CPU sample sizes of BASELINE.md §4 (upper bounds; the sample is cut to fit --cpu-budget seconds)
CPU_SAMPLE_MAX = {"c1": 10_000, "c2": 1_000_000, "c3": 1_000_000, "c4": 200_000, "c5": 1_000_000}
# --dump-outputs: per-point outputs are written for DUMP_BLOCKS blocks of DUMP_BLOCK_ROWS consecutive points at seeded
# offsets; 65536 rows of K <= 64 responsibilities are at most 32 MB, within the 64 MB the files may take in all.
DUMP_BLOCKS, DUMP_BLOCK_ROWS = 64, 1024
DUMP_LIMIT_BYTES = 64 << 20


def f_em(d):
    """Algorithmic FP64 flops per point-component pair per iteration (SURVEY.md §8d, BASELINE.md §3)."""
    return 2 * d * d + 8 * d + 6


def flops_per_iteration(kind, n, d, k):
    """EM: N K F_EM(D).  K-means: N K (3D + 1) for the assignment + N (2D + 1) for the update (SURVEY.md §8d)."""
    return n * k * f_em(d) if kind == "em" else n * k * (3 * d + 1) + n * (2 * d + 1)


def dump_sample_rows(n_total):
    """Global indices of the points whose per-point outputs --dump-outputs writes: DUMP_BLOCKS blocks of DUMP_BLOCK_ROWS
    consecutive points at offsets drawn from a fixed seed (the first points when there are too few for that)."""
    import numpy as np
    blocks = n_total // DUMP_BLOCK_ROWS
    if blocks <= DUMP_BLOCKS:
        return np.arange(min(n_total, DUMP_BLOCKS * DUMP_BLOCK_ROWS))
    starts = np.sort(np.random.default_rng(DATA_SEED).choice(blocks, DUMP_BLOCKS, replace=False)) * DUMP_BLOCK_ROWS
    return (starts[:, None] + np.arange(DUMP_BLOCK_ROWS)).ravel()


def write_outputs(directory, arrays):
    """Writes each entry of `arrays` (name -> array) as directory/<name>.npy in float64."""
    import numpy as np
    arrays = {name: np.asarray(a, dtype=np.float64) for name, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs, more than the {DUMP_LIMIT_BYTES} allowed")
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--points", type=int, default=0, help="override the workload's total point count (developer runs)")
    ap.add_argument("--no-clocks", action="store_true", help="developer runs: no NVML clock sampling thread")
    ap.add_argument("--cpu-sample", type=int, default=0, help="points of the CPU sample (0 = fit --cpu-budget)")
    ap.add_argument("--cpu-budget", type=float, default=0.0, help="seconds of CPU work for the baseline (0 = 25 s in cpu_baseline, 150 s in --impl reference)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-responsibilities", action="store_true", help="skip the separately declared lazy responsibilities() timing")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy "
                                                          "(float64; per-point outputs on a fixed sample of rows) to compare two builds")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the device path (--impl b200)")
    return args


class ClockSampler:
    """SM clock, power and clock-event (throttle) reasons DURING the timed region, polled through NVML every few
    milliseconds from a thread (a 20-step region is 0.17 s at 8 GPUs: nvidia-smi's 20 ms loop would leave a handful of
    samples).  Falls back to an `nvidia-smi -lms` subprocess when the NVML binding is unusable."""

    def __init__(self, index, uuid=None):
        self.index, self.uuid = index, uuid
        self.samples = []          # (stamp, sm_mhz, max_mhz, power_w, [reasons])
        self.t_begin = self.t_end = None
        self.stop_flag = False
        self.thread = None
        self.proc = None
        self.source = None

    def _nvml_loop(self, nv, handle, max_mhz):
        bits = []
        for name, attr in (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"), ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
                           ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"), ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap")):
            bit = getattr(nv, attr, None)
            if bit is None:
                bit = getattr(nv, attr.replace("ClocksEventReason", "ClocksThrottleReason"), None)
            if bit is not None:
                bits.append((name, bit))
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)
                mask = get_reasons(handle)
                power = nv.nvmlDeviceGetPowerUsage(handle) / 1000.0
                self.samples.append((time.time(), float(sm), float(max_mhz), power, [n for n, b in bits if mask & b]))
            except Exception:
                pass
            time.sleep(0.004)

    def _smi_loop(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                self.samples.append((time.time(), float(parts[0]), float(parts[1]), float(parts[2]), [n for n, f in zip(names, parts[3:7]) if f.lower().startswith("active")]))
            except ValueError:
                continue

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            handle = None
            if self.uuid:
                for cand in (self.uuid, "GPU-" + self.uuid):
                    try:
                        handle = nv.nvmlDeviceGetHandleByUUID(cand.encode() if hasattr(cand, "encode") else cand)
                        break
                    except Exception:
                        handle = None
            if handle is None:
                handle = nv.nvmlDeviceGetHandleByIndex(self.index)
            max_mhz = nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM)
            self.source = "nvml"
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, handle, max_mhz), daemon=True)
            self.thread.start()
            return
        except Exception:
            pass
        try:
            query = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                     "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + query, "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi -lms 20"
            self.thread = threading.Thread(target=self._smi_loop, daemon=True)
            self.thread.start()
            deadline = time.time() + 3.0
            while not self.samples and time.time() < deadline:
                time.sleep(0.01)
        except OSError:
            self.proc = None

    def mark_begin(self):
        self.t_begin = time.time()

    def mark_end(self):
        self.t_end = time.time()

    def stop(self):
        self.stop_flag = True
        if self.proc:
            time.sleep(0.05)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        if self.thread:
            self.thread.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock source available"]}
        inside = [r for r in self.samples if self.t_begin is not None and self.t_begin <= r[0] <= self.t_end]
        note = "samples inside the timed region"
        if not inside and self.t_begin is not None:
            mid = 0.5 * (self.t_begin + self.t_end)
            inside = [min(self.samples, key=lambda r: abs(r[0] - mid))]
            note = "timed region shorter than the sampling period: nearest sample"
        sm = sorted(r[1] for r in inside)
        return {"sm_mhz": sm[len(sm) // 2], "sm_mhz_min": sm[0], "sm_max_mhz": max(r[2] for r in inside), "power_w_max": max(r[3] for r in inside),
                "samples": len(inside), "reasons": sorted({n for r in inside for n in r[4]}), "note": note, "source": self.source,
                "timed_region_ms": None if self.t_begin is None else (self.t_end - self.t_begin) * 1e3}


# ----------------------------------------------------------------------------------------------- CPU baseline

def _oracle_fit(kind, data, k, init, maximum_steps, impl="port"):
    import oracle
    if kind == "em":
        return oracle.em_fit(data, k, means_init=oracle.EXPLICIT, explicit_means=init, maximum_steps=maximum_steps, absolute_tolerance=0.0,
                             relative_tolerance=0.0, want_responsibilities=False, impl=impl)
    return oracle.kmeans_fit(data, k, init=oracle.EXPLICIT, explicit_means=init, maximum_steps=maximum_steps, absolute_tolerance=0.0, impl=impl)


def _cpu_data(n_cpu, d, k):
    import numpy as np
    from tests.datasets import synthetic_gmm
    data, _, _ = synthetic_gmm(n_cpu, d, min(k, 64), seed=DATA_SEED % 1000, spread=10.0)
    return data, np.ascontiguousarray(data[:k].T)


def cpu_sample_size(workload, kind, d, k, iterations, budget_s, forced=0):
    """Points of the CPU sample: BASELINE.md §4's N_cpu (1e6; 2e5 for C4) cut down so that `iterations` iterations of the
    single-threaded oracle take about `budget_s` seconds on THIS host (rate probed on a small sample first)."""
    if forced:
        return forced, None
    probe_n = max(4 * k, min(20_000, CPU_SAMPLE_MAX[workload]))
    data, init = _cpu_data(probe_n, d, k)
    fit = _oracle_fit(kind, data, k, init, 3)
    per_point = float(min(fit.step_seconds[1:])) / probe_n
    n = int(budget_s / (iterations * per_point))
    n = max(4 * k, min(CPU_SAMPLE_MAX[workload], n))
    return n, per_point


def cpu_baseline(n_cpu, d, k, steps, warmup, kind="em"):
    """The reference's CPU algorithm on a bounded sample of the same synthetic mixture, single-threaded as the reference
    is: the oracle port (oracle/mlpp_oracle.cpp), timed by its own per-step clock.

    oracle/_ref (the reference's own ML/EM.cpp compiled against the first-party Eigen stand-in) is what pins the port
    (tests/test_oracle_vs_reference.py: bit-identical results), but it is NOT what is timed: the stand-in evaluates every
    Eigen expression eagerly into a heap-allocated temporary (one malloc per point-component pair in EM.cpp:205), which
    real Eigen does not do, so its speed says nothing about the reference.  The port runs the same loops on raw arrays
    and is about 5x faster than the stand-in build: the fair (harder to beat) baseline."""
    import numpy as np
    import oracle
    data, init = _cpu_data(n_cpu, d, k)
    fit = _oracle_fit(kind, data, k, init, warmup + steps)
    secs = fit.step_seconds[warmup:]
    mean = float(np.mean(secs))
    name = "em_fit" if kind == "em" else "kmeans_fit"
    return {"value": n_cpu * k / mean / 1e9, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"oracle {name}, N={n_cpu} D={d} K={k}, {len(secs)} timed iterations after {warmup} warm-up, single thread like the reference",
            "ms_per_step": mean * 1e3, "host_cores_available": os.cpu_count(),
            "pinned_by": "oracle/_ref (reference sources + Eigen stand-in): bit-identical, tests/test_oracle_vs_reference.py" if oracle.ref_available() else "reference property tests only"}


_ALL_CORES_SNIPPET = """
import sys, numpy as np
sys.path.insert(0, {root!r})
import bench
n, d, k, steps, warmup, kind = {n}, {d}, {k}, {steps}, {warmup}, {kind!r}
bench.DATA_SEED = {seed}
data, init = bench._cpu_data(n, d, k)
fit = bench._oracle_fit(kind, data, k, init, warmup + steps)
print(float(np.mean(fit.step_seconds[warmup:])))
"""


def cpu_all_cores(n_cpu, d, k, steps, warmup, kind):
    """SURVEY.md 8(d), optional figure: the reference algorithm has no threads, so "all host cores" means one
    independent single-threaded fit per core, each on its own sample of n_cpu points (what a user could do by hand with
    N-fold sharded data and no statistics exchange).  Aggregate throughput = cores * n_cpu * K / slowest mean step."""
    cores = os.cpu_count() or 1
    procs = [subprocess.Popen([sys.executable, "-c", _ALL_CORES_SNIPPET.format(root=ROOT, n=n_cpu, d=d, k=k, steps=steps, warmup=warmup, kind=kind,
                                                                                seed=DATA_SEED + 1 + i)],
                              stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, env=dict(os.environ, OMP_NUM_THREADS="1"))
             for i in range(cores)]
    means = []
    for p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            return None
        means.append(float(out.strip().splitlines()[-1]))
    return {"value": cores * n_cpu * k / max(means) / 1e9, "unit": UNIT, "cores": cores,
            "sample": f"{cores} independent single-threaded oracle fits, N={n_cpu} points each, {steps} timed iterations after {warmup} warm-up"}


def reference_build_timing(n_ref, d, k, kind, steps=3):
    """For the record next to the port's number: the reference's OWN translation units (oracle/_ref: ML/EM.cpp,
    ML/KMeans.cpp, ... compiled against the first-party Eigen stand-in) on a smaller sample of the same mixture.  Whole
    fit / iterations (the reference has no per-step clock).  None when oracle/_ref was not built (no /root/reference)."""
    import oracle
    if not oracle.ref_available():
        return None
    data, init = _cpu_data(n_ref, d, k)
    t0 = time.perf_counter()
    fit = _oracle_fit(kind, data, k, init, steps, impl="reference")
    seconds = time.perf_counter() - t0
    iterations = max(1, fit.iterations)
    return {"value": n_ref * k * iterations / seconds / 1e9, "unit": UNIT, "cores": 1, "kind": "reference",
            "sample": f"oracle/_ref (the reference's own sources + Eigen stand-in), N={n_ref} D={d} K={k}, whole fit of {iterations} iterations including initialisation",
            "note": "the stand-in evaluates Eigen expressions eagerly into heap temporaries, so this is slower than a real-Eigen build; the port above is the baseline"}


def describe(workload, kind, n_total, d, k):
    algo = "ml::EM full-covariance GMM" if kind == "em" else "ml::Clustering::KMeans Lloyd iterations"
    return f"{workload}: {algo}, N={n_total}, D={d}, K={k}"


def workload_shape(args):
    kind, n_total, d, k = WORKLOADS[args.workload]
    if args.points:
        n_total = args.points
    return kind, n_total, d, k


def run_reference(args):
    """--impl reference: the reference's algorithm on the host CPU: the oracle port, which oracle/_ref (the reference's
    own sources compiled against the Eigen stand-in) pins bit for bit; see cpu_baseline for why the port is what is
    timed.  ml::EM / KMeans are single-threaded, so is this.  Each step is one iteration over a bounded SAMPLE of the
    workload (per-point throughput: the algorithm is exactly O(N) per iteration, Benchmarks/bm_EM.cpp:48)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kind, n_total, d, k = workload_shape(args)
    if args.workload == "c1":
        return run_c1_reference(args)
    budget = args.cpu_budget or 150.0
    n_cpu, per_point = cpu_sample_size(args.workload, kind, d, k, args.steps + args.warmup, budget, args.cpu_sample)
    base = cpu_baseline(n_cpu, d, k, args.steps, args.warmup, kind)
    ref_build = reference_build_timing(max(4 * k, n_cpu // 20), d, k, kind)
    why = "" if n_cpu == CPU_SAMPLE_MAX[args.workload] else (
        f"; BASELINE.md §4's N_cpu={CPU_SAMPLE_MAX[args.workload]} would take {(args.steps + args.warmup) * (per_point or 0) * CPU_SAMPLE_MAX[args.workload]:.0f} s "
        f"for {args.steps + args.warmup} single-threaded iterations on this host, so the sample is cut to a {budget:.0f} s budget")
    line = {
        "impl": "reference", "metric": METRIC if kind == "em" else METRIC_KM, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": base["ms_per_step"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": describe(args.workload, kind, n_total, d, k) + f"; CPU sample of N={n_cpu} points (throughput is per point, O(N) per iteration){why}",
                   "points_total": n_total, "points": n_cpu, "dims": d, "components": k},
        "cpu_baseline": {kk: base[kk] for kk in ("value", "unit", "cores", "kind", "sample", "pinned_by")},
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if ref_build:
        line["reference_build"] = ref_build
    # for the record: what all the host's cores give when the data is sharded by hand over independent single-threaded
    # fits (the reference has no threads of its own; `value` above is the reference as it runs)
    all_cores = cpu_all_cores(max(4 * k, n_cpu // 4), d, k, 3, 1, kind)
    if all_cores:
        line["cpu_baseline"]["all_cores"] = all_cores
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- c1: whole fits

def _c1_fit_gpu(cppyml, data):
    em = cppyml.clustering.EM(3)
    em.set_seed(42)
    em.set_absolute_tolerance(1e-14)
    em.set_relative_tolerance(1e-14)
    em.set_means_initialiser(cppyml.clustering.KPP())
    em.fit(data)
    return em


def _c1_fit_cpu(data):
    import oracle
    return oracle.em_fit(data, 3, seed=42, means_init=oracle.KPP, absolute_tolerance=1e-14, relative_tolerance=1e-14, want_responsibilities=False)


def run_c1_reference(args):
    """BASELINE configuration 1 on the CPU, as Benchmarks/bm_EM.cpp:9-48 defines it: mouse data, N = 10k, K-means++ means,
    tolerances 1e-14; a step is one whole fit."""
    import oracle
    data, _ = oracle.testdata_mouse(WORKLOADS["c1"][1])
    times, iters = [], 0
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        fit = _c1_fit_cpu(data)
        if i >= args.warmup:
            times.append(time.perf_counter() - t0)
        iters = fit.iterations
    mean = sum(times) / len(times)
    n, k = data.shape[0], 3
    value = n * k * iters / mean / 1e9
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": mean * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"c1: ml::EM whole fits, mouse data N={n}, D=2, K=3, K-means++ means, tolerance 1e-14 (Benchmarks/bm_EM.cpp:9-48); a step is one fit of {iters} iterations",
                       "points_total": n, "dims": 2, "components": k, "iterations_per_fit": iters},
            "fits_per_second": 1.0 / mean,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "port", "sample": f"{len(times)} whole oracle fits of the full workload"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_c1(args):
    """BASELINE configuration 1 through the public API: whole `cppyml.clustering.EM(3).fit` calls on the mouse data.  The
    fit is launch-latency bound (N = 10k); value and e2e are the same measurement (every fit uploads its data)."""
    import numpy as np
    import oracle
    from ml_b200 import cabi, import_cppyml
    if cabi.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    cppyml = import_cppyml()
    data, _ = oracle.testdata_mouse(WORKLOADS["c1"][1])
    n, d, k = data.shape[0], 2, 3
    clocks = ClockSampler(0)
    clocks.start()
    for _ in range(max(3, args.warmup)):
        em = _c1_fit_gpu(cppyml, data)
    clocks.mark_begin()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        em = _c1_fit_gpu(cppyml, data)
        _ = em.means, em.mixing_probabilities, em.log_likelihood
    dt = (time.perf_counter() - t0) / args.steps
    clocks.mark_end()
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {"means": em.means, "covariances": [em.covariance(j) for j in range(k)],
                                          "mixing_probabilities": em.mixing_probabilities, "log_likelihood": [em.log_likelihood],
                                          "responsibilities": em.responsibilities, "labels": em.labels_array, "sample_rows": np.arange(n)})
    iters = em.number_iterations
    t0 = time.perf_counter()
    ref = _c1_fit_cpu(data)
    cpu_dt = time.perf_counter() - t0
    value = n * k * iters / dt / 1e9
    dmma, dfma = cabi.fp64_peak(0)
    achieved = n * k * iters * f_em(d) / dt / 1e12
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"c1: ml::EM whole fits, mouse data N={n}, D=2, K=3, K-means++ means, tolerance 1e-14 (Benchmarks/bm_EM.cpp:9-48); a step is one fit of {iters} iterations",
                       "points_total": n, "dims": d, "components": k, "iterations_per_fit": iters, "l2": "10k points fit the L2; the fit is launch-latency bound, not memory bound"},
            "fits_per_second": 1.0 / dt,
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": dmma, "unit": "TFLOP/s", "frac": achieved / dmma,
                         "note": "whole fits including upload and initialisation: launch latency, not the FP64 pipe, bounds this size", "traffic": None,
                         "dmma_peak_tflops": dmma, "dfma_peak_tflops": dfma},
            "cpu_baseline": {"value": n * k * ref.iterations / cpu_dt / 1e9, "unit": UNIT, "cores": 1, "kind": "port",
                             "sample": f"one whole oracle fit of the full workload ({ref.iterations} iterations, {cpu_dt * 1e3:.1f} ms)", "ms_per_step": cpu_dt * 1e3},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": n * d * 8, "d2h_bytes_per_step": (d * k + k) * 8 + iters * 8,
                    "what": "cppyml.clustering.EM(3).fit(data) on a pageable numpy array + means, weights, log-likelihood read back; identical to `value` for this workload"},
            "clocks": clocks.stop(), "gpu_launches": None,
            "parity": {"iterations_gpu": iters, "iterations_cpu": ref.iterations, "ll_gpu": em.log_likelihood, "ll_cpu": ref.log_likelihood}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- device runners (value)

class EmRunner:
    """EM through the C-ABI: a step is expectation + maximisation + statistics exchange + parameter refresh."""
    kernel = "fused E+M kernel (em_small_kernel for D <= 8, em_kernel for D = 16) or the split E / M kernels (D > 16 or K > 32)"

    def __init__(self, cabi, np, data, k, init_means):
        self.np, self.k = np, k
        self.obj = cabi.Em(data, k)
        cov = self.obj.sample_covariance()
        self.obj.set_params(init_means, np.repeat(cov[None], k, axis=0), np.full(k, 1.0 / k))

    def run(self, steps, want=False):
        return self.obj.run_steps(steps, want_ll=want)

    def outputs(self, rows, begin):
        """Parameters after the last step; responsibilities and labels of the last E-step for `rows` (global indices
        held by this rank, ascending)."""
        np = self.np
        means, covs, weights = self.obj.get_params()
        resp, labels = [np.zeros((0, self.k))], [np.zeros(0, dtype=np.uint32)]
        for run in np.split(rows, np.flatnonzero(np.diff(rows) != 1) + 1):
            if run.size:
                r, lab = self.obj.emit_range(int(run[0]), run.size)
                resp.append(r)
                labels.append(lab)
        return {"means": means, "covariances": covs, "mixing_probabilities": weights}, \
               {"responsibilities": np.concatenate(resp), "labels": np.concatenate(labels)}


class KmRunner:
    """K-means through the C-ABI: a step is assignment_step + update_step (KMeans.cpp:80-109)."""
    kernel = "km_assign_kernel (DMMA filter + exact refinement) + km_stats_kernel"

    def __init__(self, cabi, np, data, k, init_means):
        self.np, self.k = np, k
        self.obj = cabi.Km(data, k)
        self.obj.set_centroids(init_means)

    def run(self, steps, want=False):
        out = []
        for _ in range(steps):
            inertia, changed = self.obj.assign()   # the host needs `changed` for KMeans.cpp:85, so every step reads it back
            self.obj.update()
            out.append(inertia)
        return self.np.array(out)

    def outputs(self, rows, begin):
        """Centroids after the last update; labels of the last assignment for `rows` (global indices held by this rank)."""
        return {"centroids": self.obj.get_centroids()}, {"labels": self.obj.get_labels()[rows - begin]}


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    if args.workload == "c1":
        if int(os.environ.get("RANK", "0")) == 0:
            run_c1(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from ml_b200 import cabi, import_cppyml

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    cppyml = import_cppyml()
    uid = uid_host = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        # two communicators: one for the C-ABI context of the resident run, one for the host classes' context (e2e)
        box = [(cabi.nccl_unique_id(), cppyml.distributed.unique_id()) if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        uid, uid_host = box[0]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    kind, n_total, d, k = workload_shape(args)
    Runner = EmRunner if kind == "em" else KmRunner
    ctx = cabi.Context.for_rank(local_rank, rank, world, uid)
    data = cabi.Data.generate_gmm(ctx, n_total, d, min(k, 64), seed=DATA_SEED)
    _, n_local, _ = data.shape
    n_local_max = int(max_over_ranks(float(n_local)))

    # Initial means / centroids: K data points at fixed global indices (0..K-1, held by rank 0), identical on every rank.
    box = [data.download(0, k) if rank == 0 else None]
    if world > 1:
        dist.broadcast_object_list(box, src=0)
    init_rows = np.ascontiguousarray(box[0])            # (K, D)
    init_means = np.ascontiguousarray(init_rows.T)      # (D, K)

    run = Runner(cabi, np, data, k, init_means)

    # ---- value: K steps with the data resident in HBM, CUDA events on the library's stream, max over ranks
    try:
        gpu_uuid = str(torch.cuda.get_device_properties(local_rank).uuid)
    except Exception:
        gpu_uuid = None
    clocks = ClockSampler(local_rank, gpu_uuid)   # every rank samples its own GPU: a straggler GPU sets the max-over-ranks time
    if not args.no_clocks:
        clocks.start()
    warm_trace = run.run(args.warmup, True)
    launches0 = run.obj.launch_count
    direct0 = run.obj.direct_steps if kind == "em" else 0
    run.obj.set_kernel_timing(True)
    barrier()
    clocks.mark_begin()
    ctx.timer_start()
    trace = run.run(args.steps, True)
    ms_total = ctx.timer_stop()
    barrier()
    clocks.mark_end()
    kernel_ms, kernel_launches = run.obj.kernel_time_ms()
    run.obj.set_kernel_timing(False)
    launches = run.obj.launch_count - launches0
    direct_steps = run.obj.direct_steps - direct0 if kind == "em" else 0
    clock_info = clocks.stop()
    my_ms_total = ms_total
    ms_total = max_over_ranks(ms_total)
    ms_per_step = ms_total / args.steps
    value = n_total * k / (ms_per_step * 1e-3) / 1e9
    kernel_ms_avg = max_over_ranks(kernel_ms / max(1, kernel_launches))
    per_rank = None
    if world > 1:
        mine = {"rank": rank, "ms_per_step": my_ms_total / args.steps, "kernel_ms_avg": kernel_ms / max(1, kernel_launches), "points": n_local,
                "sm_mhz": clock_info.get("sm_mhz"), "sm_mhz_min": clock_info.get("sm_mhz_min"), "power_w_max": clock_info.get("power_w_max"),
                "reasons": clock_info.get("reasons")}
        gathered = [None] * world
        dist.all_gather_object(gathered, mine)
        per_rank = gathered
        if rank == 0:
            # the line's clocks are the worst rank's: lowest median SM clock, all reasons seen anywhere
            worst = min((g for g in gathered if g["sm_mhz"] is not None), key=lambda g: g["sm_mhz"], default=None)
            if worst is not None:
                clock_info = dict(clock_info, sm_mhz=worst["sm_mhz"], sm_mhz_min=min(g["sm_mhz_min"] for g in gathered if g["sm_mhz_min"] is not None),
                                  power_w_max=max(g["power_w_max"] for g in gathered if g["power_w_max"] is not None),
                                  reasons=sorted({r for g in gathered for r in (g["reasons"] or [])}),
                                  note=clock_info.get("note", "") + "; every rank sampled its own GPU, sm_mhz is the lowest median over the ranks (per_rank has each)")
    full_trace = np.concatenate([np.asarray(warm_trace, dtype=np.float64), np.asarray(trace, dtype=np.float64)])

    if args.dump_outputs:
        # the parameters are replicated on every rank; the sampled per-point outputs are gathered from the ranks holding them
        begin, _ = cabi.shard_range(n_total, world, rank)
        rows = dump_sample_rows(n_total)
        rows = rows[(rows >= begin) & (rows < begin + n_local)]
        params, points = run.outputs(rows, begin)
        points["sample_rows"] = rows
        if world > 1:
            gathered = [None] * world
            dist.all_gather_object(gathered, points)
            points = {name: np.concatenate([g[name] for g in gathered]) for name in points}
        if rank == 0:
            write_outputs(args.dump_outputs, dict(params, **points, **{"log_likelihood" if kind == "em" else "inertia": trace}))

    # ---- e2e: the plugin call.  cppyml.clustering.EM(k).fit(X) / KMeans(k).fit(X) on a plain pageable numpy array (this
    # rank's rows), then the parameters through the Python properties.  Wall clock, max over ranks.
    e2e = None
    if not args.no_e2e:
        begin, _ = cabi.shard_range(n_total, world, rank)
        host_np = data.download(begin, n_local)            # an ordinary numpy array: pageable memory
        run.obj.close(); data.close(); ctx.close()
        run = data = None
        if world > 1:
            cppyml.distributed.init(local_rank, rank, world, uid_host)
        initialiser = cppyml.clustering.ExplicitCentroids(init_rows)
        fit_steps = max(2, args.steps)   # the classes take no fewer than 2 maximum steps (set_maximum_steps)

        def one_fit():
            barrier()
            t0 = time.perf_counter()
            if kind == "em":
                model = cppyml.clustering.EM(k)
                model.set_means_initialiser(initialiser)
                model.set_absolute_tolerance(0.0)
                model.set_relative_tolerance(0.0)
                model.set_maximum_steps(fit_steps)
                model.fit(host_np)
                results = (model.means, [model.covariance(j) for j in range(k)], model.mixing_probabilities, model.log_likelihood)
                last = model.log_likelihood
                d2h = (d * k + k * d * d + k) * 8
            else:
                model = cppyml.clustering.KMeans(k)
                model.set_centroids_initialiser(initialiser)
                model.set_absolute_tolerance(0.0)
                model.set_maximum_steps(fit_steps)
                model.fit(host_np)
                results = (model.centroids, model.labels_array, model.inertia)
                last = model.inertia
                d2h = d * k * 8 + n_local * 4
            barrier()
            dt = time.perf_counter() - t0
            return dt, last, model.number_iterations, d2h, model, results

        dt, last_e2e, iters_e2e, d2h_results, model, results = one_fit()   # warm-up (allocator pools, page faults of the staging buffers)
        del model, results
        dt, last_e2e, iters_e2e, d2h_results, model, results = one_fit()
        dt = max_over_ranks(dt)
        h2d = n_local * d * 8 + (d * k + (k * d * d + k if kind == "em" else 0)) * 8
        d2h = d2h_results + iters_e2e * 16
        e2e = {"value": n_total * k * iters_e2e / dt / 1e9, "unit": UNIT, "h2d_bytes_per_step": h2d / iters_e2e, "d2h_bytes_per_step": d2h / iters_e2e,
               "fit_seconds": dt, "iterations": iters_e2e,
               "what": ("cppyml.clustering.EM(K).fit(X) with X a pageable C-contiguous numpy array of this rank's rows, ExplicitCentroids start, tolerances 0, "
                        f"maximum_steps={fit_steps}; then means, covariance(k), mixing_probabilities and log_likelihood read through the Python properties"
                        if kind == "em" else
                        "cppyml.clustering.KMeans(K).fit(X) with X a pageable C-contiguous numpy array of this rank's rows, ExplicitCentroids start, tolerance 0, "
                        f"maximum_steps={fit_steps}; then centroids, labels_array (N uint32) and inertia read through the Python properties")
                       + "; wall clock around the whole call sequence, max over ranks; bytes are per iteration (totals / iterations)",
               "last_scalar": last_e2e}
        if kind == "em" and iters_e2e <= len(full_trace):
            # iteration `iters` of the e2e fit is iteration `iters` of the resident run (same data, same start)
            assert abs(last_e2e - float(full_trace[iters_e2e - 1])) <= 1e-12 * abs(last_e2e), "the e2e fit and the resident run disagree"
            e2e["matches_resident_run"] = True
        if kind == "em" and world == 1 and not args.no_responsibilities:
            # declared separately: responsibilities() materialises the N x K matrix on first access (EM.cpp:213-218 leaves it
            # on the host; 25.6 GB at C3), so it is not part of fit() here
            import psutil
            need = n_local * k * 8
            if psutil.virtual_memory().available > 3 * need + (8 << 30):
                t0 = time.perf_counter()
                resp = model.responsibilities
                e2e["responsibilities_seconds"] = time.perf_counter() - t0
                e2e["responsibilities_bytes"] = need
                e2e["responsibilities_row0_sum"] = float(np.asarray(resp[0]).sum())
                del resp
            else:
                e2e["responsibilities_seconds"] = None
                e2e["responsibilities_note"] = "skipped: not enough free host memory for the N x K matrix"
        del model, results

    if rank == 0:
        n_per_gpu = n_local_max
        flops_per_launch = flops_per_iteration(kind, n_per_gpu, d, k)
        achieved = flops_per_launch / (kernel_ms_avg * 1e-3) / 1e12
        try:
            dmma_peak, dfma_peak = cabi.fp64_peak(local_rank)
            peak, peak_source = dmma_peak, "measured live in this run by mlb_selftest_fp64_peak (DMMA.8x8x4 chain, the instruction the kernels issue); MEASURED_PEAKS.json has no FP64 figure"
        except Exception as exc:   # noqa: BLE001
            dmma_peak = dfma_peak = None
            peak, peak_source = FP64_PEAK_TFLOPS_FALLBACK, f"fallback profiles/fp64_peaks_r01.json (live measurement failed: {exc})"
        peaks_file = os.path.join(ROOT, "MEASURED_PEAKS.json")
        hbm_peak = json.load(open(peaks_file))["hbm_gbs"] if os.path.exists(peaks_file) else 6650.0
        bytes_per_point = 8 * d if kind == "em" else 8 * d + 4
        hbm_gbs = n_per_gpu * bytes_per_point / (kernel_ms_avg * 1e-3) / 1e9
        line = {
            "metric": METRIC if kind == "em" else METRIC_KM, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": describe(args.workload, kind, n_total, d, k) + f" (fixed total; {n_per_gpu} points on the fullest of {world} GPU(s)), "
                                   "initial means = data points 0..K-1" + (", initial covariances = sample covariance" if kind == "em" else ""),
                       "points_total": n_total, "points_per_gpu": n_per_gpu, "dims": d, "components": k,
                       "parallelism": f"points sharded over {world} GPU(s), one ncclAllGather of the sufficient statistics per iteration",
                       "l2": f"input is {n_per_gpu * d * 8 / 1e6:.0f} MB per GPU, larger than the 126 MB L2; no flush needed between iterations",
                       "iterations_per_second": 1e3 / ms_per_step},
            "roofline": {"bound": "tensor", "pipe": "FP64 tensor pipe (DMMA, mma.sync.m8n8k4.f64); shares the SM's FP64 unit with DFMA",
                         "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "peak_source": peak_source,
                         "dmma_peak_tflops": dmma_peak, "dfma_peak_tflops": dfma_peak,
                         "kernel": Runner.kernel + (f"; {direct_steps} of the {args.steps} timed steps were routed to the direct-difference kernels (kappa > 3e5)"
                                                    if kind == "em" else ""),
                         "timed_steps_on_direct_kernels": direct_steps, "kernel_ms_avg": kernel_ms_avg, "kernel_launches_timed": kernel_launches,
                         "flops_per_launch": flops_per_launch,
                         "flops_per_point_component": f_em(d) if kind == "em" else 3 * d + 1,
                         "hbm_achieved_gbs": hbm_gbs, "hbm_peak_gbs": hbm_peak, "hbm_frac": hbm_gbs / hbm_peak,
                         "traffic": None},
            "clocks": clock_info,
            "gpu_launches": launches,
            "last_scalar": float(trace[-1]),
        }
        for name in ("traffic_r02.json", "traffic_r01.json"):
            prof = os.path.join(ROOT, "profiles", name)
            if os.path.exists(prof):
                entry = json.load(open(prof)).get(args.workload)
                if entry is not None:
                    if "captured_points" in entry:
                        # ncu capture of one launch at `captured_points` points: the kernels stream the points once and
                        # write per-chunk partials, both linear in N, so the capture is scaled to this launch's points
                        scale = n_per_gpu / entry["captured_points"]
                        entry = {"bytes_per_launch": (entry["dram_read"] + entry["dram_write"]) * scale, "dram_read": entry["dram_read"] * scale,
                                 "dram_write": entry["dram_write"] * scale, "algorithmic_bytes": entry["algorithmic_bytes_per_point"] * n_per_gpu,
                                 "source": entry["source"] + f"; scaled by {scale:.3f} to the {n_per_gpu} points of this launch"}
                    line["roofline"]["traffic"] = entry
                    break
        if per_rank is not None:
            line["per_rank"] = per_rank
        if e2e is not None:
            line["e2e"] = e2e
        if world == 1 and not args.no_cpu:
            budget = args.cpu_budget or 25.0
            n_cpu, _ = cpu_sample_size(args.workload, kind, d, k, 4, budget, args.cpu_sample)
            line["cpu_baseline"] = cpu_baseline(n_cpu, d, k, 3, 1, kind)
            all_cores = cpu_all_cores(max(4 * k, n_cpu // 4), d, k, 3, 1, kind)
            if all_cores:
                line["cpu_baseline"]["all_cores"] = all_cores
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
