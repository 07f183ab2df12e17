"""Times the K-means distance and inertia calls (mlb_km_transform, mlb_km_transform_range, mlb_km_score_fitted) next to
predict and the assignment step, on generated data, on the first GPU.

    python tools/km_transform_bench.py [--out FILE] [--n N]        default N = 100M (the C5 shape: D = 32, K = 256)

Recorded:
  c5          at D = 32, K = 256 with N resident points: one assign step, score_fitted, transform and predict on 1M and
              4M host points, transform_range of 4M resident points;
  widths      transform and predict on 1M host points at D = 2, 16 and 100 (K = 256, 4M resident points);
  kernel      km_transform_kernel alone (torch.profiler, in a run of its own after the timed calls): its device time per
              1M points against both of its bounds, the m K 8 output bytes over the HBM data-sheet bandwidth (7.7 TB/s)
              and 2 m K D FP64 operations over the DFMA peak mlb_selftest_fp64_peak measures.  Each (point, centroid,
              dimension) costs a DADD (x - c) and a DFMA, two issues of the FP64 pipe where the DFMA peak counts one
              instruction as two operations, so the kernel's FP64 floor is twice that bound (fp64_issue_bound_ms); the
              larger of it and the output bound applies.
Every call timing is a host clock around calls that end in a device synchronisation, the median of `reps` calls.  The
resident data (25.6 GB at C5) is far larger than the 126 MB L2.  The GPU's name and power limit are read in the same run.
"""
import argparse
import json
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, ".")
from ml_b200 import cabi

HBM_BYTES_PER_S = 7.7e12   # NVIDIA HGX B200 data sheet, one GPU


def timed(fn, reps):
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        out.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(out)), out


def kernel_ms(fn, name="km_transform_kernel"):
    """Device time (ms) and launch count of the kernels called `name` during fn(), from a torch.profiler run."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    total, count = 0.0, 0
    for evt in prof.key_averages():
        if name in evt.key:
            total += getattr(evt, "self_device_time_total", 0) or getattr(evt, "self_cuda_time_total", 0)
            count += evt.count
    return total / 1e3, count


def fitted_km(ctx, n, d, k, steps=2):
    data = cabi.Data.generate_gmm(ctx, n, d, k, seed=7)
    km = cabi.Km(data, k)
    km.set_centroids(np.ascontiguousarray(data.download(0, k).T))
    for _ in range(steps):
        km.assign()
        km.update()
    return data, km


def c5(ctx, n, reps):
    d, k = 32, 256
    data, km = fitted_km(ctx, n, d, k)
    r = dict(n=n, d=d, k=k, config=km.kernel_config())
    km.assign()
    km.score_fitted()
    r["assign_ms"], r["assign_ms_all"] = timed(km.assign, reps)
    r["score_fitted_ms"], r["score_fitted_ms_all"] = timed(km.score_fitted, reps)
    for m in (1 << 20, 4 << 20):
        pts = np.ascontiguousarray(data.download(n - m, m))
        km.transform(pts)
        km.predict(pts)
        r[f"transform_{m >> 20}M_ms"], _ = timed(lambda: km.transform(pts), reps)
        r[f"predict_{m >> 20}M_ms"], _ = timed(lambda: km.predict(pts), reps)
    m = 4 << 20
    km.transform_range(0, m)
    r["transform_range_4M_ms"], _ = timed(lambda: km.transform_range(0, m), reps)
    pts = np.ascontiguousarray(data.download(n - (1 << 20), 1 << 20))
    r["kernel"] = kernel_report(ctx, km, pts)
    r["kernel"]["transform_call_ms"] = r["transform_1M_ms"]
    r["kernel"]["outside_kernel_ms"] = r["transform_1M_ms"] - r["kernel"]["kernel_ms"]
    km.close()
    data.close()
    return r


def kernel_report(ctx, km, pts):
    m, d, k = pts.shape[0], pts.shape[1], km.k
    ms, count = kernel_ms(lambda: km.transform(pts))
    _, dfma = cabi.fp64_peak(0)
    bytes_bound = m * k * 8 / HBM_BYTES_PER_S * 1e3
    flops_bound = 2.0 * m * k * d / (dfma * 1e12) * 1e3
    issue_bound = 2.0 * flops_bound   # DADD + DFMA per element: 2 m K D FP64 instructions at dfma / 2 instructions per second
    return dict(m=m, d=d, k=k, launches=count, kernel_ms=ms, dfma_tflops=dfma, output_bytes=m * k * 8, fp64_ops=2 * m * k * d,
                bytes_bound_ms=bytes_bound, fp64_bound_ms=flops_bound, fp64_issue_bound_ms=issue_bound,
                bound="fp64 issue" if issue_bound > bytes_bound else "bytes",
                share_of_bound=max(bytes_bound, issue_bound) / ms if ms > 0 else None,
                achieved_tbytes_per_s=m * k * 8 / (ms * 1e-3) / 1e12 if ms > 0 else None,
                achieved_fp64_tflops=2.0 * m * k * d / (ms * 1e-3) / 1e12 if ms > 0 else None)


def width(ctx, d, reps, k=256, n=4 << 20):
    data, km = fitted_km(ctx, n, d, k, steps=1)
    pts = np.ascontiguousarray(data.download(0, 1 << 20))
    km.transform(pts)
    km.predict(pts)
    r = dict(d=d, k=k, m=pts.shape[0], config=km.kernel_config())
    r["transform_ms"], _ = timed(lambda: km.transform(pts), reps)
    r["predict_ms"], _ = timed(lambda: km.predict(pts), reps)
    r["kernel"] = kernel_report(ctx, km, pts)
    km.close()
    data.close()
    return r


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--n", type=int, default=100_000_000)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    ctx = cabi.Context(1)
    result = {"gpu": gpu, "c5": c5(ctx, args.n, args.reps)}
    print(json.dumps(result["c5"]), flush=True)
    result["widths"] = []
    for d in (2, 16, 100):
        result["widths"].append(width(ctx, d, args.reps))
        print(json.dumps(result["widths"][-1]), flush=True)
    ctx.close()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
