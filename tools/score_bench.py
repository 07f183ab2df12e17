"""Times scoring (mlb_em_score_fitted, mlb_em_score) next to the EM step and predict, on generated data.

    python tools/score_bench.py [--out FILE] [em:N:D:K ...]      default: C3 (em:100000000:16:32) and C4 (em:20000000:64:64)

Per case, in one process on the first GPU, after three warm-up steps:
  step_ms            one mlb_em_step (the step graph, as a fit runs it)
  score_fitted_ms    mlb_em_score_fitted, mean only
  score_fitted_out_ms  the same with every point's log p(x) copied to host memory
  score_new / predict  mlb_em_score and mlb_em_predict (responsibilities and labels) on the same 4M host points
Every timing is a host clock around calls that end in a device synchronisation, the median of `reps` calls.  The data
(12.8 GB at C3, 10.2 GB at C4) is far larger than the 126 MB L2.  The GPU's name and power limit are read in the same run.
"""
import argparse
import json
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, ".")
from ml_b200 import cabi

NEW_POINTS = 4 << 20


def timed(fn, reps):
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        out.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(out)), out


def case(ctx, n, d, k, reps=5):
    data = cabi.Data.generate_gmm(ctx, n, d, k, seed=7)
    em = cabi.Em(data, k)
    cov = em.sample_covariance()
    em.set_params(data.download(0, k).T, np.repeat(cov[None], k, axis=0), np.full(k, 1.0 / k))
    em.run_steps(3)
    r = dict(n=n, d=d, k=k, config=em.kernel_config())
    r["step_ms"], r["step_ms_all"] = timed(em.step, reps)
    r["route"] = em.conditioning()[1]
    em.score_fitted(want_log_densities=False)
    r["score_fitted_ms"], r["score_fitted_ms_all"] = timed(lambda: em.score_fitted(want_log_densities=False), reps)
    r["score_fitted_out_ms"], r["score_fitted_out_ms_all"] = timed(em.score_fitted, 3)
    pts = np.ascontiguousarray(data.download(0, NEW_POINTS))
    em.score(pts)
    em.predict(pts)
    r["new_points"] = NEW_POINTS
    r["score_new_ms"], _ = timed(lambda: em.score(pts), reps)
    r["score_new_mean_only_ms"], _ = timed(lambda: em.score(pts, want_log_densities=False), reps)
    r["predict_new_ms"], _ = timed(lambda: em.predict(pts), reps)
    r["score_new_mpoints_per_s"] = NEW_POINTS / r["score_new_ms"] / 1e3
    r["predict_new_mpoints_per_s"] = NEW_POINTS / r["predict_new_ms"] / 1e3
    r["score_fitted_over_step"] = r["score_fitted_ms"] / r["step_ms"]
    em.close()
    data.close()
    return r


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("cases", nargs="*", default=["em:100000000:16:32", "em:20000000:64:64"])
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    ctx = cabi.Context(1)
    results = []
    for c in args.cases:
        _, n, d, k = c.split(":")
        r = case(ctx, int(n), int(d), int(k))
        r["gpu"] = gpu
        print(json.dumps(r), flush=True)
        results.append(r)
    ctx.close()
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"gpu": gpu, "results": results}, f, indent=1)
