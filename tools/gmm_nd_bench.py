"""Time the mixture fits of two features (nr_gmm_fit) at the joint CLI's 2-D phasing shape, against scikit-learn.

Shape (config 2): 5 000 reads' (repeat 1, repeat 2) sizes x 100 bootstrap draws = 500 000 two-feature samples, fitted with
GaussianMixture(n, covariance_type='diag', n_init=10) for n = 1..4 -- once through nanorepeat_b200.mixture.GaussianMixture
(the drop-in, on the GPU) and once through scikit-learn on this host's CPU.  Then a batch of 2 000 problems of 3 000
samples each through nr_gmm_fit in one call.  Prints one JSON line (and writes it to --out):
  - wall_s: host clock around the call, median of --reps calls after one warm-up (includes the upload and the read-back);
  - kernel_ms: summed durations of the fit kernel's launches in one call, from torch.profiler's CUDA activity;
  - sklearn_s: scikit-learn's wall time for the same fit (one run);
  - the GPU's name, power limit and maximum SM clock (nvidia-smi), read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def locus_samples(seed, n_reads=5000, error_rate=0.07):
    """two alleles of an HTT-like locus (CAG 17 / CCG 10 and CAG 55 / CCG 7), bootstrapped 100 times"""
    rng = np.random.default_rng(seed)
    half = n_reads // 2
    sizes = np.concatenate([np.column_stack([rng.normal(17, 0.6, half), rng.normal(10, 0.4, half)]),
                            np.column_stack([rng.normal(55, 1.5, n_reads - half), rng.normal(7, 0.4, n_reads - half)])])
    sim = np.tile(sizes, (100, 1))
    return sim + error_rate * (10 + sim) * rng.standard_normal(sim.shape)


def kernel_ms(fn):
    """summed CUDA time of the fit kernel's launches during fn()"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(e.device_time_total for e in prof.key_averages() if "fit_nd_kernel" in e.key) / 1000.0


def wall(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--max-n", type=int, default=4)
    ap.add_argument("--no-sklearn", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    from nanorepeat_b200 import engine
    from nanorepeat_b200.mixture import GaussianMixture
    engine.init(0)
    res = dict(tool="gmm_nd_bench", gpu=gpu_info(), shape="500000 x 2 samples, n_init=10", per_n=[])
    X = locus_samples(1)
    for n in range(1, a.max_n + 1):
        def ours():
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                return GaussianMixture(n_components=n, covariance_type="diag", n_init=10, random_state=n).fit(X)
        row = dict(n=n, wall_s=wall(ours, a.reps), kernel_ms=kernel_ms(ours))
        g = ours()
        row.update(n_iter=g.n_iter_, lower_bound=g.lower_bound_)
        if not a.no_sklearn:
            from sklearn.mixture import GaussianMixture as SkGM
            t0 = time.perf_counter()
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                sk = SkGM(n_components=n, covariance_type="diag", n_init=10, random_state=n).fit(X)
            row.update(sklearn_s=time.perf_counter() - t0, sklearn_n_iter=int(sk.n_iter_), sklearn_lower_bound=float(sk.lower_bound_))
            row["speedup"] = row["sklearn_s"] / row["wall_s"]
        res["per_n"].append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)

    # a batch of 2 000 problems of 3 000 two-feature samples (two components each) in one call
    rng = np.random.default_rng(2)
    probs = [np.column_stack([rng.normal(rng.choice([17.0, 40.0], 3000), 1.5), rng.normal(rng.choice([7.0, 10.0], 3000), 0.8)])
             for _ in range(2000)]
    p = engine.GmmParams(max_components=2, n_init=10, seed=3)

    def batch():
        return engine.gmm_fit(p, probs, [2] * len(probs), 2)
    res["batch"] = dict(problems=2000, samples=3000, n=2, n_init=10, wall_s=wall(batch, a.reps), kernel_ms=kernel_ms(batch))
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
