"""Compare `bench.py --dump-outputs` directories of the regression workloads statistically (NUTS trajectories diverge
chaotically once the rounding of the gradient differs, so two builds are not compared file for file):

* mean tree depth of each dump, and the difference between the first two;
* per coefficient, the mean and sd of the dumped draws against the closed-form posterior N(m, V) of the workload
  (float64 from the same X, y): |mean - m| in units of the Monte-Carlo standard error, and the sd ratio.

The MCSE treats the chains as independent and the iterations of one chain as correlated: it is taken from the spread
of the per-chain means.

    python tools/compare_dumps.py DIR_A DIR_B [--workload c4]
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SHAPES = {"c4": (100000, 1000), "c3": (10000, 100)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("dirs", nargs="+")
    ap.add_argument("--workload", default="c4", choices=sorted(SHAPES))
    args = ap.parse_args()
    import mlx_mcmc_b200 as B
    from mlx_mcmc_b200 import workloads as W
    n, d = SHAPES[args.workload]
    _, _, meta = W.regression(B.ns, n, d, seed=0)
    m, V = W.regression_posterior(meta)
    sd = np.sqrt(np.diag(V))
    out = {"workload": args.workload, "dumps": {}}
    depths = []
    for p in args.dirs:
        draws = np.load(os.path.join(p, "draws.npy")).astype(np.float64)      # [iters, chains, D]
        depth = np.load(os.path.join(p, "tree_depth.npy")).astype(np.float64)
        depths.append(float(depth.mean()))
        chain_means = draws.mean(0)                                            # [chains, D]
        mean = chain_means.mean(0)
        mcse = chain_means.std(0, ddof=1) / np.sqrt(chain_means.shape[0])
        z = np.abs(mean - m) / mcse
        ratio = draws.reshape(-1, d).std(0, ddof=1) / sd
        out["dumps"][p] = {"iters": draws.shape[0], "chains": draws.shape[1], "mean_tree_depth": depths[-1],
                           "max_abs_mean_err_in_mcse": float(z.max()), "coefficients_within_4_mcse": float((z <= 4).mean()),
                           "sd_ratio_min": float(ratio.min()), "sd_ratio_max": float(ratio.max()),
                           "sd_ratio_median": float(np.median(ratio)),
                           "coefficients_sd_ratio_in_0.97_1.03": float(((ratio >= 0.97) & (ratio <= 1.03)).mean())}
    if len(depths) >= 2:
        out["mean_tree_depth_difference"] = depths[1] - depths[0]
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
