"""Time one batched value+gradient of the regression model and check it against float64, per evaluation form
(streaming: K5 + K6; Gram: one contraction against X^T X).  One JSON line per form.

    python tools/glm_eval_bench.py --n 100000 --d 1000 --chains 4096 [--path tc|tc16|simt] [--form gram,stream] [--check 64]
"""
import argparse
import json
import math
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=100000)
ap.add_argument("--d", type=int, default=1000)
ap.add_argument("--chains", type=int, default=4096)
ap.add_argument("--path", default="auto")
ap.add_argument("--form", default="auto", help="comma-separated list of auto | stream | gram")
ap.add_argument("--check", type=int, default=64)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--spread", type=float, default=0.01)
ap.add_argument("--where", default="near", choices=["near", "zero", "mixed"],
                help="chains near the mode (beta* + spread z), all at 0, or half and half")
args = ap.parse_args()

import mlx_mcmc_b200 as B
from mlx_mcmc_b200 import workloads as W
from mlx_mcmc_b200.engine import compile_model

fn, init, meta = W.regression(B.ns, args.n, args.d, seed=0)
for form in args.form.split(","):
    t0 = time.time()
    model = compile_model(fn, init, cache=False, glm_path=args.path, glm_form=form)
    torch.cuda.synchronize()
    build_s = time.time() - t0
    print(f"model built in {build_s:.2f}s ({model.glm_form} form)", file=sys.stderr)
    rng = np.random.default_rng(1)
    theta = (meta.beta_true[None, :] + args.spread * rng.standard_normal((args.chains, args.d))).astype(np.float32)
    if args.where == "zero":
        theta[:] = 0.0
    elif args.where == "mixed":
        theta[::2] = 0.0
    t = torch.from_numpy(theta).cuda()
    lp, g = model.logp_grad(t)
    torch.cuda.synchronize()
    times = []
    for _ in range(args.reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        lp, g = model.logp_grad(t)
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    ms = float(np.median(times))
    # GEMM-only time of the same calls: CUDA events inside the library around every K5 / K6 launch
    import ctypes
    from mlx_mcmc_b200 import _cabi
    lib = _cabi.load()
    four = (ctypes.c_double * 4)()
    lib.b2m_profile(1)
    for _ in range(args.reps):
        lp, g = model.logp_grad(t)
    lib.b2m_profile_read(four)
    lib.b2m_profile(0)
    k5 = four[0] / max(four[1], 1)
    k6 = four[2] / max(four[3], 1)
    flops = 4.0 * args.n * args.d * args.chains
    # executed tensor flops per evaluation (3 MMAs per product of the hi/lo split) of the form's contraction(s), against the
    # dense data-sheet rate of one B200 (fp16 2250 TFLOP/s, tf32 1125 TFLOP/s, at up to 1000 W): a share of peak of the
    # GEMM launches alone
    Dp = (args.d + 63) // 64 * 64
    Np = (args.n + 255) // 256 * 256
    executed = 3 * 2 * Dp * Dp * args.chains if model.glm_form == "gram" else 3 * 4 * Np * Dp * args.chains
    peak = 2250.0 if model.glm_path == "tc16" else 1125.0
    out = {"glm_path": model.glm_path, "glm_form": model.glm_form, "build_s": build_s,
           "gemm_ms": {"K5": k5, "K6": k6, "both": k5 + k6},
           "executed_tflop_per_eval": executed / 1e12, "gemm_executed_tflops": executed / ((k5 + k6) * 1e-3) / 1e12,
           "datasheet_dense_peak_tflops": peak, "gemm_frac_of_datasheet_peak": executed / ((k5 + k6) * 1e-3) / 1e12 / peak,
           "where": args.where, "n": args.n, "d": args.d, "chains": args.chains, "path": args.path, "ms_per_eval": ms, "all_ms": times,
           "useful_tflops": flops / ms / 1e9, "grad_evals_per_s": args.chains / ms * 1e3,
           "logical_GBps": 4.0 * args.n * args.d * args.chains / ms / 1e6}
    if args.check:
        k = args.check
        X, y, b = meta.X.astype(np.float64), meta.y.astype(np.float64), theta[:k].astype(np.float64)
        r = y[None, :] - b @ X.T
        lp64 = (-0.5 * (r ** 2).sum(1) - args.n * 0.5 * math.log(2 * math.pi)
                - 0.5 * (b ** 2).sum(1) / 100.0 - args.d * (0.5 * math.log(2 * math.pi) + math.log(10.0)))
        g64 = r @ X - b / 100.0
        out["logp_rel_err"] = float(np.max(np.abs(lp[:k].cpu().numpy() - lp64) / np.abs(lp64)))
        out["grad_normwise_err"] = float(np.max(np.abs(g[:k].cpu().numpy() - g64)) / np.max(np.abs(g64)))
        out["grad_scale"] = float(np.max(np.abs(g64)))
        # per-chain norm-wise error (each chain against its own gradient scale): the strictest reading of check 1
        out["grad_err_per_chain_max"] = float(np.max(np.max(np.abs(g[:k].cpu().numpy() - g64), axis=1) / np.max(np.abs(g64), axis=1)))
    print(json.dumps(out))
    del model
