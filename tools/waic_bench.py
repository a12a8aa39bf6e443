"""WAIC at the C4 shape on one GPU: what a b2m_loglik_stats call over many posterior draws costs.

    python tools/waic_bench.py [--n 100000 --d 1000 --chains 4096 --samples 64 500 --reps 3 --out result.json]

Three models over the same design matrix shape -- the C4 regression (Normal likelihood) in the tf32 and in the fp16
encoding, and the logistic regression (Bernoulli-logit) -- each with draws [S, 4096, D] around the posterior mode
(exact posterior draws are not needed for timing).  Per (model, S): one untimed call, then `--reps` calls timed with CUDA
events around the whole b2m_loglik_stats call, and the per-batch contraction (K5 with the statistics epilogue,
tc_gemm_kernel MODE 4 / 5) timed from the library's own launch events (b2m_profile, K5 slot).  Reported: seconds per
call, draws x observations per second, the executed tensor flops 2 * 3 * rows * N * Dp (three MMAs per 3xTF32 / 3xFP16
product) over the contraction time, and, for comparison, the sampler's K5 time per 4096 rows (one value+gradient of
4096 chains in the streaming form, same process).  The card's name, power limit and SM clocks are read with a
read-only nvidia-smi query in the same process.  Prints one JSON object (and writes it to --out)."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=100000)
ap.add_argument("--d", type=int, default=1000)
ap.add_argument("--chains", type=int, default=4096)
ap.add_argument("--samples", type=int, nargs="+", default=[64, 500])
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--out", default=None)
args = ap.parse_args()

import mlx_mcmc_b200 as B
from mlx_mcmc_b200 import _cabi, workloads as W
from mlx_mcmc_b200.engine import compile_model

assert torch.cuda.is_available(), "tools/waic_bench.py measures on a CUDA device"
lib = _cabi.load()


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        name, power, clock, clock_max = [s.strip() for s in out[torch.cuda.current_device()].split(",")]
        return {"name": name, "power_limit": power, "sm_clock": clock, "sm_clock_max": clock_max}
    except Exception as e:   # the measurement stands; the record says why the card details are missing
        return {"name": torch.cuda.get_device_name(), "power_limit": None, "sm_clock": None, "error": str(e)}


def profile_k5():
    out = (ctypes.c_double * 4)()
    _cabi.check(lib.b2m_profile_read(out))
    return out[0], int(out[1])


def call(model, draws, obs, n_obs, out):
    idx = (ctypes.c_int32 * len(obs))(*obs)
    _cabi.check(lib.b2m_loglik_stats(model.handle, ctypes.c_void_p(draws.data_ptr()), draws.shape[0] * draws.shape[1],
                                     idx, len(obs), ctypes.c_void_p(out.data_ptr()), n_obs,
                                     ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))


rows = []
info = gpu_info()
for kind, path in (("normal", "tc"), ("normal", "tc16"), ("logit", "auto")):
    make = W.regression if kind == "normal" else W.logistic_regression
    fn, init, meta = make(B.ns, args.n, args.d, seed=0)
    model = compile_model(fn, init, cache=False, glm_path=path)
    stream_model = compile_model(fn, init, cache=False, glm_path=path, glm_form="stream")
    obs = model.traced.observation_terms()
    n_obs = args.n
    Dp = (args.d + 63) // 64 * 64
    center = torch.from_numpy(meta.beta_true.astype(np.float32)).cuda()
    # the sampler's K5 per 4096 rows: one value+gradient in the streaming form
    th = (center[None, :] + 0.01 * torch.randn(args.chains, args.d, device="cuda")).contiguous()
    stream_model.logp_grad(th)
    lib.b2m_profile(1)
    for _ in range(args.reps):
        stream_model.logp_grad(th)
    k5_ms, k5_n = profile_k5()
    lib.b2m_profile(0)
    del th, stream_model
    for S in args.samples:
        draws = center[None, None, :] + 0.01 * torch.randn(S, args.chains, args.d, device="cuda")
        out = torch.empty((n_obs, 3), dtype=torch.float64, device="cuda")
        call(model, draws, obs, n_obs, out)                      # warm-up: module load, tensor maps, workspaces
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        lib.b2m_profile(1)
        e0.record()
        for _ in range(args.reps):
            call(model, draws, obs, n_obs, out)
        e1.record()
        torch.cuda.synchronize()
        gemm_ms, gemm_n = profile_k5()
        lib.b2m_profile(0)
        call_s = e0.elapsed_time(e1) / 1e3 / args.reps
        n_rows = S * args.chains
        Np = (args.n + 255) // 256 * 256
        flops = 2.0 * 3.0 * n_rows * Np * Dp
        row = {"kind": kind, "glm_path": model.glm_path, "S": S, "chains": args.chains, "draws": n_rows, "N": n_obs,
               "D": args.d, "s_per_call": call_s, "draw_obs_per_s": n_rows * n_obs / call_s,
               "contraction_s_per_call": gemm_ms / 1e3 / args.reps, "contraction_launches_per_call": gemm_n / args.reps,
               "tensor_tflops_executed": flops / (gemm_ms / 1e3 / args.reps) / 1e12,
               "contraction_share_of_call": gemm_ms / 1e3 / args.reps / call_s,
               "sampler_k5_ms_per_4096_rows": k5_ms / max(k5_n, 1) * 4096 / args.chains,
               "stats_k5_ms_per_4096_rows": gemm_ms / max(gemm_n, 1)}
        rows.append(row)
        print(json.dumps(row), flush=True)
        del draws, out
    del model
    torch.cuda.empty_cache()

result = {"gpu": info, "n": args.n, "d": args.d, "reps": args.reps, "rows": rows}
print(json.dumps(result))
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
