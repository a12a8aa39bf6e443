"""Logistic against linear regression at the C4 shape on one GPU: what the Bernoulli-logit epilogue of K5 costs.

    python tools/logistic_bench.py [--n 100000 --d 1000 --chains 4096 --rounds 6 --out result.json]

Both models -- sum Normal(0, 10)(beta) + sum Bernoulli(logits = X @ beta)(y), and the C4 regression with a Normal
likelihood -- are built in one process and run NUTS (pooled step size adapted first, max tree depth 10), alternating
one timed step of 8 transitions each, `--rounds` times.  Per step: CUDA events around the b2m_nuts_run call (with an L2
flush before it, untimed), the leapfrog gradient evaluations it took, and the K5 / K6 time per evaluation from the
library's own launch events (b2m_profile).  The card's name, power limit and maximum SM clock are read with a read-only
nvidia-smi query in the same process.  Then `--probe-d` times one value+gradient of each kind at a small D (same N
and chains): K5's MMAs shrink with D, its epilogue does not, so the difference between the kinds there is the
epilogue's cost.  Prints one JSON object (and writes it to --out)."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=100000)
ap.add_argument("--d", type=int, default=1000)
ap.add_argument("--chains", type=int, default=4096)
ap.add_argument("--rounds", type=int, default=6)
ap.add_argument("--iters", type=int, default=8, help="NUTS transitions per timed step")
ap.add_argument("--adapt", type=int, default=40)
ap.add_argument("--path", default="auto")
ap.add_argument("--probe-d", type=int, default=64,
                help="also time one value+gradient of both kinds at this D (same N and chains): K5's epilogue cost does "
                     "not depend on D, its MMAs do")
ap.add_argument("--out", default=None)
args = ap.parse_args()

import mlx_mcmc_b200 as B
from mlx_mcmc_b200 import _cabi, workloads as W
from mlx_mcmc_b200.engine import ChainState, compile_model, launch_nuts

assert torch.cuda.is_available(), "tools/logistic_bench.py measures on a CUDA device"
lib = _cabi.load()


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        name, power, clock = [s.strip() for s in out[torch.cuda.current_device()].split(",")]
        return {"name": name, "power_limit": power, "sm_clock_max": clock}
    except Exception as e:   # the measurement stands; the record says why the card details are missing
        return {"name": torch.cuda.get_device_name(), "power_limit": None, "sm_clock_max": None, "error": str(e)}


def setup(kind, seed=1234):
    """model, chains around the posterior mode, pooled dual averaging (untimed)"""
    n, d, C = args.n, args.d, args.chains
    if kind == "logistic":
        fn, init, meta = W.logistic_regression(B.ns, n, d, seed=0)
        curv, eps0 = 0.3 * n, 1.8e-3      # X'X ~ n I; the Bernoulli weights sigma (1 - sigma) are ~0.2 here, at most 0.25
    else:
        fn, init, meta = W.regression(B.ns, n, d, seed=0)
        curv, eps0 = float(n), 8e-4
    # the Normal reference runs the streaming form: the comparison is of the two kinds' K5 epilogues over the same K6
    model = compile_model(fn, init, cache=False, glm_path=args.path, glm_form="stream")
    th = torch.zeros(128, d, device="cuda")
    for _ in range(30):                    # gradient ascent with a step below 1 / (largest curvature): the mode
        _, g = model.logp_grad(th)
        th = th + g / curv
    gen = torch.Generator(device="cuda")
    gen.manual_seed(seed)
    theta = th[0][None, :] + torch.randn(C, d, device="cuda", generator=gen) / (0.7 * curv) ** 0.5
    st = ChainState(model, theta.contiguous(), eps0)
    st.da_state[:, 0] = 0.0
    st.da_state[:, 1] = 1.0
    st.da_state[:, 2] = float(np.log(np.float32(10.0 * eps0)))
    launch_nuts(st, args.adapt, 6, _cabi.ADAPT_POOLED, _cabi.COMPAT_CORRECT, 0.65, seed, 0)
    st.step_size.copy_(st.da_state[:, 1])
    torch.cuda.synchronize()
    return {"model": model, "st": st, "it": args.adapt, "seed": seed, "glm_path": model.glm_path,
            "depths": torch.empty((args.iters, C), dtype=torch.int32, device="cuda"), "rounds": []}


flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")


def timed_step(m):
    st = m["st"]
    leaves0 = int(st.n_leaves.sum().item())
    four = (ctypes.c_double * 4)()
    flush.fill_(1)
    torch.cuda.synchronize()
    lib.b2m_profile(1)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    launch_nuts(st, args.iters, 10, _cabi.ADAPT_NONE, _cabi.COMPAT_CORRECT, 0.65, m["seed"], m["it"], depths=m["depths"])
    b.record()
    torch.cuda.synchronize()
    lib.b2m_profile_read(four)
    lib.b2m_profile(0)
    m["it"] += args.iters
    ms = a.elapsed_time(b)
    evals = int(st.n_leaves.sum().item()) - leaves0
    launches5, launches6 = max(four[1], 1.0), max(four[3], 1.0)
    m["rounds"].append({"ms": ms, "grad_evals": evals, "grad_evals_per_s": evals / (ms / 1e3),
                        "k5_ms_per_launch": four[0] / launches5, "k6_ms_per_launch": four[2] / launches6,
                        "k5_launches": int(four[1]), "k6_launches": int(four[3]),
                        "mean_depth": float(m["depths"].float().mean().item())})


t0 = time.time()
info = gpu_info()
models = {k: setup(k) for k in ("logistic", "normal")}
for m in models.values():              # warm-up step of each, untimed
    timed_step(m)
    m["rounds"].clear()
for _ in range(args.rounds):
    for m in models.values():
        timed_step(m)

res = {"tool": "tools/logistic_bench.py", "gpu": info, "shape": {"n": args.n, "d": args.d, "chains": args.chains,
       "transitions_per_step": args.iters, "max_tree_depth": 10, "adapt": "pooled dual averaging", "flush": "256 MB before each step"}}
for k, m in models.items():
    r = m["rounds"]
    med = lambda key: float(np.median([x[key] for x in r]))   # noqa: E731
    res[k] = {"glm_path": m["glm_path"], "step_size": float(m["st"].step_size[0]),
              "grad_evals_per_s_median": med("grad_evals_per_s"),
              "k5_ms_per_eval_median": med("k5_ms_per_launch"), "k6_ms_per_eval_median": med("k6_ms_per_launch"),
              "mean_depth": med("mean_depth"), "rounds": r}
res["k5_logistic_over_normal"] = res["logistic"]["k5_ms_per_eval_median"] / res["normal"]["k5_ms_per_eval_median"]
res["k6_logistic_over_normal"] = res["logistic"]["k6_ms_per_eval_median"] / res["normal"]["k6_ms_per_eval_median"]


def probe(kind, d):
    """K5 / K6 ms of one value+gradient at [chains, d] x [d, n], median of 5 (b2m_profile events)"""
    fn, init, _ = (W.logistic_regression if kind == "logistic" else W.regression)(B.ns, args.n, d, seed=0)
    # the Normal reference runs the streaming form: the comparison is of the two kinds' K5 epilogues over the same K6
    model = compile_model(fn, init, cache=False, glm_path=args.path, glm_form="stream")
    gen = torch.Generator(device="cuda")
    gen.manual_seed(3)
    theta = (0.05 * torch.randn(args.chains, d, device="cuda", generator=gen)).contiguous()
    model.logp_grad(theta)
    k5, k6 = [], []
    for _ in range(5):
        four = (ctypes.c_double * 4)()
        flush.fill_(1)
        torch.cuda.synchronize()
        lib.b2m_profile(1)
        model.logp_grad(theta)
        lib.b2m_profile_read(four)
        lib.b2m_profile(0)
        k5.append(four[0] / max(four[1], 1.0))
        k6.append(four[2] / max(four[3], 1.0))
    return {"d": d, "glm_path": model.glm_path, "k5_ms": float(np.median(k5)), "k6_ms": float(np.median(k6))}


if args.probe_d > 0:
    res["probe"] = {k: probe(k, args.probe_d) for k in ("logistic", "normal")}
    res["probe"]["k5_extra_ms_logistic"] = res["probe"]["logistic"]["k5_ms"] - res["probe"]["normal"]["k5_ms"]
    res["k5_extra_ms_logistic_at_full_d"] = (res["logistic"]["k5_ms_per_eval_median"] - res["normal"]["k5_ms_per_eval_median"])
res["wall_s"] = time.time() - t0
print(json.dumps(res))
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
