#!/usr/bin/env python
"""Benchmark of the sampling hot path (BASELINE.json metric: leapfrog grad-evals/sec, min-ESS/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c4|c3|c2|c1|c5] [--scaling strong|weak] [--impl reference]
                    [--dump-outputs DIR]

Default workload = BASELINE.json's Target configuration (configs[3], "C4"): Bayesian linear regression with 1000
coefficients and 100,000 observations, NUTS, 4096 chains in lock-step (it fits one GPU: X is 400 MB).  With N GPUs the
default is the configuration as BASELINE.json writes it -- the SAME 4096 chains with the observations sharded over the
ranks (strong scaling): every rank contracts its 100000 / N rows for all chains, K6's epilogue stores each finished
gradient tile into its owner's peer window over NVLink, the owner finishes / advances its 4096 / N chains and publishes
the next leaf's packed rows to every rank.  `--scaling weak` shards the chains instead (4096 per GPU, no data-path
collective).  The other configurations
(`--workload`, and the `other_workloads` object of the default line) are C3 (100 x 10K regression, NUTS, 1024 chains),
C2 (examples/04 event-rate model, 65,536 HMC chains), C1 and C5 (examples/03, 1M Metropolis chains).

A *step*:  GLM workloads (c4, c3) -- one b2m_nuts_run call = 4 (c4) / 16 (c3) NUTS transitions of every chain of the rank
           (momentum draw, iterative tree build with one lock-step value+gradient per leaf = two tcgen05 GEMMs on
           hi/lo split operands, U-turn / slice bookkeeping, draws written to HBM);
           pointwise workloads (c2, c1, c5) -- one launch of the persistent kernel covering ITERS whole iterations.
A *grad-eval* = one value-and-gradient of log_prob for one chain (= one leapfrog step / NUTS leaf; masked lanes of
the lock-step are not counted).  Metropolis counts value evaluations.

The JSON line carries
  value        whole-job grad-evals/s over the timed region (CUDA events, inputs resident in HBM, max over ranks)
  e2e          the same metric through the public API (`nuts(...)` / `hmc(...)`) with HOST initial values and draws
               copied back to pinned host memory inside the timed region
  roofline     dominant kernel against its bound: GLM -> tensor pipe (executed tf32 flops of the two GEMM kernels, each
               timed with CUDA events on the launching stream, vs a measured tf32 cuBLAS peak); pointwise -> HBM bytes
  cpu_baseline the oracle restatement (reference source semantics on a torch-CPU stand-in for MLX, which cannot be
               installed here) on the box's host cores, on a bounded sample of the same workload
`--impl reference` times that same restatement alone (rank 0 only), same metric / unit / config.
"""
from __future__ import annotations

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

import numpy as np  # noqa: E402

WORKLOADS = {
    "c4": dict(kind="glm", n=100000, d=1000, chains=4096, eps0=8e-4, adapt_iters=40, max_tree_depth=10, iters=8,
               desc="Bayesian linear regression 1000 params x 100K obs (README 'Large'), NUTS, 4096 chains/GPU"),
    "c3": dict(kind="glm", n=10000, d=100, chains=1024, eps0=5e-3, adapt_iters=60, max_tree_depth=10, iters=16,
               desc="Bayesian linear regression 100 params x 10K obs (README 'Medium'), NUTS, 1024 chains/GPU"),
    "c2": dict(kind="pointwise", model="c2_event_rate", method="hmc", chains=65536, step_size=0.1, L=10, iters=100,
               desc="examples/04_event_rates Gamma/Exponential rate model, 65536 chains/GPU, HMC eps0=0.1 L=10"),
    "c1": dict(kind="pointwise", model="c1_normal", method="hmc", chains=65536, step_size=0.01, L=10, iters=50,
               desc="examples/01-02 Normal(mu,sigma) posterior, 100 obs, HMC L=10, 65536 chains/GPU"),
    "c5": dict(kind="pointwise", model="c5_ab_test", method="metropolis", chains=1048576, proposal_scale=0.02, iters=100,
               desc="examples/03_ab_testing Beta A/B model, 1M Metropolis chains/GPU"),
}
METRIC = "leapfrog_grad_evals_per_sec"
UNIT = "grad-evals/s"
# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full captures (profiles/)
NCU_TRAFFIC = {"c4": {"bytes": 0.564e9 + 1.616e9 + 3.281e9 + 0.126e9,
                      "source": "profiles/r02_tc_gemm_c4_ncu_summary.md, later capture (K5 0.56 GB read + 1.62 GB written, K6 3.28 GB read + "
                                "0.13 GB written with the column-tile-fastest tile order; tensor pipe active 92.6 % / 92.6 % of the "
                                "elapsed cycles; the opt-in concurrent K5 || K6 launch moves 1.09 GB: "
                                "profiles/r02_tc_gemm_fused_c4_ncu_summary.md)"}}


# issue-side evidence of the pointwise kernels from the committed ncu captures (profiles/): the bound of these paths
PW_ISSUE = {"c2": {"source": "profiles/r02_hmc_kernel_c2_specialised_ncu_summary.md",
                   "specialised": {"issue_slots_busy_pct": 64.9, "ipc_per_sm": 2.41, "warp_occupancy_pct": 19.2, "waves": 0.49,
                                   "registers": 72, "thread_instructions_per_grad_eval": 368},
                   "interpreter": {"issue_slots_busy_pct": 50.1, "ipc_per_sm": 1.93, "warp_occupancy_pct": 20.4, "waves": 0.43,
                                   "registers": 64, "thread_instructions_per_grad_eval": 625}}}


# ----------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx_ = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx_) if mx_ else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------- CPU baseline (oracle port)
def _mode_numpy(X, y, iters=25):
    """posterior mode of the regression by Richardson iteration on the normal equations (X'X ~ N I for this data)"""
    n = X.shape[0]
    b = np.zeros(X.shape[1], dtype=np.float64)
    Xd = X.astype(np.float64)
    for _ in range(iters):
        b = b + (Xd.T @ (y.astype(np.float64) - Xd @ b) - b / 100.0) / n
    return b.astype(np.float32)


_CPU_GLM_CACHE = {}


def _cpu_glm(wl_name: str, threads: int, n_iter: int, seed: int = 0):
    """`n_iter` NUTS transitions of ONE chain of the regression workload on the oracle restatement, started at the
    posterior mode with the workload's step size (no adaptation), all host threads for the matvecs."""
    import torch
    from oracle.ns import Tape, ns as ons, samplers
    from mlx_mcmc_b200 import workloads as W
    wl = WORKLOADS[wl_name]
    torch.set_num_threads(max(threads, 1))
    if wl_name not in _CPU_GLM_CACHE:          # synthetic data + starting point: built once per process, not timed
        fn, _, meta = W.regression(ons, wl["n"], wl["d"], seed=0)
        _CPU_GLM_CACHE[wl_name] = (fn, {"beta": _mode_numpy(meta.X, meta.y)})
    fn, init = _CPU_GLM_CACHE[wl_name]
    tape = Tape()
    t0 = time.perf_counter()
    samplers.nuts_port(fn, init, num_samples=n_iter, num_warmup=1, step_size=wl["eps0"], adapt_step_size=False,
                       max_tree_depth=wl["max_tree_depth"], key=ons.mx.random.key(seed), tape=tape)
    dt = time.perf_counter() - t0
    return tape.leapfrogs, dt, tape.grad_evals


def _ref_compute_ess(x):
    """the estimator of examples/06_nuts_comparison.py:22-41, restated (oracle/refport/diagnostics.py holds the pinned copy)"""
    from oracle.refport.diagnostics import compute_ess
    return float(compute_ess(np.asarray(x, dtype=np.float64)))


def _cpu_chain(args):
    """one chain of the oracle restatement of a pointwise workload (runs in a worker process); returns
    (evals, seconds, mx.grad calls, min over parameters of the reference-estimator ESS of the kept draws)"""
    wl_name, seed, n_warm, n_samp = args
    from oracle.ns import Tape, ns as ons, samplers
    from mlx_mcmc_b200 import workloads as W
    wl = WORKLOADS[wl_name]
    fn, init, _ = W.ALL_SMALL[wl["model"]](ons)
    tape = Tape()
    t0 = time.perf_counter()
    if wl["method"] == "hmc":
        out = samplers.hmc_port(fn, init, num_samples=n_samp, num_warmup=n_warm, step_size=wl["step_size"],
                                num_leapfrog_steps=wl["L"], key=ons.mx.random.key(seed), tape=tape)
        evals = tape.leapfrogs
    else:
        out = samplers.run_port(fn, init, num_samples=n_samp, num_warmup=n_warm, method="metropolis",
                                proposal_scale=wl["proposal_scale"], random_seed=seed, tape=tape)
        evals = n_samp + n_warm
    dt = time.perf_counter() - t0
    try:
        ess = min(_ref_compute_ess(np.asarray(v)) for v in out[0].values())
    except Exception:
        ess = float("nan")
    return evals, dt, tape.grad_evals, ess


def cpu_baseline(wl_name: str, cores: int, scale: float = 1.0, full_length: bool = False):
    """The oracle port on `cores` host cores on a bounded sample of the workload.  Returns the cpu_baseline object.
    GLM: one chain, the matvecs use `cores` torch threads.  Pointwise: one independent chain per core (the
    reference is a single Python thread per chain).  `full_length`: the example's own run length (1000 warm-up + 5000
    draws) so that min-ESS/s (examples/06_nuts_comparison.py:22-41 estimator) is the reference's own figure."""
    wl = WORKLOADS[wl_name]
    t0 = time.perf_counter()
    extra = {}
    if wl["kind"] == "glm":
        n_iter = max(1, int(round((10 if wl_name == "c4" else 60) * scale)))   # ~10-15 s of host work at scale 1
        evals, busy, grads = _cpu_glm(wl_name, cores, n_iter)
        sample = (f"1 chain x {n_iter} NUTS transition(s) (+1 warm-up transition) from the posterior mode, step size "
                  f"{wl['eps0']}, no adaptation, on the oracle restatement (reference source semantics on a torch-CPU "
                  f"stand-in for MLX) with {cores} torch threads; one leaf counted as one grad-eval (the reference spends "
                  f"2 mx.grad + 2 value traces per leaf: {grads} mx.grad calls here)")
        extra["min_ess_per_s"] = None
        extra["min_ess_note"] = (f"{n_iter} transitions carry no autocorrelation estimate; the full-length single-chain runs "
                                 "with the reference's estimator are in cpu_baseline.full_length (C1, C2, C5)")
    else:
        n_warm, n_samp = (1000, 5000) if full_length else (max(10, int(150 * scale)), max(20, int(350 * scale)))
        jobs = [(wl_name, 1000 + i, n_warm, n_samp) for i in range(cores)]
        if cores == 1:
            res = [_cpu_chain(jobs[0])]
        else:
            import multiprocessing as mp
            with mp.get_context("spawn").Pool(cores) as pool:
                res = pool.map(_cpu_chain, jobs)
        evals, busy, grads = sum(r[0] for r in res), max(r[1] for r in res), sum(r[2] for r in res)
        ess = [r[3] for r in res if r[3] == r[3]]
        sample = (f"{cores} chain(s) x ({n_warm} warm-up + {n_samp} draws) of the same model/sampler settings on the "
                  f"oracle restatement (reference source semantics on a torch-CPU stand-in for MLX); one leapfrog step "
                  f"counted as one grad-eval (the reference spends 2 mx.grad + value traces per step: {grads} mx.grad "
                  f"calls here)")
        extra["min_ess_per_s"] = (sum(ess) / busy) if ess else None
        extra["min_ess_note"] = ("sum over chains of min-over-parameters ESS (examples/06_nuts_comparison.py:22-41 estimator) / "
                                 "wall time including warm-up")
    wall = time.perf_counter() - t0
    out = {"value": evals / busy, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample + f"; wall {wall:.1f}s"}
    out.update(extra)
    return out


def _full_length_job(name):
    """worker: one chain, the example's full run length, for cpu_baseline.full_length"""
    r = cpu_baseline(name, 1, 1.0, full_length=True)
    return name, {"grad_evals_per_s": r["value"], "min_ess_per_s": r["min_ess_per_s"], "sample": r["sample"]}


def cpu_full_length(names=("c1", "c2", "c5")):
    """C1 / C2 / C5 at the reference examples' own length (1000 + 5000, BASELINE.md section 3), one chain each, run side
    by side on separate host cores: grad-evals/s and min-ESS/s of the reference arithmetic (oracle port)."""
    import multiprocessing as mp
    with mp.get_context("spawn").Pool(len(names)) as pool:
        return dict(pool.map(_full_length_job, list(names)))


def reference_arm(args, wl, config):
    """The reference's CPU implementation of the path on the box's host cores (`--impl reference`): the oracle
    restatement -- pinned bit-equal to the unmodified reference source by oracle/make_golden.py; MLX itself is not
    installable here and /root/reference does not exist on the GPU box, so the unmodified source cannot run there --
    with all the host threads it can use.  W warm-up + exactly K timed steps, each a bounded sample of the workload;
    `run` says what one step was."""
    cores = os.cpu_count() or 1
    if wl["kind"] == "pointwise":
        cores = min(cores, 32)
    W_, K = max(args.warmup, 0), args.steps
    # a step sized so that K of them end within a few minutes: C4 ~ 1 s (2 transitions), C3 / pointwise ~ 2-4 s
    scale = 0.2 if args.workload == "c4" else 0.3
    for _ in range(min(W_, 2)):
        cpu_baseline(args.workload, cores, scale)
    vals, t0, per = [], time.perf_counter(), None
    for _ in range(K):
        per = cpu_baseline(args.workload, cores, scale)
        vals.append(per["value"])
    v = float(np.mean(vals))
    per["value"] = v
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": len(vals),
            "warmup": W_, "ms_per_step": 1e3 * (time.perf_counter() - t0) / len(vals), "higher_is_better": True,
            "scaling": config.pop("_scaling", "weak"), "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "run": {"what": "reference arm: CPU, no GPU, none of this repo's kernels", "chains": 1 if wl["kind"] == "glm" else cores,
                    "kind": "port", "cores": cores, "one_step": per["sample"]},
            "cpu_baseline": per, "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if "min_ess_per_s" in per:
        line["min_ess_per_s"] = per["min_ess_per_s"]
    emit(line)
    return 0


# ----------------------------------------------------------------------------------------- helpers
_T0 = time.perf_counter()


def log(msg):
    print(f"[bench {time.perf_counter() - _T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def tf32_peak_probe(torch):
    """cuBLAS tf32 GEMM 8192^3 on fp32 inputs: best of 6 (burst) -- the measured tensor-pipe peak for kind::tf32."""
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        a = torch.randn(8192, 8192, device="cuda")
        b = torch.randn(8192, 8192, device="cuda")
        (a @ b)
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(6):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            (a @ b)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return 2 * 8192 ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


class Timed:
    """K CUDA-event-timed steps with an L2 flush before each (not timed)."""

    def __init__(self, torch, steps):
        self.torch = torch
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        self.ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]

    def run(self, step_fn):
        for a, b in self.ev:
            self.flush.fill_(1)
            a.record()
            step_fn()
            b.record()

    def total_ms(self):
        return float(sum(a.elapsed_time(b) for a, b in self.ev))


DUMP_BYTES = 48 << 20      # C4's draws are 131 MB a step: about 1500 of its 4096 chains fit


def dump_outputs(out_dir, draws, depths=None):
    """--dump-outputs: what the last timed step returned, as float32 .npy files -- the draws [iters, chains, D] of a
    fixed sample of chains (numpy default_rng(0), as many as keep the whole dump within DUMP_BYTES; all of them when
    they fit) and the NUTS tree depth [iters, chains] of every chain.  The inputs of a run depend only on the command
    line, so two builds of the project can be compared file for file."""
    os.makedirs(out_dir, exist_ok=True)
    out = {}
    if depths is not None:
        out["tree_depth"] = depths.float().cpu().numpy()
    iters, C, D = draws.shape
    left = DUMP_BYTES - sum(a.nbytes for a in out.values()) - 4096
    keep = min(C, left // (4 * iters * D))
    if keep < C:
        import torch
        idx = np.sort(np.random.default_rng(0).choice(C, keep, replace=False))
        draws = draws.index_select(1, torch.from_numpy(idx).to(draws.device))
    out["draws"] = draws.float().cpu().numpy()
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log(f"outputs of the last timed step in {out_dir}: " + ", ".join(f"{k}{list(a.shape)}" for k, a in out.items()))


# ----------------------------------------------------------------------------------------- GLM workloads (c4, c3)
def glm_setup(torch, B, wl, C, chain_offset, seed, obs_sharded=False, peer=False):
    """model + chains started in the posterior's typical set + dual-averaging warm-up (all untimed).
    obs_sharded: every rank holds all C chains (same ids, same seed) and a row shard of (X, y); peer: with the peer
    window of the fused gradient exchange attached."""
    from mlx_mcmc_b200 import _cabi, dist as D_, workloads as W
    from mlx_mcmc_b200.engine import ChainState, compile_model, launch_nuts
    fn, init, meta = W.regression(B.ns, wl["n"], wl["d"], seed=0)
    model = D_.compile_obs_sharded(fn, init, peer_chains=C if peer else None) if obs_sharded else compile_model(fn, init)
    N, D = wl["n"], wl["d"]
    # posterior mode by Richardson iteration on the device gradient (X'X ~ N I for this synthetic X)
    th = torch.zeros(128, D, device="cuda")
    for _ in range(25):
        _, g = model.logp_grad(th)
        th = th + g / N
    mode = th[0].clone()
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1234 + chain_offset)
    theta = mode[None, :] + torch.randn(C, D, device="cuda", generator=gen) / (N ** 0.5)
    st = ChainState(model, theta.contiguous(), wl["eps0"], chain_offset)
    st.da_state[:, 0] = 0.0
    st.da_state[:, 1] = 1.0
    st.da_state[:, 2] = float(np.log(np.float32(10.0 * wl["eps0"])))
    log(f"{wl['desc'][:40]}: model on device, mode found; adapting step sizes ({wl['adapt_iters']} iterations)")
    # adaptation runs with a shallower tree cap: the reference's dual averaging starts at 10 x eps0 and
    # overshoots down before settling, and a depth-10 tree of lock-step leaves is ~9 s at C4
    launch_nuts(st, wl["adapt_iters"], min(6, wl["max_tree_depth"]), _cabi.ADAPT_POOLED, _cabi.COMPAT_CORRECT, 0.65, seed, 0)
    st.step_size.copy_(st.da_state[:, 1])
    torch.cuda.synchronize()
    log(f"adapted: median step size {float(st.step_size.median()):.3e}")
    return fn, meta, model, st, mode


def glm_roofline(torch, four, leaves, N, D, C, total_ms, model, wl_name, rows_note=""):
    """roofline of the dominant kernels: every GEMM launch of the timed region was timed with CUDA events inside the
    library (b2m_profile).  N = observation rows this rank contracts (all of them, or its shard)."""
    peaks = load_peaks()
    tf32_probe = tf32_peak_probe(torch)
    k5_ms, k5_n, k6_ms, k6_n = [float(x) for x in four]
    # flops of one contraction for the batch the timed launches ran on (compacted batches are smaller: use the leaves)
    useful_per_gemm = 2.0 * N * D * (leaves / max(k5_n, 1))
    k5 = k5_ms / max(k5_n, 1)
    k6 = k6_ms / max(k6_n, 1)
    # concurrent launch (tc_gemm_fused_kernel: K5 and K6 as two roles of ONE kernel): its events are recorded under K5
    # and there is no K6 entry; the launch time is then the time of both contractions
    fused = k6_n == 0 and k5_n > 0
    both = k5 + k6
    executed_tflops = 3 * 2 * useful_per_gemm / (both * 1e-3) / 1e12
    f16 = getattr(model, "glm_path", "tc") == "tc16"
    bf16_sus = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 0.0)) or 0.0)
    bf16_half = 0.5 * bf16_sus
    if f16:      # kind::f16 MMAs: fp16 and bf16 share the tensor rate; the kernels run inside a long step => sustained figure
        peak = bf16_sus if bf16_sus else 2.0 * tf32_probe
        peak_source = (f"bf16_tflops_sustained of MEASURED_PEAKS.json = {bf16_sus:.1f} (kind::f16 runs at the bf16 rate; "
                       f"cuBLAS tf32 probe in this run = {tf32_probe:.1f})")
    else:
        peak = max(tf32_probe, bf16_half) if bf16_half else tf32_probe
        peak_source = (f"max(cuBLAS tf32 8192^3 probe in this run = {tf32_probe:.1f}, 0.5 x bf16_tflops_sustained of "
                       f"MEASURED_PEAKS.json = {bf16_half:.1f})")
    enc = "fp16" if f16 else "tf32"
    alg_bytes = 4.0 * (N * D + N + 2 * C * D)
    traffic = NCU_TRAFFIC.get(wl_name) if not rows_note else None
    return {
        "bound": "tensor", "achieved": executed_tflops, "peak": peak, "unit": "TFLOP/s", "frac": executed_tflops / peak,
        "traffic": traffic["bytes"] if traffic else None,
        "kernel": ("tc_gemm_fused_kernel: K5 (M = (beta-beta0) X^T + residual epilogue) on half of the CTA pairs || K6 (G = R X) on "
                   "the other half, one slab of observations behind, residual operand in an L2-resident ring" if fused else
                   "tc_gemm_kernel<256,RESID> (K5: M = (beta-beta0) X^T + residual epilogue) + tc_gemm_kernel<*,PLAIN|PUSH> (K6: G = R X)"),
        "avg_launch_ms": ({"K5||K6": both, "K5": both / 2, "K6": both / 2} if fused else {"K5": k5, "K6": k6}),
        "launches_timed": int(k5_n + k6_n),
        "gemm_share_of_step": (k5_ms + k6_ms) / total_ms,
        "encoding": f"3x{enc.upper()} split (hi.hi + hi.lo + lo.hi), fp32 accumulate in TMEM with round-to-nearest promotion",
        "executed_tflops": ({"K5||K6": executed_tflops} if fused else
                            {"K5": 3 * useful_per_gemm / (k5 * 1e-3) / 1e12, "K6": 3 * useful_per_gemm / (k6 * 1e-3) / 1e12}),
        "useful_tflops": 2 * useful_per_gemm / (both * 1e-3) / 1e12,
        "peak_source": peak_source,
        "algorithmic_bytes_per_eval": alg_bytes,
        "logical_GBps_per_chain_view": 2 * useful_per_gemm / (both * 1e-3) / 1e9,
        "hbm_peak_GBps": float(peaks.get("hbm_gbs", 6650.0)),
        "traffic_source": traffic["source"] if traffic else None,
        "rows": rows_note or f"all {N} observation rows on this GPU",
        "note": "achieved = executed tensor flops (3 MMAs per useful product: the hi/lo split is what holds the 1e-5 gate; "
                "north_star names 3xTF32, the fp16 split is the same construction at twice the MMA rate and is checked "
                "against float64 at full size in tests/test_gpu_glm_tc.py) of one lock-step value+gradient / (K5 + K6 "
                "launch time); useful_tflops = 4 N D C / t.  "
                "logical_GBps_per_chain_view = C x 4 N D / t is the north-star's 'HBM roofline per gradient eval' reading "
                "(each chain would stream X once per gradient if it ran alone); the batch actually moves "
                "algorithmic_bytes_per_eval."}


def bench_glm(torch, dist, B, lib, args, wl, wl_name, rank, world, local_rank, full=True):
    import mlx_mcmc_b200.core as mx
    from mlx_mcmc_b200 import _cabi
    from mlx_mcmc_b200.diagnostics import ess_geyer
    from mlx_mcmc_b200.engine import launch_nuts
    C = args.chains or wl["chains"]
    chain_offset = rank * C
    seed = 1234
    N, D, MD = wl["n"], wl["d"], wl["max_tree_depth"]
    fn, meta, model, st, mode = glm_setup(torch, B, wl, C, chain_offset, seed)
    it0 = [wl["adapt_iters"]]
    ITERS = wl["iters"]                     # NUTS transitions per step (one b2m_nuts_run call)
    draws = torch.empty((ITERS, C, D), dtype=torch.float32, device="cuda")
    depths = torch.empty((ITERS, C), dtype=torch.int32, device="cuda")

    def one_step():
        launch_nuts(st, ITERS, MD, _cabi.ADAPT_NONE, _cabi.COMPAT_CORRECT, 0.65, seed, it0[0], draws=draws, depths=depths)
        it0[0] += ITERS

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    warm = max(args.warmup, 3)
    timed = Timed(torch, args.steps)
    for _ in range(warm):
        timed.flush.fill_(1)
        one_step()
    barrier()
    clocks = ClockSampler(local_rank)
    clocks.start()
    leaves0 = int(st.n_leaves.sum().item())
    n0 = lib.b2m_launch_count()
    import ctypes
    ten = (ctypes.c_double * 10)()
    lib.b2m_profile(1)          # CUDA events around every GEMM / state-kernel launch of the timed region, on the launching stream
    barrier()
    timed.run(one_step)
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, draws, depths)
    lib.b2m_profile_read_ex(ten)
    lib.b2m_profile(0)
    four = list(ten)[:4]
    launches = lib.b2m_launch_count() - n0
    leaves = int(st.n_leaves.sum().item()) - leaves0
    total_ms = timed.total_ms()
    mean_depth = float(depths.float().mean().item())

    # ---- e2e: public API, HOST initial values in, draws back to pinned host memory, inside the timed region
    S_e2e, e2e_steps = ITERS, max(2, min(args.steps, 3))
    host_theta = st.theta.cpu().numpy().copy()                    # [C, D] per-chain starting points (host memory)
    host_init = {"beta": np.zeros(D, dtype=np.float32)}
    eps_host = float(st.step_size.median().item())

    def api_call(k):
        return B.nuts(fn, host_init, num_samples=S_e2e, num_warmup=1, step_size=eps_host, max_tree_depth=MD,
                      adapt_step_size=False, key=mx.random.key(100 + k), num_chains=C, chain_offset=chain_offset,
                      compat="correct", return_info=True, theta0=host_theta)

    api_call(0)
    barrier()
    t0 = time.perf_counter()
    e2e_evals = 0
    for k in range(e2e_steps):
        _, _, info = api_call(k + 1)
        e2e_evals += info.grad_evals
    barrier()
    e2e_s = time.perf_counter() - t0
    clock_info = clocks.stop()
    log(f"timed {args.steps} steps of {ITERS} transitions: {total_ms / args.steps:.1f} ms/step, mean depth {mean_depth:.2f}; e2e {e2e_s:.1f}s")

    t = torch.tensor([total_ms, e2e_s], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([leaves, e2e_evals, launches], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    total_ms, e2e_s = float(t[0]), float(t[1])
    leaves_all, e2e_all, launches_all = float(cnt[0]), float(cnt[1]), int(cnt[2])
    value = leaves_all / (total_ms * 1e-3)
    out = {"value": value, "ms_per_step": total_ms / args.steps, "gpu_launches": launches_all, "clocks": clock_info,
           "e2e": {"value": e2e_all / e2e_s, "unit": UNIT, "h2d_bytes_per_step": C * D * 4, "d2h_bytes_per_step": S_e2e * C * D * 4,
                   "call": f"nuts(num_warmup=1, num_samples={S_e2e}, num_chains={C}, adapt_step_size=False) with [C, D] host "
                           f"initial values; draws returned as host numpy"},
           "config_extra": {"chains_per_gpu": C, "iters_per_step": ITERS, "mean_tree_depth": mean_depth,
                            "grad_evals_per_step_per_gpu": leaves / args.steps,
                            "adapted_step_size_median": eps_host}}
    if rank != 0:
        return out

    out["roofline"] = glm_roofline(torch, four, leaves, N, D, C, total_ms, model, wl_name)
    both = out["roofline"]["avg_launch_ms"]["K5"] + out["roofline"]["avg_launch_ms"]["K6"]
    out["issue"] = {"grad_evals_per_s_per_gpu": value / world, "lockstep_eval_ms": both, "nuts_step_ms": total_ms / args.steps,
                    "state_kernel_ms_avg": ten[4] / max(ten[5], 1), "state_kernel_launches": int(ten[5])}

    log("roofline pass done")
    if full and not args.no_ess:
        out["ess"] = glm_ess_public_run(torch, B, wl, fn, C, chain_offset)
    return out


def bench_glm_strong(torch, dist, B, lib, args, wl, wl_name, rank, world, local_rank):
    """N > 1, BASELINE.json configs[3] as written: the SAME C chains in total, observations sharded over the ranks
    (strong scaling).  Timed path: sliced state through the peer window -- per gradient, K6's epilogue stores every
    finished [256, D] tile into its owner's window over NVLink while the next tile's MMAs run, the owner sums the
    per-source slots in rank order, advances its C / N chains and publishes the next leaf's packed fp16 rows to every
    rank; flags with release / acquire semantics at system scope, no NCCL call inside the sampling loop."""
    import ctypes
    import mlx_mcmc_b200.core as mx
    from mlx_mcmc_b200 import _cabi
    from mlx_mcmc_b200.engine import ChainState, compile_model, launch_nuts
    C = args.chains or wl["chains"]
    seed = 1234
    N, D, MD = wl["n"], wl["d"], wl["max_tree_depth"]
    ITERS = wl["iters"]
    if C % (128 * world) or C % 256:
        raise SystemExit(f"--scaling strong needs chains % (128 x ranks) == 0 and % 256 == 0 (got {C} on {world} ranks)")
    exchange_note = None
    try:
        fn, meta, model, st, mode = glm_setup(torch, B, wl, C, 0, seed, obs_sharded=True, peer=True)
        SLICE = _cabi.SLICE_PEER
    except RuntimeError as e:       # the peer window could not be set up on this box (the error is raised on every rank):
        log(f"peer window unavailable ({e}); timing the NCCL reduce-scatter form instead")      # say so, never silently
        fn, meta, model, st, mode = glm_setup(torch, B, wl, C, 0, seed, obs_sharded=True, peer=False)
        SLICE = _cabi.SLICE_NCCL
        exchange_note = f"peer window unavailable on this box ({e}): NCCL reduce-scatter / all-gather per gradient"
    rows_local = next(int(a_.shape[0]) for a_ in model._arrays if a_.dim() == 2)   # this rank's rows of X
    it0 = [wl["adapt_iters"]]
    draws = torch.zeros((ITERS, C, D), dtype=torch.float32, device="cuda")
    depths = torch.zeros((ITERS, C), dtype=torch.int32, device="cuda")

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    def step(mode_):
        launch_nuts(st, ITERS, MD, _cabi.ADAPT_NONE, _cabi.COMPAT_CORRECT, 0.65, seed, it0[0], draws=draws, depths=depths,
                    slice_state=mode_)
        it0[0] += ITERS

    def leaves_all():       # sliced: every rank counts its own chains; replicated: every rank counts all of them
        return st.n_leaves.sum().double().reshape(1)

    # ---- parity self-check (untimed), part 1: observation-sharded log p / gradient against the unsharded model
    parity = {}
    gen = torch.Generator(device="cuda")
    gen.manual_seed(99)
    probe = (mode[None, :] + torch.randn(256, D, device="cuda", generator=gen) / (N ** 0.5)).contiguous()
    lp_s, g_s = model.logp_grad(probe)                      # collective: NCCL all-reduce of the partials
    if rank == 0:
        from mlx_mcmc_b200 import workloads as W
        fn_full, init_full, _ = W.regression(B.ns, N, D, seed=0)
        full = compile_model(fn_full, init_full, cache=False)
        lp_f, g_f = full.logp_grad(probe)
        parity["obs_sharded_logp_rel_err"] = float(((lp_s - lp_f).abs() / lp_f.abs()).max())
        parity["obs_sharded_grad_normwise_err"] = float((g_s - g_f).abs().max() / g_f.abs().max())
        del full
        torch.cuda.empty_cache()
    # part 2: one transition of every chain, peer exchange vs the replicated NCCL all-reduce, from identical states
    saved = (st.theta.clone(), st.n_leaves.clone(), st.n_accept.clone(), st.n_diverge.clone())
    d1 = torch.zeros((1, C, D), device="cuda")
    launch_nuts(st, 1, MD, _cabi.ADAPT_NONE, _cabi.COMPAT_CORRECT, 0.65, seed, 10 ** 6, draws=d1, slice_state=_cabi.SLICE_OFF)
    rep_leaves = int((st.n_leaves - saved[1]).sum().item())
    for t_, s_ in zip((st.theta, st.n_leaves, st.n_accept, st.n_diverge), saved):
        t_.copy_(s_)
    d2 = torch.zeros((1, C, D), device="cuda")
    launch_nuts(st, 1, MD, _cabi.ADAPT_NONE, _cabi.COMPAT_CORRECT, 0.65, seed, 10 ** 6, draws=d2, slice_state=SLICE)
    peer_leaves = (st.n_leaves - saved[1]).sum().double().reshape(1)
    dist.all_reduce(d2)                                     # merge the slices (each rank wrote its own chains' rows)
    dist.all_reduce(peer_leaves)
    # Energies of this model are ~N/2 = 5e4, where float32 resolves 0.004: the two summation orders (NCCL ring vs
    # per-source slots in rank order) differ at that level, so a slice / multinomial decision that sits on its boundary
    # flips for a few chains and those chains continue on different -- equally valid -- trajectories.  Report how many
    # chains agree and how closely, not a max over all 4 M entries.
    spread = float((d1 - mode[None, None, :]).std().item())
    per_chain = (d1 - d2).abs().amax(dim=2)[0] / max(spread, 1e-30)          # [C] max |diff| in posterior sds
    parity["peer_vs_allreduce_first_draw"] = {
        "chains_agreeing_within_1e-2_sd": float((per_chain < 1e-2).float().mean().item()),
        "median_chain_maxdiff_in_posterior_sd": float(per_chain.median().item()),
        "grand_mean_diff_in_standard_errors": float(((d1.mean(dim=(0, 1)) - d2.mean(dim=(0, 1))).abs().max().item())
                                                    / max(spread / C ** 0.5, 1e-30))}
    parity["peer_vs_allreduce_grad_evals"] = [int(peer_leaves.item()), rep_leaves]
    chk = torch.stack([d2.double().sum(), d2.double().abs().sum(), (d2.double() ** 2).sum()])
    allc = [torch.empty_like(chk) for _ in range(world)]
    dist.all_gather(allc, chk)
    parity["merged_draws_bit_equal_across_ranks"] = bool(all(torch.equal(allc[0], c_) for c_ in allc))
    for t_, s_ in zip((st.theta, st.n_leaves, st.n_accept, st.n_diverge), saved):
        t_.copy_(s_)
    log(f"parity self-check: {parity}")

    # ---- timed: peer-sliced steps
    warm = max(args.warmup, 3)
    timed = Timed(torch, args.steps)
    for _ in range(warm):
        timed.flush.fill_(1)
        step(SLICE)
    barrier()
    clocks = ClockSampler(local_rank)
    clocks.start()
    l0 = leaves_all()
    n0 = lib.b2m_launch_count()
    ten = (ctypes.c_double * 10)()
    lib.b2m_profile(1)
    barrier()
    timed.run(lambda: step(SLICE))
    barrier()
    if args.dump_outputs and rank == 0:     # rank 0 advances (and writes the draws of) the first C / N chains
        dump_outputs(args.dump_outputs, draws[:, :C // world], depths[:, :C // world])
    lib.b2m_profile_read_ex(ten)
    lib.b2m_profile(0)
    four = list(ten)[:4]
    launches = lib.b2m_launch_count() - n0
    dl = leaves_all() - l0
    total_ms = timed.total_ms()
    own_depths = depths[:, rank * (C // world):(rank + 1) * (C // world)]
    mean_depth = float(own_depths.float().mean().item())
    leaves_local = float(dl.item())

    # ---- e2e: public API with host buffers; the front-end merges the slices' draws over torch.distributed
    S_e2e, e2e_steps = ITERS, max(2, min(args.steps, 3))
    host_theta = st.theta.cpu().numpy().copy()
    host_init = {"beta": np.zeros(D, dtype=np.float32)}
    eps_host = float(st.step_size.median().item())

    def api_call(k):
        return B.nuts(fn, host_init, num_samples=S_e2e, num_warmup=1, step_size=eps_host, max_tree_depth=MD,
                      adapt_step_size=False, key=mx.random.key(100 + k), num_chains=C, compat="correct", return_info=True,
                      theta0=host_theta, model=model, slice_state="peer" if SLICE == _cabi.SLICE_PEER else "nccl")

    api_call(0)
    barrier()
    t0 = time.perf_counter()
    e2e_evals = 0
    for k in range(e2e_steps):
        _, _, info = api_call(k + 1)
        e2e_evals += info.grad_evals
    barrier()
    e2e_s = time.perf_counter() - t0
    clock_info = clocks.stop()

    # ---- for the record: the same steps through NCCL (replicated state + all-reduce; sliced reduce-scatter / all-gather)
    others = {}
    for name_, mode_ in (("nccl_allreduce_replicated", _cabi.SLICE_OFF), ("nccl_reduce_scatter_sliced", _cabi.SLICE_NCCL)):
        tm = Timed(torch, 2)
        step(mode_)
        barrier()
        b0 = leaves_all()
        tm.run(lambda: step(mode_))
        barrier()
        d_ = leaves_all() - b0
        tt = torch.tensor([tm.total_ms()], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        if mode_ != _cabi.SLICE_OFF:
            dist.all_reduce(d_)
        others[name_] = {"value": float(d_.item()) / (float(tt[0]) * 1e-3), "ms_per_step": float(tt[0]) / 2}

    t = torch.tensor([total_ms, e2e_s], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([leaves_local, launches], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    total_ms, e2e_s = float(t[0]), float(t[1])
    leaves_tot, launches_all = float(cnt[0]), int(cnt[1])
    value = leaves_tot / (total_ms * 1e-3)
    log(f"strong scaling, {world} ranks: {total_ms / args.steps:.1f} ms/step of {ITERS} transitions, mean depth {mean_depth:.2f}")
    out = {"value": value, "ms_per_step": total_ms / args.steps, "gpu_launches": launches_all, "clocks": clock_info,
           "e2e": {"value": e2e_evals / e2e_s, "unit": UNIT, "h2d_bytes_per_step": C * D * 4, "d2h_bytes_per_step": S_e2e * C * D * 4,
                   "call": f"nuts(num_warmup=1, num_samples={S_e2e}, num_chains={C}, adapt_step_size=False, model=<obs-sharded>, "
                           f"slice_state='peer') with [C, D] host initial values on every rank; merged draws returned as host numpy"},
           "parity": parity, "obs_sharded_nccl": others,
           "config_extra": {"chains_total": C, "chains_advanced_per_gpu": C // world, "rows_per_gpu": rows_local,
                            "iters_per_step": ITERS, "mean_tree_depth": mean_depth,
                            "grad_evals_per_step_total": leaves_tot / args.steps, "adapted_step_size_median": eps_host,
                            "exchange": exchange_note or (
                                "peer window: K6 epilogue -> owner's slot (NVLink stores), owner -> all: packed fp16 rows; "
                                f"{4 * C * D * (world - 1) / world / 1e6:.1f} MB out per rank per gradient, no NCCL in the loop")}}
    if rank != 0:
        return out
    out["roofline"] = glm_roofline(torch, four, leaves_tot, rows_local, D, C, total_ms, model, wl_name,
                                   rows_note=f"{rows_local} of {N} observation rows per GPU (observation shard)")
    both = out["roofline"]["avg_launch_ms"]["K5"] + out["roofline"]["avg_launch_ms"]["K6"]
    ticks = out["roofline"]["launches_timed"] / 2 / args.steps
    out["issue"] = {"lockstep_eval_ms_gemms": both, "tick_ms": total_ms / args.steps / max(ticks, 1), "ticks_per_step": ticks,
                    "non_gemm_ms_per_tick": total_ms / args.steps / max(ticks, 1) - both,
                    "state_kernel_ms_avg": ten[4] / max(ten[5], 1), "wait_kernel_ms_avg": ten[6] / max(ten[7], 1),
                    "signal_kernel_ms_avg": ten[8] / max(ten[9], 1),
                    "note": "rank 0, CUDA events around every launch: the state kernel's time includes its wait for the other ranks' "
                            "gradient partials, the wait kernel's its wait for their packed rows (rank skew shows up there)"}
    return out


def glm_ess_public_run(torch, B, wl, fn, C, chain_offset, n_warm=150, n_samp=500):
    """min-ESS/s as SURVEY.md 8(d) defines it: the public MCMC.run from beta = 0 -- warm-up included in the wall time --
    then the ESS of every (chain, coefficient) series on the device, summed over chains, minimum over coefficients."""
    import mlx_mcmc_b200.core as mx  # noqa: F401
    D = wl["d"]
    m = B.MCMC(fn)
    kw = dict(num_samples=n_samp, num_warmup=n_warm, method="nuts", step_size=wl["eps0"], max_tree_depth=wl["max_tree_depth"],
              num_chains=C, chain_offset=chain_offset, compat="correct", step_size_adaptation="pooled", adapt_mass_matrix=True,
              step_size_jitter=0.2, return_torch=True, return_info=True, verbose=False, random_seed=7)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    m.run({"beta": np.zeros(D, dtype=np.float32)}, **kw)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    tab = m.diagnostics()["beta"]
    info = m.info
    log(f"public run(): {n_warm}+{n_samp} iterations x {C} chains in {wall:.1f}s, mean depth {float(info.depths.mean()):.2f}")
    return {"min_ess_per_s_geyer": float(tab["ess_geyer"].min()) / wall,
            "min_ess_per_s_reference_estimator": float(tab["ess"].min()) / wall,
            "max_rhat": float(np.nanmax(tab["rhat"])), "draws": n_samp, "warmup": n_warm, "wall_s": wall, "chains": C,
            "grad_evals": int(info.grad_evals), "grad_evals_per_s_incl_warmup": info.grad_evals / wall,
            "mean_tree_depth": float(info.depths.mean()), "step_size": float(np.median(info.step_size)),
            "call": "MCMC(log_prob).run({'beta': 0}, num_warmup=%d, num_samples=%d, method='nuts', num_chains=%d, compat='correct', "
                    "step_size_adaptation='pooled', adapt_mass_matrix=True, step_size_jitter=0.2, return_torch=True)" % (n_warm, n_samp, C),
            "note": "wall time of the whole run() call from beta = 0 including warm-up (windowed step-size + diagonal mass-matrix "
                    "adaptation); ESS of every (chain, coefficient) series computed on the device (b2m_diag_series), summed over "
                    "chains, minimum over the coefficients; per GPU.  The reference estimator (examples/06:22-41) goes negative "
                    "on antithetic chains; the Geyer figure is the one to read (SURVEY.md 8d)."}


# ----------------------------------------------------------------------------------------- pointwise workloads
def bench_pointwise(torch, dist, B, lib, args, wl, wl_name, rank, world, local_rank, full=True):
    import mlx_mcmc_b200.core as mx
    from mlx_mcmc_b200 import _cabi, workloads as W
    from mlx_mcmc_b200.diagnostics import compute_ess, ess_geyer, min_ess
    from mlx_mcmc_b200.engine import ChainState, compile_model, launch_hmc, launch_mh
    C = args.chains or wl["chains"]
    chain_offset = rank * C
    fn, init, meta = W.ALL_SMALL[wl["model"]](B.ns)
    model = compile_model(fn, init)
    D, ITERS = model.D, wl["iters"]
    st = ChainState(model, model.pack(init, C), wl.get("step_size", 0.0), chain_offset)
    draws = torch.empty((ITERS, C, D), dtype=torch.float32, device="cuda")
    seed = 1234
    if wl["method"] == "hmc":   # untimed: adapt the step size exactly as run() would (reference rule, 300 iterations)
        launch_hmc(st, 300, wl["L"], _cabi.ADAPT_REFERENCE, 0.8, seed, 0)
        st.reset_counters()
    it_count = [300]

    def one_step():
        if wl["method"] == "hmc":
            launch_hmc(st, ITERS, wl["L"], _cabi.ADAPT_NONE, 0.8, seed, it_count[0], draws=draws)
        else:
            launch_mh(st, ITERS, wl["proposal_scale"], seed, it_count[0], draws=draws)
        it_count[0] += ITERS

    evals_per_step = C * ITERS * (wl["L"] if wl["method"] == "hmc" else 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # first the generic kernels (term table interpreted on every evaluation), for the record; then the kernels NVRTC
    # specialised to this model (mlx_mcmc_b200/jit.py: same source, table baked in as literals) -- the timed path
    from mlx_mcmc_b200.jit import specialize
    generic_ms = None
    if not args.no_jit:
        tg = Timed(torch, 3)
        for _ in range(3):
            one_step()
        barrier()
        tg.run(one_step)
        barrier()
        generic_ms = tg.total_ms() / 3
    t_jit = time.perf_counter()
    jit_on = False if args.no_jit else specialize(model, "auto")
    t_jit = time.perf_counter() - t_jit
    timed = Timed(torch, args.steps)
    for _ in range(max(args.warmup, 3)):
        timed.flush.fill_(1)
        one_step()
    barrier()
    clocks = ClockSampler(local_rank)
    clocks.start()
    n0 = lib.b2m_launch_count()
    barrier()
    timed.run(one_step)
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, draws)
    launches = lib.b2m_launch_count() - n0
    total_ms = timed.total_ms()

    e2e_steps = max(2, min(args.steps, 5))
    n_warm_e2e = ITERS

    def api_call(k):
        if wl["method"] == "hmc":
            return B.hmc(fn, init, num_samples=ITERS, num_warmup=n_warm_e2e, step_size=wl["step_size"],
                         num_leapfrog_steps=wl["L"], key=mx.random.key(k), num_chains=C, chain_offset=chain_offset)
        return B.metropolis_hastings(fn, init, num_samples=ITERS, proposal_scale=wl["proposal_scale"], random_seed=k,
                                     num_chains=C, chain_offset=chain_offset)

    api_call(0)
    barrier()
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        api_call(k + 1)
    barrier()
    e2e_s = time.perf_counter() - t0
    clock_info = clocks.stop()
    e2e_evals = e2e_steps * C * ((ITERS + n_warm_e2e) * wl["L"] if wl["method"] == "hmc" else ITERS)

    t = torch.tensor([total_ms, e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_s = float(t[0]), float(t[1])
    value = world * evals_per_step * args.steps / (total_ms * 1e-3)
    out = {"value": value, "ms_per_step": total_ms / args.steps, "gpu_launches": int(launches) * world, "clocks": clock_info,
           "e2e": {"value": world * e2e_evals / e2e_s, "unit": UNIT, "h2d_bytes_per_step": C * D * 4,
                   "d2h_bytes_per_step": ITERS * C * D * 4,
                   "call": f"hmc(num_warmup={n_warm_e2e}, num_samples={ITERS}, num_chains={C})" if wl["method"] == "hmc"
                   else f"metropolis_hastings(num_samples={ITERS}, num_chains={C})"},
           "config_extra": {"chains_per_gpu": C, "iters_per_step": ITERS, "specialised_kernels": bool(jit_on),
                            "nvrtc_compile_s": t_jit if jit_on else None,
                            "generic_interpreter_kernels_value": (world * evals_per_step / (generic_ms * 1e-3)) if generic_ms else None}}
    if rank != 0:
        return out
    peaks = load_peaks()
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    launch_ms = total_ms / max(launches, 1)
    alg_bytes = ITERS * C * D * 4 + C * (D * 4 + 8 + 16) * 2     # draws written + chain state read and written back
    hbm_achieved = alg_bytes / (launch_ms * 1e-3) / 1e9
    # SURVEY.md 8(d): these configurations are bound by FP32 / SFU instruction issue, not by HBM or the tensor pipe.
    # Algorithmic flops per evaluation = N x f_term (Normal likelihood 10, Exponential likelihood 4 per observation) +
    # the scalar prior terms (~12 each: a log, a divide, a few multiply-adds) + the integrator (6 D per leapfrog step).
    n_obs = int(getattr(meta, "N", 0))
    f_term = {"c1_normal": 10.0, "c2_event_rate": 4.0}.get(wl["model"], 0.0)
    n_prior = {"c1_normal": 2, "c2_event_rate": 1, "c5_ab_test": 4}.get(wl["model"], 1)
    flops_per_eval = n_obs * f_term + 12.0 * n_prior + 6.0 * D
    sm_max = float(peaks.get("sm_max_mhz", 1965.0))
    fp32_peak = 148 * 128 * 2 * sm_max * 1e6 / 1e12                  # 148 SMs x 128 FP32 lanes x FMA, at the maximum SM clock
    achieved_tf = (value / world) * flops_per_eval / 1e12
    out["roofline"] = {"bound": "fp32", "achieved": achieved_tf, "peak": fp32_peak, "unit": "TFLOP/s", "frac": achieved_tf / fp32_peak,
                       "traffic": None, "kernel": "hmc_kernel" if wl["method"] == "hmc" else "mh_kernel",
                       "flops_per_eval": flops_per_eval,
                       "peak_source": f"148 SMs x 128 FP32 lanes x 2 (FMA) x {sm_max:.0f} MHz (sm_max_mhz of MEASURED_PEAKS.json); no tensor-pipe work "
                                      "on this path",
                       "hbm": {"achieved_GBps": hbm_achieved, "peak_GBps": hbm_peak, "frac": hbm_achieved / hbm_peak,
                               "bytes": "draws written + chain state in/out; observations live in shared memory"},
                       "issue_profile": PW_ISSUE.get(wl_name),
                       "note": "FP32-issue bound (SURVEY.md 8d): achieved = algorithmic flops (N x f_term + priors + integrator) x grad-evals/s "
                               "against the FP32 FMA peak.  The executed instruction mix per evaluation (interpreter control, Philox, "
                               "logf / expf) and the issue-slot utilisation are in issue_profile, from the committed ncu capture."}
    out["issue"] = {"grad_evals_per_s_per_gpu": value / world, "obs_terms_per_s_per_gpu": value / world * n_obs,
                    "avg_launch_ms": launch_ms}
    if full and not args.no_ess and wl["method"] == "hmc":
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        from mlx_mcmc_b200.diagnostics import device_summary
        s, rate = B.hmc(fn, init, num_samples=1000, num_warmup=1000, step_size=wl["step_size"], num_leapfrog_steps=wl["L"],
                        key=mx.random.key(99), num_chains=C, return_torch=True)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        dr = torch.stack([v.reshape(C, 1000, -1) for v in s.values()], dim=-1).reshape(C, 1000, -1).permute(1, 0, 2).contiguous()
        tab = device_summary(dr)
        out["ess"] = {"min_ess_per_s_geyer": float(tab["ess_geyer"].min()) / wall,
                      "min_ess_per_s_reference_estimator": float(tab["ess"].min()) / wall,
                      "max_rhat": float(np.nanmax(tab["rhat"])),
                      "accept_rate": rate, "run": "1000 warm-up + 1000 draws incl. warm-up time", "wall_s": wall, "chains": C,
                      "note": "ESS of every chain computed on the device (b2m_diag_series), summed over chains, minimum over "
                              "the parameters; per GPU"}
    return out


def c1_single_chain(torch, B):
    """BASELINE.json configs[0]: the reference's own CPU-runnable case through the public API, ONE chain, exactly the
    settings of examples/02_hmc_comparison.py:87-97 (HMC eps0 = 0.1, L = 10, target 0.8, 1000 warm-up + 5000 draws, seed 42)."""
    import mlx_mcmc_b200.core as mx
    from mlx_mcmc_b200 import workloads as W
    from mlx_mcmc_b200.diagnostics import compute_ess, ess_geyer
    fn, init, _ = W.c1_normal(B.ns)
    B.hmc(fn, init, num_samples=10, num_warmup=10, key=mx.random.key(1))      # trace + first launch outside the timing
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    s, rate = B.hmc(fn, init, num_samples=5000, num_warmup=1000, step_size=0.1, num_leapfrog_steps=10, target_accept=0.8,
                    key=mx.random.key(42))
    wall = time.perf_counter() - t0
    ess_ref = min(compute_ess(v) for v in s.values())
    ess_g = min(ess_geyer(v) for v in s.values())
    return {"call": "hmc(log_prob, {'mu': 0, 'sigma': 1}, num_samples=5000, num_warmup=1000, step_size=0.1, num_leapfrog_steps=10, "
                    "target_accept=0.8, key=mx.random.key(42))  [1 chain, reference's +-5 % step-size rule, host numpy draws]",
            "wall_s": wall, "grad_evals_per_s": 6000 * 10 / wall, "accept_rate": rate,
            "min_ess_reference_estimator": ess_ref, "min_ess_geyer": ess_g, "min_ess_per_s_reference_estimator": ess_ref / wall,
            "min_ess_per_s_geyer": ess_g / wall,
            "posterior_mean": {k: float(np.mean(v)) for k, v in s.items()},
            "note": "one chain cannot fill a GPU: the launch is latency bound (32 lanes of one warp stride the 100 observations); "
                    "the reference's rule collapses the step size on this model exactly as the reference does (BASELINE.md section 2)"}


def c1_chain_sweep(torch, B, lib):
    """C1 throughput against the number of lock-step chains (device-timed, one launch of 50 iterations x L = 10)."""
    from mlx_mcmc_b200 import _cabi, workloads as W
    from mlx_mcmc_b200.engine import ChainState, compile_model, launch_hmc
    fn, init, _ = W.c1_normal(B.ns)
    model = compile_model(fn, init)
    rows = []
    for C in (1, 32, 1024, 16384, 65536, 262144, 1048576):
        st = ChainState(model, model.pack(init, C), 0.01, 0)
        launch_hmc(st, 20, 10, _cabi.ADAPT_NONE, 0.8, 7, 0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        launch_hmc(st, 50, 10, _cabi.ADAPT_NONE, 0.8, 7, 20)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        rows.append({"chains": C, "ms": ms, "grad_evals_per_s": C * 50 * 10 / (ms * 1e-3)})
    return rows


# ----------------------------------------------------------------------------------------- main
def emit(line: dict):
    """the ONE JSON line, written to the process's original stdout"""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def main():
    # Libraries (NCCL's version banner, for one) print to file descriptor 1; rank 0 must print exactly one JSON line
    # there.  Keep a private copy of stdout for that line and point fd 1 at stderr for everything else.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--chains", type=int, default=0, help="chains per GPU (default: the workload's)")
    ap.add_argument("--scaling", default="auto", choices=["auto", "strong", "weak"],
                    help="multi-GPU partitioning: strong = observation sharding of the same chains (default for c4), "
                         "weak = chain sharding")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ess", action="store_true")
    ap.add_argument("--no-others", action="store_true", help="skip the short runs of the other configurations")
    ap.add_argument("--no-jit", action="store_true", help="pointwise workloads: keep the generic interpreter kernels")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the draws (and NUTS tree depths) of the last timed step to DIR/<name>.npy, float32, "
                         "at most 48 MiB in all (a fixed sample of the chains when the draws are larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the device path computed; the reference arm keeps no outputs")
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    scaling = args.scaling
    if scaling == "auto":      # BASELINE.json configs[3] is written observation-sharded; every other configuration shards chains
        scaling = "strong" if args.workload == "c4" else "weak"
    if scaling == "strong" and wl["kind"] != "glm":
        raise SystemExit("--scaling strong (observation sharding) is defined for the regression workloads")
    # `config` describes the workload and is the same object for both arms; what an arm actually executed is in `run`
    config = {"workload": wl["desc"], "l2": "flushed between timed steps (256 MiB write)", "_scaling": scaling}
    if wl["kind"] == "glm":
        config.update({"n_obs": wl["n"], "n_params": wl["d"], "chains": args.chains or wl["chains"],
                       "sampler": f"NUTS, max_tree_depth={wl['max_tree_depth']}, identity mass matrix, no jitter, slice kept in log space "
                                  "(compat=correct), chains at stationarity (started in the typical set), fixed adapted step size",
                       "multi_gpu": ("strong scaling: the same chains in total, observations sharded over the ranks" if scaling == "strong"
                                     else "weak scaling: chains sharded, per-GPU chains fixed, no data-path collective")})
    else:
        config.update({"chains_per_gpu": args.chains or wl["chains"], "multi_gpu": "weak scaling: chains sharded, no data-path collective"})

    if args.impl == "reference":
        if rank != 0:
            return 0
        return reference_arm(args, wl, config)
    config.pop("_scaling")

    import torch
    import torch.distributed as dist
    import mlx_mcmc_b200 as B
    from mlx_mcmc_b200 import _cabi

    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = _cabi.load(build_if_missing=False)

    if wl["kind"] == "glm" and scaling == "strong" and world > 1:
        res = bench_glm_strong(torch, dist, B, lib, args, wl, args.workload, rank, world, local_rank)
    else:
        run = bench_glm if wl["kind"] == "glm" else bench_pointwise
        res = run(torch, dist, B, lib, args, wl, args.workload, rank, world, local_rank)

    if rank == 0:
        run_info = res.pop("config_extra")
        run_info["what"] = ("b200 arm: hand-written sm_100a kernels through libb200mcmc.so; GLM arithmetic = tcgen05 GEMMs on hi/lo split "
                            "operands (3xFP16 with power-of-two operand scaling when the data's dynamic range allows, else 3xTF32), fp32 "
                            "accumulate, centred contraction; NUTS = iterative tree, iteration-asynchronous lock-step schedule with a "
                            "fused per-chain state kernel")
        line = {"metric": METRIC, "value": res.pop("value"), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": res.pop("ms_per_step"), "higher_is_better": True,
                "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config, "run": run_info}
        line.update(res)
        if world == 1 and not args.no_others:
            others = {}
            small = argparse.Namespace(**vars(args))
            small.steps, small.warmup, small.chains, small.no_ess, small.dump_outputs = 5, 3, 0, True, None
            for name in ("c3", "c2", "c1", "c5"):
                if name == args.workload:
                    continue
                w2 = WORKLOADS[name]
                r2 = (bench_glm if w2["kind"] == "glm" else bench_pointwise)(torch, dist, B, lib, small, w2, name, 0, 1,
                                                                             local_rank, full=False)
                others[name] = {"workload": w2["desc"], "value": r2["value"], "unit": UNIT, "ms_per_step": r2["ms_per_step"],
                                "e2e": r2["e2e"]["value"], "roofline": {k: r2["roofline"][k] for k in
                                                                       ("bound", "achieved", "peak", "unit", "frac", "kernel", "hbm")
                                                                       if k in r2["roofline"]},
                                "config": r2["config_extra"]}
            others["c1"]["single_chain_drop_in"] = c1_single_chain(torch, B)
            others["c1"]["chain_sweep"] = c1_chain_sweep(torch, B, lib)
            line["other_workloads"] = others
        log("device part done; cpu baseline")
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline(args.workload, (os.cpu_count() or 1) if wl["kind"] == "glm" else 1)
            if not args.no_others:
                try:
                    line["cpu_baseline"]["full_length"] = cpu_full_length()
                except Exception as e:      # a worker died: say so, keep the line
                    line["cpu_baseline"]["full_length"] = {"error": repr(e)}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
