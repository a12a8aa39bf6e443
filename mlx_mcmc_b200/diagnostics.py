"""Effective-sample-size estimators used for the min-ESS/s metric (SURVEY.md 8d).

`compute_ess` is the ad-hoc estimator of the reference's examples (examples/06_nuts_comparison.py:22-41),
reported verbatim; `ess_geyer` is the standard initial-positive-sequence estimator, used whenever the
two disagree in sign (the reference's estimator goes negative on antithetic chains)."""
from __future__ import annotations

import ctypes as C

import numpy as np


def compute_ess(samples) -> float:
    """n / (1 + 2 sum rho_k), lags 1..min(n/2,100)-1, stopping after the first rho_k < 0.05."""
    x = np.asarray(samples, dtype=np.float64)
    n = len(x)
    mean, var = np.mean(x), np.var(x)
    if var == 0:
        return float(n)
    acf = []
    for lag in range(1, min(n // 2, 100)):
        c = np.mean((x[:-lag] - mean) * (x[lag:] - mean)) / var
        acf.append(c)
        if c < 0.05:
            break
    return float(n / (1 + 2 * np.sum(acf)))


def _autocov_fft(x):
    n = len(x)
    m = 1 << int(np.ceil(np.log2(2 * n)))
    f = np.fft.rfft(x - np.mean(x), m)
    return np.fft.irfft(f * np.conj(f), m)[:n] / n


def ess_geyer(samples) -> float:
    """Geyer's initial positive sequence: sum autocorrelation pairs while their sum stays positive."""
    x = np.asarray(samples, dtype=np.float64)
    n = len(x)
    if n < 4:
        return float(n)
    acov = _autocov_fft(x)
    if acov[0] <= 0:
        return float(n)
    rho = acov / acov[0]
    tau = -1.0
    for k in range(0, n - 1, 2):
        pair = rho[k] + rho[k + 1]
        if pair < 0:
            break
        tau += 2.0 * pair
    tau = max(tau, 1.0 / n)
    return float(n / tau)


def min_ess(draws: dict, num_chains: int = 1, estimator=ess_geyer, max_chains: int = 256) -> float:
    """Sum over chains (a strided subset of at most `max_chains`, scaled up) of per-chain ESS, minimum over
    scalar parameters.  `draws[name]` is (S,) / (S, n) when num_chains == 1, else (C, S) / (C, S, n)."""
    best = None
    for v in draws.values():
        a = np.asarray(v)
        if num_chains == 1:
            a = a[None]
        if a.ndim == 2:
            a = a[:, :, None]
        C = a.shape[0]
        idx = range(0, C, max(1, C // max_chains))
        for j in range(a.shape[2]):
            tot = sum(estimator(a[c, :, j]) for c in idx) * (C / len(idx))
            best = tot if best is None else min(best, tot)
    return float(best)


# ------------------------------------------------------------------------------------------ on the device
def device_series_stats(draws, ess: bool = True, ess_mode: int = 0):
    """Per (chain, parameter) statistics of `draws` [S, C, D] (float32 CUDA tensor, the samplers' own layout),
    computed by libb200mcmc.so without moving the draws: dict of [C, D] tensors `mean`, `var` (ddof 0) and, with
    ``ess``, `ess` (the reference examples' estimator: examples/06_nuts_comparison.py:22-41 for ess_mode 0,
    examples/02_hmc_comparison.py:111-128 for 1) and `ess_geyer`."""
    import torch
    from . import _cabi
    if not (draws.is_cuda and draws.dtype == torch.float32 and draws.dim() == 3):
        raise ValueError("device_series_stats expects a float32 CUDA tensor of shape [S, C, D]")
    draws = draws.contiguous()
    S, Cn, D = draws.shape
    lib = _cabi.load()
    out = {k: torch.empty((Cn, D), dtype=torch.float32, device=draws.device)
           for k in (("mean", "var", "ess", "ess_geyer") if ess else ("mean", "var"))}
    ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
    with torch.cuda.device(draws.device):
        _cabi.check(lib.b2m_diag_series(ptr(draws), S, Cn, D, ess_mode, ptr(out["mean"]), ptr(out["var"]),
                                        ptr(out.get("ess")), ptr(out.get("ess_geyer")),
                                        C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return out


def device_summary(draws, layout=None, ess: bool = True, ess_mode: int = 0):
    """Per-parameter posterior diagnostics of `draws` [S, C, D] on the device: pooled `mean` and `std` (what
    ``MCMC.summary`` reports, mcmc.py:219-220), Gelman-Rubin `rhat` across the C chains, and `ess` / `ess_geyer`
    summed over chains.  Returns ``{name: {stat: float | np.ndarray}}`` when `layout` (the model's parameter
    layout) is given, else a dict of [D] numpy arrays.  Only D x 5 doubles travel to the host."""
    import torch
    from . import _cabi
    st = device_series_stats(draws, ess, ess_mode)
    S, Cn, D = draws.shape
    lib = _cabi.load()
    out = torch.empty((D, 5), dtype=torch.float64, device=draws.device)
    ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
    with torch.cuda.device(draws.device):
        _cabi.check(lib.b2m_diag_params(ptr(st["mean"]), ptr(st["var"]), ptr(st.get("ess")), ptr(st.get("ess_geyer")),
                                        S, Cn, D, ptr(out), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    h = out.cpu().numpy()
    cols = {"mean": h[:, 0], "std": h[:, 1], "rhat": h[:, 2]}
    if ess:
        cols.update(ess=h[:, 3], ess_geyer=h[:, 4])
    if layout is None:
        return cols
    table = {}
    for name, (off, n, shp) in layout.items():
        table[name] = {k: (float(v[off]) if not shp else v[off:off + n].copy()) for k, v in cols.items()}
    return table


def device_quantiles(x, q):
    """Quantiles `q` (fractions in [0, 1]) of the float32 CUDA tensor `x` (any shape, pooled), numpy's default linear
    interpolation, by the library's radix-select kernels (b2m_quantiles): three histogram passes over x resolve all
    requested order statistics at once; replaces np.median / np.percentile of mlx_mcmc/inference/mcmc.py:221-224."""
    import torch
    from . import _cabi
    if not (x.is_cuda and x.dtype == torch.float32):
        raise ValueError("device_quantiles expects a float32 CUDA tensor")
    x = x.contiguous().reshape(-1)
    q = [float(v) for v in q]
    if not q or len(q) > 8 or any(not 0.0 <= v <= 1.0 for v in q):
        raise ValueError("device_quantiles: 1..8 quantiles in [0, 1]")
    lib = _cabi.load()
    qa = (C.c_double * len(q))(*q)
    out = (C.c_double * len(q))()
    with torch.cuda.device(x.device):
        _cabi.check(lib.b2m_quantiles(C.c_void_p(x.data_ptr()), x.numel(), qa, len(q), out,
                                      C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return [float(v) for v in out]


# ------------------------------------------------------------------------------------------ model comparison (WAIC)
def waic_totals(lppd, mean, var, n_draws: int) -> dict:
    """WAIC from the per-observation statistics of the pointwise log-likelihood ll[s, n] over S draws (Vehtari, Gelman &
    Gabry 2017): lppd_n = log mean_s exp ll[s, n], mean_n = mean_s ll[s, n], var_n = sample variance (ddof 1).
        elpd_waic = sum_n (lppd_n - var_n),  p_waic = sum_n var_n,  waic = -2 elpd_waic,
        se = sqrt(N Var_n(lppd_n - var_n)),  n_warn = #{n : var_n > 0.4}
    plus ``pointwise`` = {lppd, p_waic, elpd} as [N] float64 arrays (what ``waic_compare`` needs)."""
    lppd = np.asarray(lppd, dtype=np.float64)
    mean = np.asarray(mean, dtype=np.float64)
    var = np.asarray(var, dtype=np.float64)
    elpd_i = lppd - var
    n = elpd_i.size
    elpd = float(np.sum(elpd_i))
    return {"elpd_waic": elpd, "p_waic": float(np.sum(var)), "waic": -2.0 * elpd,
            "se": float(np.sqrt(n * np.var(elpd_i))) if n > 0 else 0.0, "lppd": float(np.sum(lppd)),
            "n_warn": int(np.sum(var > 0.4)), "n_obs": int(n), "n_draws": int(n_draws),
            "pointwise": {"lppd": lppd, "p_waic": var, "elpd": elpd_i, "mean": mean}}


def waic(model, draws) -> dict:
    """WAIC of `model` (an ``engine.DeviceModel``) over the posterior `draws` [S, C, D] (float32 CUDA tensor in model
    coordinates, as the samplers write them).  The pointwise log-likelihood of every draw and every observation of the
    model's observation terms (``TracedModel.observation_terms``) is reduced on the device (b2m_loglik_stats: for the
    GLM class inside the B X^T contraction); only [N, 3] float64 statistics reach the host.  Returns ``waic_totals``."""
    import torch
    from . import _cabi
    if not (hasattr(draws, "is_cuda") and draws.is_cuda and draws.dtype == torch.float32 and draws.dim() == 3):
        raise ValueError("waic expects a float32 CUDA tensor of shape [S, C, D]")
    if draws.shape[2] != model.D:
        raise ValueError(f"waic: draws have D = {draws.shape[2]}, the model has {model.D} parameters")
    obs = model.traced.observation_terms()
    if not obs:
        raise ValueError("waic: the model has no observation terms (no term's value is data while one of its "
                         "distribution parameters depends on the model parameters)")
    if getattr(model, "_comm", None) is not None or getattr(model, "_peer", None) is not None:
        raise ValueError("waic: observation-sharded models are not supported (each rank holds only its rows)")
    draws = draws.contiguous()
    if not bool(torch.isfinite(draws).all()):
        raise ValueError("waic: the draws contain non-finite values")
    S = draws.shape[0] * draws.shape[1]
    n_obs = sum(model.traced.terms[i].length for i in obs)
    out = torch.empty((n_obs, 3), dtype=torch.float64, device=draws.device)
    idx = (C.c_int32 * len(obs))(*obs)
    with torch.cuda.device(draws.device):
        _cabi.check(model.lib.b2m_loglik_stats(model.handle, C.c_void_p(draws.data_ptr()), S, idx, len(obs),
                                               C.c_void_p(out.data_ptr()), n_obs,
                                               C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    h = out.cpu().numpy()
    return waic_totals(h[:, 0], h[:, 1], h[:, 2], S)


def waic_compare(a: dict, b: dict) -> dict:
    """Difference of two ``waic`` results on the same observations: elpd_diff = elpd_a - elpd_b and its standard error
    sqrt(N Var_n(elpd_a,n - elpd_b,n)) from the pointwise arrays.  Positive elpd_diff favours `a`."""
    if a["n_obs"] != b["n_obs"]:
        raise ValueError(f"waic_compare: the results cover different observations ({a['n_obs']} vs {b['n_obs']})")
    d = np.asarray(a["pointwise"]["elpd"], dtype=np.float64) - np.asarray(b["pointwise"]["elpd"], dtype=np.float64)
    return {"elpd_diff": float(np.sum(d)), "se_diff": float(np.sqrt(d.size * np.var(d)))}
