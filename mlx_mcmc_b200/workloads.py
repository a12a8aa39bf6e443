"""The benchmark / parity models, written once against an abstract namespace.

Every factory takes ``ns`` -- any object exposing ``mx`` (an ``mlx.core``-like module) and
the distribution classes -- and returns ``(log_prob_fn, initial_params, meta)``.  The product
passes ``mlx_mcmc_b200.ns``; the tests' checker passes the oracle's namespace.  The model
bodies follow the reference's example scripts (cited per factory); synthetic inputs use the
seeds fixed in SURVEY.md section 8(d).
"""
from __future__ import annotations

from types import SimpleNamespace

import numpy as np


def data_c1(n=100):
    """examples/02_hmc_comparison.py:21-28 -- np.random.seed(42); normal(5, 2, 100)."""
    rs = np.random.RandomState(42)
    return rs.normal(5.0, 2.0, n)


def data_c2(n=50):
    """examples/04_event_rates.py:30-35 -- np.random.seed(42); exponential(1/3, 50)."""
    rs = np.random.RandomState(42)
    return rs.exponential(scale=1 / 3.0, size=n)


def data_c5():
    """examples/03_ab_testing.py:25-39 -- np.random.seed(42); two binomial(1000, p) draws."""
    rs = np.random.RandomState(42)
    a = int(rs.binomial(1000, 0.12))
    b = int(rs.binomial(1000, 0.15))
    return 1000, a, 1000, b


def data_regression(n, d, seed=0, noise=1.0):
    """SURVEY.md 8(d) C3/C4: X~N(0,1) [n,d], beta*~N(0,1), y = X beta* + N(0, noise)."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, d), dtype=np.float32)
    beta = rng.standard_normal(d).astype(np.float32)
    y = (X.astype(np.float64) @ beta.astype(np.float64) + noise * rng.standard_normal(n)).astype(np.float32)
    return X, y, beta


# --------------------------------------------------------------------------------------
def c1_normal(ns, n=100, style="vector"):
    """Normal(mu, sigma) posterior over 100 observations.

    style='vector'   examples/02_hmc_comparison.py:40-52  (mx.sum over one array)
    style='unrolled' examples/01_simple_normal.py:37-50   (python loop, one scalar term per obs)
    style='stack'    tests/test_nuts.py:197-209           (mx.array([...traced scalars...]))
    """
    mx, Normal, HalfNormal = ns.mx, ns.Normal, ns.HalfNormal
    y = data_c1(n)

    def log_prob(params):
        mu, sigma = params["mu"], params["sigma"]
        prior = Normal(0, 10).log_prob(mu) + HalfNormal(5).log_prob(sigma)
        if style == "vector":
            lik = mx.sum(Normal(mu, sigma).log_prob(mx.array(y)))
        elif style == "unrolled":
            lik = mx.array(0.0)
            for yi in y:
                lik = lik + Normal(mu, sigma).log_prob(mx.array(yi))
        else:
            lik = mx.sum(mx.array([Normal(mu, sigma).log_prob(mx.array(yi)) for yi in y]))
        return prior + lik

    return log_prob, {"mu": 0.0, "sigma": 1.0}, SimpleNamespace(name="c1_normal", D=2, N=n, y=y)


def c2_event_rate(ns, n=50, style="vector"):
    """Gamma(2,1) prior on the rate, Exponential(rate) likelihood (examples/04_event_rates.py:43-55)."""
    mx, Gamma, Exponential = ns.mx, ns.Gamma, ns.Exponential
    t = data_c2(n)

    def log_prob(params):
        rate = params["rate"]
        prior = Gamma(alpha=2, beta=1).log_prob(rate)
        if style == "vector":
            lik = mx.sum(Exponential(rate).log_prob(mx.array(t)))
        else:
            lik = mx.array(0.0)
            for ti in t:
                lik = lik + Exponential(rate).log_prob(mx.array(ti))
        return prior + lik

    # exact posterior: Gamma(2 + n, 1 + sum t)
    meta = SimpleNamespace(name="c2_event_rate", D=1, N=n, t=t, post_shape=2.0 + n, post_rate=1.0 + float(np.sum(t)))
    return log_prob, {"rate": 2.0}, meta


def c5_ab_test(ns):
    """Two Beta posteriors, no observation arrays (examples/03_ab_testing.py:46-59)."""
    Beta = ns.Beta
    n_a, k_a, n_b, k_b = data_c5()

    def log_prob(params):
        p_a, p_b = params["p_A"], params["p_B"]
        return (Beta(1, 1).log_prob(p_a) + Beta(1, 1).log_prob(p_b)
                + Beta(k_a + 1, n_a - k_a + 1).log_prob(p_a) + Beta(k_b + 1, n_b - k_b + 1).log_prob(p_b))

    meta = SimpleNamespace(name="c5_ab_test", D=2, N=0, post_a=(k_a + 1, n_a - k_a + 1), post_b=(k_b + 1, n_b - k_b + 1))
    return log_prob, {"p_A": 0.1, "p_B": 0.1}, meta


def regression(ns, n, d, seed=0, prior_scale=10.0, noise=1.0):
    """Bayesian linear regression with known noise (SURVEY.md 8(d) C3/C4; README 'Medium'/'Large').

    log p = sum Normal(0, prior_scale)(beta) + sum Normal(X @ beta, noise)(y); the posterior is the
    closed-form N(m, V), V = (X'X/noise^2 + I/prior_scale^2)^-1, m = V X'y / noise^2.
    """
    mx, Normal = ns.mx, ns.Normal
    X, y, beta_true = data_regression(n, d, seed, noise)
    Xa, ya = mx.array(X), mx.array(y)

    def log_prob(params):
        beta = params["beta"]
        return mx.sum(Normal(0, prior_scale).log_prob(beta)) + mx.sum(Normal(Xa @ beta, noise).log_prob(ya))

    meta = SimpleNamespace(name=f"regression_{d}x{n}", D=d, N=n, X=X, y=y, beta_true=beta_true,
                           prior_scale=prior_scale, noise=noise)
    return log_prob, {"beta": np.zeros(d, dtype=np.float32)}, meta


def regression_posterior(meta):
    """Closed-form posterior mean / covariance of `regression` in float64."""
    X = meta.X.astype(np.float64)
    A = X.T @ X / meta.noise ** 2 + np.eye(meta.D) / meta.prior_scale ** 2
    V = np.linalg.inv(A)
    m = V @ (X.T @ meta.y.astype(np.float64)) / meta.noise ** 2
    return m, V


def data_logistic(n, d, seed=0):
    """X ~ N(0, 1) [n, d], beta* ~ N(0, 1/d) (logits of order 1), y ~ Bernoulli(sigmoid(X beta*)) as float32 0 / 1."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, d), dtype=np.float32)
    beta = (rng.standard_normal(d) / np.sqrt(d)).astype(np.float32)
    eta = X.astype(np.float64) @ beta.astype(np.float64)
    y = (rng.uniform(size=n) < 1.0 / (1.0 + np.exp(-eta))).astype(np.float32)
    return X, y, beta


def logistic_regression(ns, n, d, seed=0, prior_scale=10.0):
    """Bayesian logistic regression: log p = sum Normal(0, prior_scale)(beta) + sum Bernoulli(logits = X @ beta)(y).
    Same design-matrix shape as `regression`, so it runs on the same GLM contractions with the Bernoulli-logit
    epilogue."""
    mx, Normal, Bernoulli = ns.mx, ns.Normal, ns.Bernoulli
    X, y, beta_true = data_logistic(n, d, seed)
    Xa, ya = mx.array(X), mx.array(y)

    def log_prob(params):
        beta = params["beta"]
        return mx.sum(Normal(0, prior_scale).log_prob(beta)) + mx.sum(Bernoulli(logits=Xa @ beta).log_prob(ya))

    meta = SimpleNamespace(name=f"logistic_{d}x{n}", D=d, N=n, X=X, y=y, beta_true=beta_true, prior_scale=prior_scale)
    return log_prob, {"beta": np.zeros(d, dtype=np.float32)}, meta


# small models taken from the reference's own sampler tests -------------------------------
def t_normal_1d(ns, loc=5.0, scale=2.0):
    """tests/test_nuts.py:13-17, tests/test_hmc.py:13-20."""
    def log_prob(params):
        return ns.Normal(loc, scale).log_prob(params["mu"])
    return log_prob, {"mu": 0.0}, SimpleNamespace(name="t_normal_1d", D=1, N=0)


def t_normal_2d(ns):
    """tests/test_nuts.py:34-40."""
    def log_prob(params):
        return ns.Normal(0, 1).log_prob(params["mu1"]) + ns.Normal(5, 2).log_prob(params["mu2"])
    return log_prob, {"mu1": 0.0, "mu2": 0.0}, SimpleNamespace(name="t_normal_2d", D=2, N=0)


def t_halfnormal_scale(ns):
    """tests/test_nuts.py:88-94 -- parameter in the *scale* slot, constant in the value slot."""
    def log_prob(params):
        s = params["sigma"]
        return ns.HalfNormal(5.0).log_prob(s) + ns.Normal(0, s).log_prob(ns.mx.array(0.5))
    return log_prob, {"sigma": 1.0}, SimpleNamespace(name="t_halfnormal_scale", D=1, N=0)


def t_halfnormal(ns, scale=2.0):
    """tests/test_hmc.py:118-124."""
    def log_prob(params):
        return ns.HalfNormal(scale).log_prob(params["sigma"])
    return log_prob, {"sigma": 1.0}, SimpleNamespace(name="t_halfnormal", D=1, N=0)


def t_vector_normal(ns, d=3):
    """A vector parameter with independent Normal(loc_i, scale_i) components (vector-parameter NUTS,
    the only shape nuts.py:338-339 stores with .tolist())."""
    loc = np.linspace(-1.0, 2.0, d).astype(np.float32)
    sc = np.linspace(0.5, 2.0, d).astype(np.float32)

    def log_prob(params):
        return ns.mx.sum(ns.Normal(ns.mx.array(loc), ns.mx.array(sc)).log_prob(params["x"]))
    return log_prob, {"x": np.zeros(d, dtype=np.float32)}, SimpleNamespace(name="t_vector_normal", D=d, N=0, loc=loc, scale=sc)


def t_regression_small(ns, n=40, d=3):
    """A small instance of the regression model (vector parameter, X @ beta) for decision-level NUTS parity;
    H0 stays below the reference's float32 slice underflow (SURVEY.md F6)."""
    fn, init, meta = regression(ns, n, d, seed=3)
    meta.name = "t_regression_small"
    return fn, init, meta


def t_regression_mid(ns, n=2048, d=64):
    """A mid-size instance of the regression model: large enough for the tcgen05 contractions to run whole 128 x 256
    tiles with a real K loop (the decision-level NUTS parity of the tensor-core path), small enough for the reference
    to run a dozen transitions in seconds.  H0 is far above the reference's float32 slice underflow (SURVEY.md F6)."""
    fn, init, meta = regression(ns, n, d, seed=7)
    meta.name = "t_regression_mid"
    return fn, init, meta


def t_regression_sigma(ns, n=60, d=4):
    """Regression with an unknown noise scale: sigma is a scalar parameter next to the coefficient vector."""
    mx, Normal, HalfNormal = ns.mx, ns.Normal, ns.HalfNormal
    X, y, beta_true = data_regression(n, d, seed=5, noise=0.7)
    Xa, ya = mx.array(X), mx.array(y)

    def log_prob(params):
        beta, sigma = params["beta"], params["sigma"]
        return (mx.sum(Normal(0, 5.0).log_prob(beta)) + HalfNormal(2.0).log_prob(sigma)
                + mx.sum(Normal(Xa @ beta, sigma).log_prob(ya)))

    meta = SimpleNamespace(name="t_regression_sigma", D=d + 1, N=n, X=X, y=y, beta_true=beta_true)
    return log_prob, {"beta": np.zeros(d, dtype=np.float32), "sigma": 1.0}, meta


ALL_SMALL = {
    "c1_normal": c1_normal, "c2_event_rate": c2_event_rate, "c5_ab_test": c5_ab_test,
    "t_normal_1d": t_normal_1d, "t_normal_2d": t_normal_2d, "t_halfnormal_scale": t_halfnormal_scale,
    "t_halfnormal": t_halfnormal, "t_vector_normal": t_vector_normal,
    "t_regression_small": t_regression_small, "t_regression_sigma": t_regression_sigma,
    "t_regression_mid": t_regression_mid,
}
