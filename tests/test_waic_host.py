"""CPU: which traced terms count as observations for WAIC (TracedModel.observation_terms), the WAIC totals and
waic_compare against a direct numpy evaluation of a pointwise log-likelihood matrix, and the C ABI entry point."""
import numpy as np
from scipy import special

import mlx_mcmc_b200 as B
from mlx_mcmc_b200 import _cabi, workloads as W
from mlx_mcmc_b200.diagnostics import waic_compare, waic_totals
from mlx_mcmc_b200.tracer import BERNOULLI, EXPONENTIAL, NORMAL, OP_LIN, OP_MATVEC, trace


def _obs(fn, init):
    tm = trace(fn, init)
    idx = tm.observation_terms()
    return tm, idx, [tm.terms[i].length for i in idx]


# ----------------------------------------------------------------------------- observation terms
def test_c1_styles_give_the_same_observations():
    seen = []
    for style in ("vector", "unrolled", "stack"):
        fn, init, _ = W.c1_normal(B.ns, style=style)
        tm, idx, lens = _obs(fn, init)
        assert lens == [100], (style, lens)
        t = tm.terms[idx[0]]
        assert t.dist == NORMAL
        seen.append(np.asarray(tm.arrays[t.x.a]))
    for y in seen[1:]:
        np.testing.assert_array_equal(y, seen[0])


def test_c2_and_c5():
    fn, init, _ = W.c2_event_rate(B.ns)
    tm, idx, lens = _obs(fn, init)
    assert lens == [50] and tm.terms[idx[0]].dist == EXPONENTIAL
    fn, init, _ = W.c5_ab_test(B.ns)
    assert _obs(fn, init)[1] == []          # priors and conjugate Beta terms only: no observation


def test_glm_workloads_have_the_matvec_term():
    for make, dist in ((W.regression, NORMAL), (W.logistic_regression, BERNOULLI)):
        fn, init, _ = make(B.ns, 300, 7, seed=1)
        tm, idx, lens = _obs(fn, init)
        assert lens == [300]
        t = tm.terms[idx[0]]
        assert t.dist == dist and OP_MATVEC in (t.p0.kind, t.p1.kind)
    fn, init, _ = W.t_regression_sigma(B.ns)
    assert _obs(fn, init)[2] == [60]        # the HalfNormal prior on sigma is not an observation


def test_two_observed_arrays_of_different_distributions():
    rs = np.random.default_rng(0)
    a, b = rs.normal(size=17).astype(np.float32), rs.exponential(size=9).astype(np.float32)

    def fn(p):
        return (B.ns.Normal(0, 5).log_prob(p["mu"]) + B.ns.Exponential(1.0).log_prob(p["rate"])
                + B.ns.mx.sum(B.ns.Normal(p["mu"], 1.5).log_prob(B.ns.mx.array(a)))
                + B.ns.mx.sum(B.ns.Exponential(p["rate"]).log_prob(B.ns.mx.array(b))))
    tm, idx, lens = _obs(fn, {"mu": 0.0, "rate": 1.0})
    assert lens == [17, 9]
    assert [tm.terms[i].dist for i in idx] == [NORMAL, EXPONENTIAL]


def test_affine_lin_bernoulli_logit():
    rs = np.random.default_rng(1)
    x, y = rs.normal(size=40).astype(np.float32), (rs.uniform(size=40) < 0.5).astype(np.float32)

    def fn(p):
        return (B.ns.Normal(0, 5).log_prob(p["a"]) + B.ns.Normal(0, 5).log_prob(p["b"])
                + B.ns.mx.sum(B.ns.Bernoulli(logits=p["a"] + p["b"] * B.ns.mx.array(x)).log_prob(B.ns.mx.array(y))))
    tm, idx, lens = _obs(fn, {"a": 0.0, "b": 0.0})
    assert lens == [40]
    assert tm.terms[idx[0]].p0.kind == OP_LIN


def test_glm_with_an_extra_observed_term():
    fr, _, meta = W.regression(B.ns, 64, 5, seed=2)
    z = np.linspace(-1, 1, 11).astype(np.float32)

    def fn(p):
        return fr({"beta": p["beta"]}) + B.ns.mx.sum(B.ns.Normal(p["m"], 2.0).log_prob(B.ns.mx.array(z)))
    tm, idx, lens = _obs(fn, {"beta": np.zeros(5, np.float32), "m": 0.0})
    assert tm.is_glm
    assert lens == [64, 11]                 # term order: X @ beta likelihood, then the extra observed vector


# ----------------------------------------------------------------------------- totals against numpy
def _stats(ll):
    S = ll.shape[0]
    return special.logsumexp(ll, axis=0) - np.log(S), ll.mean(axis=0), ll.var(axis=0, ddof=1)


def test_waic_totals_and_compare_match_numpy():
    rs = np.random.default_rng(3)
    S, N = 400, 57
    ll_a = -0.5 * rs.normal(1.0, 0.7, size=(S, N)) ** 2 - 1.0
    ll_b = ll_a - 0.3 * rs.uniform(size=(S, N))
    ra, rb = waic_totals(*_stats(ll_a), S), waic_totals(*_stats(ll_b), S)
    lppd = np.log(np.mean(np.exp(ll_a), axis=0))
    pw = np.var(ll_a, axis=0, ddof=1)
    elpd_i = lppd - pw
    assert np.isclose(ra["elpd_waic"], elpd_i.sum(), rtol=1e-12)
    assert np.isclose(ra["p_waic"], pw.sum(), rtol=1e-12)
    assert np.isclose(ra["waic"], -2 * elpd_i.sum(), rtol=1e-12)
    assert np.isclose(ra["se"], np.sqrt(N * np.var(elpd_i)), rtol=1e-12)
    assert ra["n_warn"] == int(np.sum(pw > 0.4)) and ra["n_obs"] == N and ra["n_draws"] == S
    np.testing.assert_allclose(ra["pointwise"]["elpd"], elpd_i, rtol=1e-12)
    cmp = waic_compare(ra, rb)
    d = elpd_i - (np.log(np.mean(np.exp(ll_b), axis=0)) - np.var(ll_b, axis=0, ddof=1))
    assert np.isclose(cmp["elpd_diff"], d.sum(), rtol=1e-10)
    assert np.isclose(cmp["se_diff"], np.sqrt(N * np.var(d)), rtol=1e-10)
    try:
        waic_compare(ra, waic_totals(*_stats(ll_a[:, :10]), S))
    except ValueError:
        pass
    else:
        raise AssertionError("waic_compare accepted results over different observations")


# ----------------------------------------------------------------------------- C ABI
def test_loglik_stats_is_exported_and_abi_stays_4():
    assert "b2m_loglik_stats" in _cabi.EXPORTS
    assert _cabi.ABI_VERSION == 4
    lib = _cabi.load()
    assert hasattr(lib, "b2m_loglik_stats") and lib.b2m_abi_version() == 4
