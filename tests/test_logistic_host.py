"""CPU: the Bernoulli distribution and the logistic-regression model -- tracer terms, host log_prob against scipy, the
traced model's value and gradient against direct float64 numpy, refusal of observation sharding, and the library's
term-tag validation."""
import ctypes
import math

import numpy as np
import pytest
from scipy import special, stats

import mlx_mcmc_b200 as B
import mlx_mcmc_b200.core as mx
from mlx_mcmc_b200 import _cabi, dist, workloads as W
from mlx_mcmc_b200.tracer import (BERNOULLI, NORMAL, OP_DATA, OP_LIN, OP_MATVEC, OP_PARAM, OP_PARAMVEC,
                                  UnsupportedOpError, trace)


# ----------------------------------------------------------------------------- float64 reference of a traced table
def _operand64(o, theta, arrays, n):
    from mlx_mcmc_b200 import tracer as T
    if o.kind == T.OP_CONST:
        return np.full(n, o.c)
    if o.kind == T.OP_PARAM:
        return np.full(n, theta[o.a])
    if o.kind == T.OP_DATA:
        return np.broadcast_to(np.asarray(arrays[o.a], dtype=np.float64), (n,))
    if o.kind == T.OP_PARAMVEC:
        return theta[o.a:o.a + o.b]
    if o.kind == T.OP_LIN:
        out = np.full(n, o.c)
        for param, array, coef in o.lin:
            v = coef * (np.asarray(arrays[array], dtype=np.float64) if array >= 0 else 1.0)
            out = out + v * (theta[param] if param >= 0 else 1.0)
        return out
    X = np.asarray(arrays[o.a], dtype=np.float64)
    return X @ theta[o.b:o.b + X.shape[1]] + o.c


def _table_logp64(model, theta):
    """log p of a traced table with Normal and Bernoulli terms, float64"""
    total = 0.0
    for t in model.terms:
        x, p0, p1 = (_operand64(o, theta, model.arrays, t.length) for o in (t.x, t.p0, t.p1))
        if t.dist == NORMAL:
            lp = -0.5 * math.log(2 * math.pi) - np.log(p1) - 0.5 * (x - p0) ** 2 / p1 ** 2
        elif t.dist == BERNOULLI:
            lp = np.where((x == 0) | (x == 1), x * p0 - np.logaddexp(0.0, p0), -np.inf)
        else:
            raise AssertionError(t.dist)
        total += t.weight * float(np.sum(lp))
    return total


# ----------------------------------------------------------------------------- tracer
def test_logistic_regression_traces_to_one_bernoulli_matvec_term():
    fn, init, meta = W.logistic_regression(B.ns, 300, 7, seed=1)
    tm = trace(fn, init)
    assert tm.is_glm and tm.D == 7
    prior, lik = tm.terms
    assert prior.dist == NORMAL and prior.x.kind == OP_PARAMVEC
    assert (lik.dist, lik.length, lik.p0.kind, lik.x.kind) == (BERNOULLI, 300, OP_MATVEC, OP_DATA)
    assert BERNOULLI == 7
    np.testing.assert_array_equal(tm.arrays[lik.x.a], meta.y)
    assert tm.arrays[lik.p0.a].shape == (300, 7)
    assert set(np.unique(meta.y)) <= {0.0, 1.0}


def test_bernoulli_logit_operand_kinds():
    x = np.linspace(-1, 1, 5).astype(np.float32)
    y = np.array([0, 1, 1, 0, 1], dtype=np.float32)
    lin = trace(lambda p: mx.sum(B.Bernoulli(logits=p["a"] + p["b"] * mx.array(x)).log_prob(mx.array(y))), {"a": 0.0, "b": 0.0})
    assert (lin.terms[0].dist, lin.terms[0].p0.kind, lin.terms[0].x.kind) == (BERNOULLI, OP_LIN, OP_DATA)
    scal = trace(lambda p: mx.sum(B.Bernoulli(logits=p["a"]).log_prob(mx.array(y))), {"a": 0.0})
    assert scal.terms[0].p0.kind == OP_PARAM and scal.terms[0].length == 5
    vec = trace(lambda p: mx.sum(B.Bernoulli(logits=p["v"]).log_prob(y)), {"v": np.zeros(5, dtype=np.float32)})
    assert vec.terms[0].p0.kind == OP_PARAMVEC
    shifted = trace(lambda p: mx.sum(B.Bernoulli(logits=mx.array(np.ones((5, 2), np.float32)) @ p["b"] + 0.5).log_prob(y)),
                    {"b": np.zeros(2, dtype=np.float32)})
    assert shifted.terms[0].p0.kind == OP_MATVEC and shifted.terms[0].p0.c == 0.5


def test_traced_probs_and_traced_value_are_refused():
    with pytest.raises(UnsupportedOpError, match="logits="):
        trace(lambda p: B.Bernoulli(probs=p["x"]).log_prob(1.0), {"x": 0.5})
    with pytest.raises(UnsupportedOpError, match="traced value"):
        trace(lambda p: B.Bernoulli(logits=0.3).log_prob(p["x"]), {"x": 0.5})
    with pytest.raises(ValueError):
        B.Bernoulli()
    with pytest.raises(ValueError):
        B.Bernoulli(probs=0.5, logits=0.0)


# ----------------------------------------------------------------------------- host class
def test_host_log_prob_matches_scipy():
    y = np.array([0, 1, 1, 0, 1, 0], dtype=np.float32)
    p = np.array([0.1, 0.5, 0.99, 1e-6, 0.3, 0.7], dtype=np.float32)
    got = B.Bernoulli(probs=p).log_prob(y)
    want = stats.bernoulli.logpmf(y.astype(int), p.astype(np.float64))
    np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-7)
    logits = np.array([-100.0, -100.0, -3.0, 0.0, 2.5, 100.0, 100.0], dtype=np.float32)
    yl = np.array([0, 1, 1, 0, 1, 0, 1], dtype=np.float32)
    got = B.Bernoulli(logits=logits).log_prob(yl)
    assert np.all(np.isfinite(got))
    l64 = logits.astype(np.float64)
    # sigmoid(100) rounds to 1 in float64: take the mirrored form logpmf(1 - y, sigmoid(-l)) for positive logits
    want = np.where(l64 <= 0, stats.bernoulli.logpmf(yl.astype(int), special.expit(l64)),
                    stats.bernoulli.logpmf(1 - yl.astype(int), special.expit(-l64)))
    np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-7)
    assert float(B.Bernoulli(logits=100.0).log_prob(0.0)) == pytest.approx(-100.0, rel=1e-7)
    assert float(B.Bernoulli(logits=-100.0).log_prob(0.0)) == pytest.approx(-math.exp(-100), rel=1e-5)
    for bad in (-1.0, 0.5, 2.0):
        assert float(B.Bernoulli(logits=0.3).log_prob(bad)) == -math.inf
        assert float(B.Bernoulli(probs=0.3).log_prob(bad)) == -math.inf


def test_host_moments_and_sampling():
    b = B.Bernoulli(probs=0.3)
    assert float(b.mean()) == pytest.approx(0.3) and float(b.variance()) == pytest.approx(0.21)
    assert float(B.Bernoulli(logits=0.0).mean()) == 0.5
    s = b.sample(mx.random.key(0), (20000,))
    assert set(np.unique(s)) <= {0.0, 1.0} and abs(float(np.mean(s)) - 0.3) < 0.02
    assert b._device_sample_spec()[:2] == (BERNOULLI, pytest.approx(0.3))
    assert "Bernoulli" in B.__all__ and B.ns.Bernoulli is B.Bernoulli


# ----------------------------------------------------------------------------- model value and gradient
def test_traced_logistic_model_value_and_gradient_in_float64():
    fn, init, meta = W.logistic_regression(B.ns, 400, 6, seed=2)
    tm = trace(fn, init)
    X, y = meta.X.astype(np.float64), meta.y.astype(np.float64)
    rng = np.random.default_rng(5)
    for scale in (0.0, 0.5, 20.0):
        beta = meta.beta_true.astype(np.float64) + scale * rng.standard_normal(6)
        eta = X @ beta
        want = (np.sum(y * eta - np.logaddexp(0.0, eta))
                + np.sum(-0.5 * math.log(2 * math.pi) - math.log(10.0) - 0.5 * beta ** 2 / 100.0))
        got = _table_logp64(tm, beta)
        assert abs(got - want) <= 1e-12 * max(1.0, abs(want)), (scale, got, want)
        g = X.T @ (y - special.expit(eta)) - beta / 100.0
        fd = np.zeros(6)
        for i in range(6):
            h = 1e-6 * max(1.0, abs(beta[i]))
            up, dn = beta.copy(), beta.copy()
            up[i] += h
            dn[i] -= h
            fd[i] = (_table_logp64(tm, up) - _table_logp64(tm, dn)) / (2 * h)
        assert np.max(np.abs(fd - g)) <= 1e-5 * max(1.0, np.max(np.abs(g))), (scale, fd, g)


# ----------------------------------------------------------------------------- sharding / C ABI
def test_observation_sharding_refuses_a_bernoulli_likelihood():
    fn, init, _ = W.logistic_regression(B.ns, 100, 3)
    with pytest.raises(ValueError, match="Normal likelihood"):
        dist.shard_observations(trace(fn, init), 0, 2)


def test_library_term_tags():
    """7 (Bernoulli) passes the tag check; 6 (the value of B2M_SAMPLE_CATEGORICAL in b2m_sample) and 99 do not"""
    lib = _cabi.load()
    assert _cabi.ABI_VERSION == 4 and lib.b2m_abi_version() == 4
    for tag in (6, 99):
        t = (_cabi.Term * 1)()
        t[0].dist, t[0].length = tag, 1
        assert lib.b2m_model_create(t, 1, None, 0, None, 0, 1, None, ctypes.byref(ctypes.c_void_p())) != 0
        assert b"unknown distribution tag" in lib.b2m_last_error()
    t = (_cabi.Term * 1)()
    t[0].dist, t[0].length, t[0].weight = BERNOULLI, 1, 1.0
    t[0].x.kind, t[0].x.c = 0, 1.0          # constant label 1, constant logit 0
    h = ctypes.c_void_p()
    rc = lib.b2m_model_create(t, 1, None, 0, None, 0, 1, None, ctypes.byref(h))
    if rc == 0:                              # a device is present
        lib.b2m_model_destroy(h)
    else:                                    # no device here: the failure is the allocation, not the tag
        assert b"unknown distribution tag" not in lib.b2m_last_error()
