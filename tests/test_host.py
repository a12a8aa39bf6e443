"""CPU: tracer, host distribution classes, API surface, and that the C-ABI library loads and exports
every symbol include/b200mcmc.h declares (no compute calls)."""
import ctypes
import math
import os
import re

import numpy as np
import pytest

import mlx_mcmc_b200 as B
import mlx_mcmc_b200.core as mx
from mlx_mcmc_b200 import _cabi, tracer, workloads as W
from mlx_mcmc_b200.tracer import (EXPONENTIAL, GAMMA, NORMAL, OP_CONST, OP_DATA, OP_LIN, OP_MATVEC, OP_PARAM,
                                  OP_PARAMVEC, UnsupportedOpError, trace)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ----------------------------------------------------------------------------- C ABI
def test_library_loads_and_exports_every_declared_symbol():
    lib = _cabi.load()
    header = open(os.path.join(ROOT, "include", "b200mcmc.h")).read()
    declared = set(re.findall(r"\b(b2m_[a-z_0-9]+)\s*\(", header))
    assert declared == set(_cabi.EXPORTS), declared ^ set(_cabi.EXPORTS)
    for sym in declared:
        assert hasattr(lib, sym), f"{sym} not exported"
    assert lib.b2m_abi_version() == _cabi.ABI_VERSION
    sizes = (ctypes.c_int32 * 6)()
    lib.b2m_struct_sizes(sizes)
    assert list(sizes) == [ctypes.sizeof(t) for t in (_cabi.Term, _cabi.Operand, _cabi.LinEntry, _cabi.HmcArgs,
                                                        _cabi.MhArgs, _cabi.NutsArgs)]


def test_library_is_sm100a_only():
    import subprocess
    out = subprocess.run(["cuobjdump", "--list-elf", _cabi.lib_path()], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_bad_arguments_return_errors_not_crashes():
    lib = _cabi.load()
    assert lib.b2m_model_create(None, 0, None, 0, None, 0, 1, None, ctypes.byref(ctypes.c_void_p())) != 0
    assert b"terms" in lib.b2m_last_error()
    t = (_cabi.Term * 1)()
    t[0].dist = 99
    t[0].length = 1
    assert lib.b2m_model_create(t, 1, None, 0, None, 0, 1, None, ctypes.byref(ctypes.c_void_p())) != 0
    assert b"unknown distribution" in lib.b2m_last_error()
    # options travel in the ABI (they were environment variables in ABI 1): bad values are errors, not defaults
    opt = _cabi.ModelOptions()
    opt.glm_path = 9
    assert lib.b2m_model_create(t, 1, None, 0, None, 0, 1, ctypes.byref(opt), ctypes.byref(ctypes.c_void_p())) != 0
    assert b"glm_path" in lib.b2m_last_error()
    opt.glm_path = 0
    opt.reserved[2] = 1
    assert lib.b2m_model_create(t, 1, None, 0, None, 0, 1, ctypes.byref(opt), ctypes.byref(ctypes.c_void_p())) != 0
    assert b"reserved" in lib.b2m_last_error()
    assert lib.b2m_hmc_run(None, None, None) != 0
    assert lib.b2m_quantiles(None, 0, None, 0, None, None) != 0
    assert lib.b2m_mass_from_draws(None, 0, 0, 0, None, None) != 0
    assert lib.b2m_peer_alloc(0, None, None) != 0
    assert lib.b2m_model_peer_attach(None, None, 2, 0, 512, 0) != 0


# ----------------------------------------------------------------------------- tracer
def test_trace_c1_all_three_idioms_give_the_same_table():
    tabs = []
    for style in ("vector", "unrolled", "stack"):
        fn, init, meta = W.c1_normal(B.ns, style=style)
        tm = trace(fn, init)
        assert tm.D == 2 and len(tm.terms) == 3 and not tm.is_glm
        lik = tm.terms[2]
        assert (lik.dist, lik.length, lik.x.kind, lik.p0.kind, lik.p1.kind) == (NORMAL, 100, OP_DATA, OP_PARAM, OP_PARAM)
        np.testing.assert_array_equal(tm.arrays[lik.x.a], meta.y.astype(np.float32))
        tabs.append(tm.describe())
    assert tabs[0] == tabs[1] == tabs[2]


def test_trace_c2_and_param_in_scale_slot():
    fn, init, _ = W.c2_event_rate(B.ns, style="unrolled")
    tm = trace(fn, init)
    assert [t.dist for t in tm.terms] == [GAMMA, EXPONENTIAL] and tm.terms[1].length == 50
    assert tm.terms[0].k[0] == 2.0 and abs(tm.terms[0].k[1]) < 1e-7       # lgamma(2) = 0
    fn, init, _ = W.t_halfnormal_scale(B.ns)
    tm = trace(fn, init)
    t = tm.terms[1]
    assert (t.x.kind, t.x.c, t.p0.kind, t.p1.kind, t.p1.a) == (OP_CONST, 0.5, OP_CONST, OP_PARAM, 0)


def test_trace_regression_is_glm_class():
    fn, init, meta = W.regression(B.ns, 64, 5)
    tm = trace(fn, init)
    assert tm.is_glm and tm.D == 5
    prior, lik = tm.terms
    assert prior.x.kind == OP_PARAMVEC and prior.length == 5
    assert lik.p0.kind == OP_MATVEC and lik.length == 64 and tm.arrays[lik.p0.a].shape == (64, 5)


def test_trace_affine_operands_and_weights():
    x = np.linspace(-1, 1, 7).astype(np.float32)
    y = (2 * x + 1).astype(np.float32)

    def log_prob(p):
        mean = p["a"] + p["b"] * mx.array(x)
        return 0.5 * mx.sum(B.Normal(mean, 2.0).log_prob(mx.array(y))) - B.Normal(0, 1).log_prob(p["a"]) * 2 + 3.0

    tm = trace(log_prob, {"a": 0.0, "b": 0.0})
    lik = tm.terms[0]
    assert lik.p0.kind == OP_LIN and lik.weight == 0.5 and lik.length == 7
    ents = tm.lin[lik.p0.a: lik.p0.a + lik.p0.b]
    assert (0, -1, 1.0) in ents and any(e[0] == 1 and e[1] >= 0 for e in ents)
    assert tm.terms[1].weight == -2.0
    assert tm.terms[-1].dist == tracer.CONSTANT and tm.terms[-1].k[0] == 3.0


@pytest.mark.parametrize("body, needle", [
    (lambda p: B.Normal(0, 1).log_prob(mx.log(p["x"])), "mx.log of a traced value"),
    (lambda p: B.Normal(0, 1).log_prob(p["x"] * p["x"]), "product of two traced values"),
    (lambda p: B.Normal(0, 1).log_prob(p["x"]) if float(p["x"]) > 0 else 0.0, "float()"),
    (lambda p: B.Gamma(p["x"], 1.0).log_prob(2.0), "shape parameter"),
    (lambda p: B.Categorical(probs=[p["x"], 0.5]).log_prob(0), "Categorical with traced"),
    (lambda p: p["x"] + 1.0, "raw expression"),
    (lambda p: B.Normal(0, 1).log_prob(mx.array(np.ones(3, dtype=np.float32)) * p["x"]), "scalar"),
    (lambda p: 1.0, "does not depend"),
])
def test_unsupported_ops_raise_at_trace_time(body, needle):
    with pytest.raises(UnsupportedOpError) as e:
        trace(body, {"x": 0.5})
    assert needle in str(e.value)


# ----------------------------------------------------------------------------- host distribution classes
def test_known_answers_host_classes():
    """The reference's known-answer tests (tests/test_distributions.py:18-32,67-79;
    tests/test_new_distributions.py:18-37,89-99,144-154,203-226)."""
    assert np.isclose(float(B.Normal(0, 1).log_prob(0.0)), -0.5 * math.log(2 * math.pi), rtol=1e-5)
    assert float(B.Normal(0, 1).log_prob(1.0)) == float(B.Normal(0, 1).log_prob(-1.0))
    assert np.isclose(float(B.HalfNormal(1).log_prob(0.0)), math.log(2) - 0.5 * math.log(2 * math.pi), rtol=1e-5)
    assert float(B.HalfNormal(1).log_prob(-1.0)) == -math.inf
    for x in (-0.1, 1.5, 0.0, 1.0):
        assert float(B.Beta(2, 2).log_prob(x)) == -math.inf
    assert math.isfinite(float(B.Beta(2, 2).log_prob(0.5)))
    assert float(B.Gamma(2, 1).log_prob(-1.0)) == -math.inf and float(B.Gamma(2, 1).log_prob(1.5)) < 0
    assert np.isclose(float(B.Exponential(2).log_prob(0.0)), math.log(2)) and float(B.Exponential(2).log_prob(-1.0)) == -math.inf
    c = B.Categorical(probs=[0.2, 0.5, 0.3])
    assert np.isclose(float(c.log_prob(0)), math.log(0.2), rtol=1e-2) and np.isclose(float(c.log_prob(1)), math.log(0.5), rtol=1e-2)
    assert float(c.log_prob(-1)) == -math.inf and float(c.log_prob(3)) == -math.inf
    with pytest.raises(ValueError):
        B.Categorical()
    with pytest.raises(ValueError):
        B.Categorical(probs=[0.5, 0.5], logits=[0.0, 0.0])
    assert np.isclose(float(B.Beta(2, 5).mean()), 2 / 7) and np.isclose(float(B.Gamma(3, 2).mean()), 1.5)
    assert np.isclose(float(B.Exponential(4).mean()), 0.25) and int(B.Categorical(probs=[.1, .7, .2]).mode()) == 1


def test_host_classes_agree_with_oracle_classes():
    from oracle.ns import ns as ons
    xs = np.array([-1.0, 0.0, 0.3, 0.99, 2.5], dtype=np.float32)
    pairs = [(B.Normal(0.5, 1.5), ons.Normal(0.5, 1.5)), (B.HalfNormal(2.0), ons.HalfNormal(2.0)),
             (B.Exponential(1.7), ons.Exponential(1.7)), (B.Gamma(2.5, 0.7), ons.Gamma(2.5, 0.7)),
             (B.Beta(2.0, 3.0), ons.Beta(2.0, 3.0))]
    for mine, theirs in pairs:
        a, b = np.asarray(mine.log_prob(xs)), np.asarray(theirs.log_prob(ons.mx.array(xs)))
        np.testing.assert_allclose(a, b, rtol=2e-6, atol=1e-6)


def test_sampling_moments():
    k = mx.random.key(0)
    assert abs(np.mean(B.Normal(2.0, 3.0).sample(k, (20000,))) - 2.0) < 0.1
    assert np.all(B.HalfNormal(1.0).sample(k, (1000,)) >= 0)
    assert abs(np.mean(B.Gamma(3.0, 2.0).sample(k, (20000,))) - 1.5) < 0.05
    assert abs(np.mean(B.Beta(2.0, 5.0).sample(k, (20000,))) - 2 / 7) < 0.02
    assert abs(np.mean(B.Exponential(4.0).sample(k, (20000,))) - 0.25) < 0.02
    s = B.Categorical(probs=[0.2, 0.5, 0.3]).sample(k, (20000,))
    assert abs(np.mean(s == 1) - 0.5) < 0.02


# ----------------------------------------------------------------------------- API surface
def test_export_list_matches_reference():
    for name in ["Normal", "HalfNormal", "Beta", "Gamma", "Exponential", "Categorical", "metropolis_hastings", "hmc",
                 "nuts", "MCMC"]:
        assert name in B.__all__ and hasattr(B, name)


def test_mcmc_errors_before_any_device_work():
    m = B.MCMC(lambda p: B.Normal(0, 1).log_prob(p["x"]))
    with pytest.raises(ValueError, match="Unknown sampling method"):
        m.run({"x": 0.0}, method="gibbs", verbose=False)
    with pytest.raises(ValueError, match="Must run sampling first"):
        m.summary()
    with pytest.raises(ZeroDivisionError):
        B.hmc(lambda p: B.Normal(0, 1).log_prob(p["x"]), {"x": 0.0}, num_warmup=0)
    with pytest.raises(ZeroDivisionError):
        B.nuts(lambda p: B.Normal(0, 1).log_prob(p["x"]), {"x": 0.0}, num_warmup=0)


def test_run_extension_keywords_are_validated_before_device_work():
    m = B.MCMC(lambda p: B.Normal(0, 1).log_prob(p["x"]))
    with pytest.raises(ValueError, match="shard"):
        m.run({"x": 0.0}, method="nuts", shard="rows", verbose=False)
    with pytest.raises(ValueError, match="one process drives one GPU"):
        m.run({"x": 0.0}, method="nuts", devices=[0, 1], verbose=False)


def test_sampler_option_validation_happens_on_the_host():
    fn, init = (lambda p: B.Normal(0, 1).log_prob(p["x"])), {"x": 0.0}
    with pytest.raises(ValueError, match="compat"):
        B.nuts(fn, init, compat="fast")
    with pytest.raises(ValueError, match="step_size_adaptation"):
        B.nuts(fn, init, step_size_adaptation="global")
    with pytest.raises(ValueError, match="step_size_jitter"):
        B.nuts(fn, init, step_size_jitter=1.0)
    with pytest.raises(ValueError, match="max_tree_depth"):
        B.nuts(fn, init, max_tree_depth=0)
    with pytest.raises(ValueError, match="adapt"):
        B.hmc(fn, init, adapt="nesterov")
    with pytest.raises(TypeError):       # kwargs go to the sampler verbatim, as in the reference (mcmc.py:156,177)
        B.MCMC(fn).run(init, method="metropolis", step_size=0.1, verbose=False)


def test_device_only_helpers_refuse_host_input():
    import torch
    from mlx_mcmc_b200.diagnostics import device_series_stats
    with pytest.raises(ValueError, match="CUDA"):
        device_series_stats(torch.zeros(4, 2, 3))
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="CUDA"):
            B.Normal(0, 1).sample_device(B.core.random.key(0), (4,))


def test_product_never_imports_the_oracle():
    import subprocess
    import sys
    code = ("import sys; import mlx_mcmc_b200, mlx_mcmc_b200.engine, mlx_mcmc_b200.workloads; "
            "bad=[m for m in sys.modules if m.split('.')[0] in ('oracle','mlx')]; print(bad); sys.exit(1 if bad else 0)")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


def test_no_cuda_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(RuntimeError, match="no CUDA device"):
        B.MCMC(lambda p: B.Normal(0, 1).log_prob(p["x"])).run({"x": 0.0}, num_samples=5, num_warmup=5, verbose=False)


@pytest.mark.parametrize("name", sorted(W.ALL_SMALL))
def test_traced_table_means_what_the_model_says(name):
    """Tracing preserves the model: a plain float64 evaluation of the term table (tests/table_eval.py) gives the
    oracle's log p and gradient at the initial point and at perturbed points inside the support."""
    from oracle.ns import ns as ons, value_and_grad
    from table_eval import table_grad, table_logp
    fn, init, _ = W.ALL_SMALL[name](B.ns)
    fo, _, _ = W.ALL_SMALL[name](ons)
    model = trace(fn, init)
    rng = np.random.default_rng(7)
    for trial in range(3):
        params = {k: (np.asarray(v, dtype=np.float64) * (1.0 + 0.1 * trial * rng.uniform(-1, 1, np.shape(v)))
                      + 0.01 * trial * rng.uniform(0, 1, np.shape(v))) for k, v in init.items()}
        params = {k: (float(v) if np.ndim(v) == 0 else v) for k, v in params.items()}
        lp64, g64 = value_and_grad(fo, params, "float64")
        theta = np.concatenate([np.atleast_1d(np.asarray(params[k], dtype=np.float64)).ravel() for k in model.layout])
        want = np.concatenate([np.atleast_1d(g64[k]).ravel() for k in model.layout])
        # the table holds observations and normalising constants in float32 (the reference's device dtype), the
        # oracle call keeps float64: the bound is float32 rounding of the largest addend
        scale = max([1.0, abs(lp64)] + [abs(k) for t in model.terms for k in t.k])
        assert abs(table_logp(model, theta) - lp64) <= 2e-7 * scale, (name, trial)
        got = table_grad(model, theta)
        assert np.max(np.abs(got - want)) <= 1e-5 * max(1.0, np.max(np.abs(want))), (name, trial, got, want)


def _idiom_models():
    """namespace-generic models exercising the tracer's operand forms beyond the benchmark workloads"""
    x = np.linspace(-1, 1, 7).astype(np.float32)
    y = (2 * x + 1 + 0.1 * np.cos(5 * x)).astype(np.float32)
    t = np.array([0.3, 1.1, 0.2, 0.7], dtype=np.float32)

    def affine(ns):       # OP_LIN location, fractional / negative weights, additive constant
        def f(p):
            mean = p["a"] + p["b"] * ns.mx.array(x) - 0.25
            return (0.5 * ns.mx.sum(ns.Normal(mean, 2.0).log_prob(ns.mx.array(y)))
                    - ns.Normal(0, 1).log_prob(p["a"]) * 2 + 3.0 + ns.Normal(1.0, 3.0).log_prob(p["b"]) / 4)
        return f, {"a": 0.3, "b": -0.2}

    def unrolled(ns):     # python loop over observations + parameter in the scale slot (examples/01:46-48)
        def f(p):
            lp = ns.HalfNormal(5.0).log_prob(p["s"]) + ns.Gamma(2.0, 1.5).log_prob(p["r"])
            for ti in t:
                lp = lp + ns.Exponential(p["r"]).log_prob(ns.mx.array(ti))
            for yi in y[:3]:
                lp += ns.Normal(0.5, p["s"]).log_prob(ns.mx.array(yi))
            return lp
        return f, {"s": 1.2, "r": 0.8}

    def stacked(ns):      # mx.array([...traced scalars...]) summed (tests/test_nuts.py:205-207)
        def f(p):
            return (ns.mx.sum(ns.mx.array([ns.Normal(p["m"] * float(xi), 0.7).log_prob(ns.mx.array(yi)) for xi, yi in zip(x, y)]))
                    + ns.Beta(2.0, 3.0).log_prob(p["q"]) + ns.Normal(p["m"], 2.0).log_prob(0.1))
        return f, {"m": 0.4, "q": 0.35}

    return {"affine": affine, "unrolled": unrolled, "stacked": stacked}


@pytest.mark.parametrize("name", ["affine", "unrolled", "stacked"])
def test_traced_idioms_keep_value_and_gradient(name):
    from oracle.ns import ns as ons, value_and_grad
    from table_eval import table_grad, table_logp
    fn, init = _idiom_models()[name](B.ns)
    fo, _ = _idiom_models()[name](ons)
    model = trace(fn, init)
    rng = np.random.default_rng(11)
    for trial in range(3):
        params = {k: float(v * (1.0 + 0.2 * trial * rng.uniform(-1, 1))) for k, v in init.items()}
        lp64, g64 = value_and_grad(fo, params, "float64")
        theta = np.array([params[k] for k in model.layout], dtype=np.float64)
        want = np.array([float(g64[k]) for k in model.layout])
        scale = max([1.0, abs(lp64)] + [abs(k) for t in model.terms for k in t.k])
        assert abs(table_logp(model, theta) - lp64) <= 5e-7 * scale, (name, trial, table_logp(model, theta), lp64)
        assert np.max(np.abs(table_grad(model, theta) - want)) <= 1e-5 * max(1.0, np.max(np.abs(want))), (name, trial)


# ----------------------------------------------------------------------------- round 2: host logic of the new features
def test_list_valued_observations_give_a_full_length_term():
    """ADVICE r01: `Normal(mu, 1).log_prob([1.0, 2.0, 3.0])` -- the reference does `value = mx.array(value)`, so a Python
    list is data; it must trace to a length-3 term over an observed array, never to its first element."""
    t = B.trace(lambda p: mx.sum(B.Normal(p["mu"], 1.0).log_prob([1.0, 2.0, 3.0])), {"mu": 0.0})
    assert len(t.terms) == 1 and t.terms[0].length == 3
    assert np.array_equal(t.arrays[t.terms[0].x.a], np.asarray([1.0, 2.0, 3.0], dtype=np.float32))
    t2 = B.trace(lambda p: mx.sum(B.Normal([0.5, 1.5], (2.0, 3.0)).log_prob(p["x"])), {"x": np.zeros(2, dtype=np.float32)})
    assert t2.terms[0].length == 2 and t2.terms[0].p0.kind == 2 and t2.terms[0].p1.kind == 2
    with pytest.raises(B.UnsupportedOpError):     # lengths that do not broadcast are an error, not a truncation
        B.trace(lambda p: mx.sum(B.Normal(p["mu"], np.ones(2, dtype=np.float32)).log_prob(np.ones(3, dtype=np.float32))), {"mu": 0.0})


def test_transform_codes_follow_the_support_of_the_value_distribution():
    from mlx_mcmc_b200 import workloads as W
    want = {"c1_normal": [0, 1], "c2_event_rate": [1], "c5_ab_test": [2, 2], "t_normal_2d": [0, 0], "t_halfnormal_scale": [1],
            "t_regression_sigma": [0, 0, 0, 0, 1], "t_regression_small": [0, 0, 0]}
    for name, codes in want.items():
        fn, init, _ = W.ALL_SMALL[name](B.ns)
        assert B.trace(fn, init).transform_codes().tolist() == codes, name
    # a parameter claimed by a positive AND a unit-interval distribution keeps its own coordinate
    t = B.trace(lambda p: B.HalfNormal(1.0).log_prob(p["x"]) + B.Beta(2, 2).log_prob(p["x"]), {"x": 0.5})
    assert t.transform_codes().tolist() == [0]


def test_warmup_window_schedule():
    from mlx_mcmc_b200.kernels._common import warmup_windows
    assert warmup_windows(10) == [(0, 10, False)]
    assert warmup_windows(1000) == [(0, 75, False), (75, 100, True), (100, 150, True), (150, 250, True), (250, 450, True),
                                    (450, 950, True), (950, 1000, False)]
    assert warmup_windows(200) == [(0, 75, False), (75, 100, True), (100, 150, True), (150, 200, False)]
    for n in (20, 33, 60, 100, 149, 150, 151, 333, 2000):
        segs = warmup_windows(n)
        assert segs[0][0] == 0 and segs[-1][1] == n and all(a[1] == b[0] for a, b in zip(segs, segs[1:]))
        assert all(e > s for s, e, _ in segs) and any(u for _, _, u in segs)


def test_model_cache_is_keyed_by_the_content_of_the_trace():
    """ADVICE r01: the cache must not serve a stale model when the data a log_prob closes over changes; it is keyed by a
    fingerprint of the re-traced terms and observed arrays, and bounded."""
    from mlx_mcmc_b200 import engine
    y = np.arange(6, dtype=np.float32)

    def fn(p):
        return mx.sum(B.Normal(p["mu"], 1.0).log_prob(mx.array(y)))

    k1 = engine._trace_fingerprint(B.trace(fn, {"mu": 0.0}), (0,))
    assert k1 == engine._trace_fingerprint(B.trace(fn, {"mu": 0.0}), (0,))
    y[3] = 99.0                                     # same function object, same shapes, different data
    k2 = engine._trace_fingerprint(B.trace(fn, {"mu": 0.0}), (0,))
    assert k1 != k2
    y[3], y[4] = y[4], 99.0                         # a permutation is a different data set too
    assert engine._trace_fingerprint(B.trace(fn, {"mu": 0.0}), (0,)) != k2
    assert k1 != engine._trace_fingerprint(B.trace(fn, {"mu": 0.0}), (0, "tc"))      # options are part of the key
    big = np.random.default_rng(0).standard_normal((3000, 40)).astype(np.float32)   # id-keyed inside the tracer
    f1 = engine._array_fingerprint(big)
    big[1234, 7] += 1.0
    assert engine._array_fingerprint(big) != f1
    assert engine._CACHE_SIZE <= 8 and callable(engine.clear_model_cache)


def test_peer_window_layout_is_what_the_header_documents():
    """b2m_model_peer_bytes validates its arguments on the host (no device work)."""
    lib = _cabi.load()
    n = ctypes.c_int64()
    assert lib.b2m_model_peer_bytes(None, 4096, 8, ctypes.byref(n)) != 0
    assert b"NULL" in lib.b2m_last_error()
    assert lib.b2m_options_size() == ctypes.sizeof(_cabi.ModelOptions)


def test_specialised_kernels_compile_with_nvrtc_on_the_cpu_box():
    """mlx_mcmc_b200/jit.py: the translation unit generated for a traced model compiles with NVRTC for sm_100a (no GPU
    needed to compile) and exports the four entry points b2m_model_attach_module looks up; ineligible models are refused."""
    from mlx_mcmc_b200 import jit as J
    if not J.available():
        pytest.skip("cuda-python / NVRTC not importable here")
    fn, init, _ = W.c2_event_rate(B.ns)
    tr = B.trace(fn, init)
    assert J.eligible(tr) and J.dmax_for(tr.D) == 2
    src = J.generate_source(tr, tr.transform_codes())
    assert "#define B2M_JIT_HAS_TF 1" in src and src.count("  F(") == len(tr.terms)
    assert "jit_const(0x" in src                      # constants travel as opaque bit patterns (bit-identity with the interpreter)
    cubin = J.compile_cubin(src)
    assert cubin[:4] == b"\x7fELF" and len(cubin) > 10000
    for name in (b"b2m_jit_logp_grad", b"b2m_jit_hmc", b"b2m_jit_mh", b"b2m_jit_nuts"):
        assert name in cubin
    assert J.compile_cubin(src) is cubin              # memory cache
    fr, ir, _ = W.t_regression_small(B.ns)
    assert not J.eligible(B.trace(fr, ir))            # GLM class: the tensor-core path, not these kernels
    affine = B.trace(lambda p: mx.sum(B.Normal(p["a"] + p["b"] * mx.array(np.arange(4.0)), 1.0).log_prob(mx.array(np.ones(4)))),
                     {"a": 0.0, "b": 0.0})
    assert not J.eligible(affine)                     # affine operands keep the interpreter kernels
