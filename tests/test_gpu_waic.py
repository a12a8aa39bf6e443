"""GPU: pointwise log-likelihood statistics (b2m_loglik_stats) and WAIC against float64 evaluations of the traced term
table on the same draws -- GLM class on the three contraction paths, the pointwise class, a C4-size model, a conjugate
model with known answers, MCMC.waic end to end, model comparison, determinism and refusals."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import mlx_mcmc_b200 as B
from mlx_mcmc_b200 import _cabi, tracer as T, workloads as W
from mlx_mcmc_b200.diagnostics import waic, waic_compare, waic_totals
from mlx_mcmc_b200.engine import compile_model

pytestmark = pytest.mark.gpu
mx = B.ns.mx


# ----------------------------------------------------------------------------- float64 reference on the device
def _ll64(tm, theta, cols=None):
    """[S, N] float64 pointwise log-likelihood of the observation terms of traced model `tm` at theta [S, D] (float64
    CUDA); `cols` restricts a single-term model to those observations"""
    dev = theta.device
    arr = lambda a: torch.as_tensor(np.asarray(tm.arrays[a], dtype=np.float64), device=dev)  # noqa: E731
    out = []
    for i in tm.observation_terms():
        t = tm.terms[i]

        def op(o):
            if o.kind == T.OP_CONST:
                return torch.full((1, 1), o.c, dtype=torch.float64, device=dev)
            if o.kind == T.OP_PARAM:
                return theta[:, o.a:o.a + 1]
            if o.kind == T.OP_DATA:
                v = arr(o.a)[: t.length]
                return (v if cols is None else v[cols])[None, :]
            if o.kind == T.OP_PARAMVEC:
                return theta[:, o.a:o.a + o.b]
            if o.kind == T.OP_LIN:
                v = torch.full((1, 1), o.c, dtype=torch.float64, device=dev)
                for p, a, coef in o.lin:
                    e = coef * (arr(a)[None, :] if a >= 0 else 1.0)
                    if a >= 0 and cols is not None:
                        e = e[:, cols]
                    v = v + e * (theta[:, p:p + 1] if p >= 0 else 1.0)
                return v
            X = arr(o.a)
            if cols is not None:
                X = X[cols]
            return theta[:, o.b:o.b + X.shape[1]] @ X.T + o.c
        x, p0, p1 = op(t.x), op(t.p0), op(t.p1)
        if t.dist == T.NORMAL:
            ll = -0.5 * math.log(2 * math.pi) - torch.log(p1) - 0.5 * ((x - p0) / p1) ** 2
        elif t.dist == T.EXPONENTIAL:
            ll = torch.where(x >= 0, torch.log(p0) - p0 * x, torch.full_like(x * p0, -math.inf))
        elif t.dist == T.BERNOULLI:
            ll = x * p0 - torch.nn.functional.softplus(p0)
        else:
            raise AssertionError(t.dist)
        n = t.length if cols is None else len(cols)
        out.append(t.weight * ll.expand(theta.shape[0], n))
    return torch.cat(out, dim=1)


def _stats64(ll):
    S = ll.shape[0]
    return ((torch.logsumexp(ll, 0) - math.log(S)).cpu().numpy(), ll.mean(0).cpu().numpy(),
            ll.var(0, unbiased=True).cpu().numpy())


def _check(res, ref, cols=None):
    lppd, mean, var = ref
    pw = res["pointwise"]
    g_l, g_m, g_v = pw["lppd"], pw["mean"], pw["p_waic"]
    if cols is not None:
        g_l, g_m, g_v = g_l[cols], g_m[cols], g_v[cols]
    err_l = np.max(np.abs(g_l - lppd) / np.maximum(1.0, np.abs(lppd)))
    err_m = np.max(np.abs(g_m - mean) / np.maximum(1.0, np.abs(mean)))
    err_v = np.max(np.abs(g_v - var) - (1e-3 * var + 1e-6))
    assert err_l <= 1e-5, f"lppd error {err_l:.3g}"
    assert err_m <= 1e-5, f"mean error {err_m:.3g}"
    assert err_v <= 0, f"var error over the bar by {err_v:.3g}"
    if cols is None:
        tot = waic_totals(lppd, mean, var, res["n_draws"])
        for k in ("elpd_waic", "p_waic"):
            assert abs(res[k] - tot[k]) <= 1e-5 * max(1.0, abs(tot[k])), (k, res[k], tot[k])


def _draws(center, spread, S, Cn, seed, positive=None):
    rs = np.random.default_rng(seed)
    d = center[None, None, :] + spread * rs.standard_normal((S, Cn, center.size))
    if positive is not None:
        d[..., positive] = np.abs(d[..., positive]) + 0.2
    return torch.from_numpy(d.astype(np.float32)).cuda()


def _glm_case(kind, n, d, seed=0):
    rs = np.random.default_rng(seed)
    X = rs.standard_normal((n, d)).astype(np.float32)
    beta = (rs.standard_normal(d) / np.sqrt(d)).astype(np.float32)
    Xa = mx.array(X)
    if kind == "logit":
        eta = X.astype(np.float64) @ beta
        y = (rs.uniform(size=n) < 1 / (1 + np.exp(-eta))).astype(np.float32)

        def fn(p):
            return mx.sum(B.ns.Normal(0, 5.0).log_prob(p["beta"])) + mx.sum(B.ns.Bernoulli(logits=Xa @ p["beta"]).log_prob(mx.array(y)))
        return fn, {"beta": np.zeros(d, np.float32)}, beta, None
    c, w, s = (1.5, 0.7, 0.9) if kind == "normal_cw" else (0.0, 1.0, 0.8)
    y = (X @ beta + c + s * rs.standard_normal(n)).astype(np.float32)
    ya = mx.array(y)
    if kind == "normal_sigma":
        def fn(p):
            return (mx.sum(B.ns.Normal(0, 5.0).log_prob(p["beta"])) + B.ns.HalfNormal(2.0).log_prob(p["sigma"])
                    + mx.sum(B.ns.Normal(Xa @ p["beta"], p["sigma"]).log_prob(ya)))
        return fn, {"beta": np.zeros(d, np.float32), "sigma": 1.0}, np.concatenate([beta, [s]]), [d]

    def fn(p):
        return mx.sum(B.ns.Normal(0, 5.0).log_prob(p["beta"])) + w * mx.sum(B.ns.Normal(Xa @ p["beta"] + c, s).log_prob(ya))
    return fn, {"beta": np.zeros(d, np.float32)}, beta, None


# ----------------------------------------------------------------------------- 1. GLM class against float64
@pytest.mark.parametrize("path", ["simt", "tc", "tc16"])
@pytest.mark.parametrize("kind", ["normal_const", "normal_sigma", "normal_cw", "logit", "logit_far"])
@pytest.mark.parametrize("n,d,S,Cn", [(1000, 37, 3, 97), (255, 63, 1, 129), (4097, 129, 2, 150)])
def test_glm_against_float64(cuda, path, kind, n, d, S, Cn):
    fn, init, center, pos = _glm_case("logit" if kind == "logit_far" else kind, n, d, seed=n + d)
    model = compile_model(fn, init, cache=False, glm_path=path)
    spread = 0.05
    if kind == "logit_far":
        # draws far from the posterior: |eta| up to ~100, where ll ~ -100 and exp(ll) underflows without the max shift
        t = model.traced.terms[model.traced.observation_terms()[0]]
        center = center * (60.0 / np.max(np.abs(np.asarray(model.traced.arrays[t.p0.a]) @ center)))
        spread = 0.3
    draws = _draws(center, spread, S, Cn, seed=1, positive=pos)
    res = waic(model, draws)
    ref = _stats64(_ll64(model.traced, draws.reshape(-1, model.D).double()))
    if kind == "logit_far":
        assert np.min(ref[1]) < -20
    _check(res, ref)


# ----------------------------------------------------------------------------- 2. C4 size
@pytest.mark.parametrize("path", ["tc", "tc16"])
def test_c4_size_exact_posterior(cuda, path):
    fn, init, meta = W.regression(B.ns, 100000, 1000, seed=0)
    m, V = W.regression_posterior(meta)
    L = torch.linalg.cholesky(torch.from_numpy(V).cuda())
    g = torch.Generator(device="cuda").manual_seed(5)
    z = torch.randn((16 * 4096, 1000), dtype=torch.float64, device="cuda", generator=g)
    draws = (torch.from_numpy(m).cuda()[None, :] + z @ L.T).float().reshape(16, 4096, 1000)
    del z
    model = compile_model(fn, init, cache=False, glm_path=path)
    res = waic(model, draws)
    cols = np.sort(np.random.default_rng(0).choice(100000, 1024, replace=False))
    ref = _stats64(_ll64(model.traced, draws.reshape(-1, 1000).double(), cols=torch.from_numpy(cols).cuda()))
    _check(res, ref, cols)


# ----------------------------------------------------------------------------- 3. known answer
def test_conjugate_normal_known_answer(cuda):
    fn, init, meta = W.regression(B.ns, 200, 5, seed=4, noise=0.8)
    m, V = W.regression_posterior(meta)
    S = 1 << 20
    L = torch.linalg.cholesky(torch.from_numpy(V).cuda())
    g = torch.Generator(device="cuda").manual_seed(9)
    th = torch.from_numpy(m).cuda()[None, :] + torch.randn((S, 5), dtype=torch.float64, device="cuda", generator=g) @ L.T
    model = compile_model(fn, init, cache=False)
    res = waic(model, th.float().reshape(S, 1, 5))
    X, y, s2 = meta.X.astype(np.float64), meta.y.astype(np.float64), meta.noise ** 2
    q = np.einsum("nd,de,ne->n", X, V, X)          # x_n' V x_n
    mu = y - X @ m
    lppd_true = -0.5 * np.log(2 * np.pi * (s2 + q)) - 0.5 * mu ** 2 / (s2 + q)
    var_true = (2 * q ** 2 + 4 * mu ** 2 * q) / (4 * s2 ** 2)
    # Monte Carlo standard errors from the draws themselves
    ll = _ll64(model.traced, th.float().double())
    S_ = ll.shape[0]
    e = torch.exp(ll - ll.max(0).values)
    se_lppd = (e.std(0) / e.mean(0) / math.sqrt(S_)).cpu().numpy()
    c = ll - ll.mean(0)
    se_var = torch.sqrt(((c ** 4).mean(0) - ll.var(0) ** 2) / S_).cpu().numpy()
    pw = res["pointwise"]
    assert np.all(np.abs(pw["lppd"] - lppd_true) <= 5 * se_lppd + 1e-7), np.max(np.abs(pw["lppd"] - lppd_true) / se_lppd)
    assert np.all(np.abs(pw["p_waic"] - var_true) <= 5 * se_var + 1e-9), np.max(np.abs(pw["p_waic"] - var_true) / se_var)


# ----------------------------------------------------------------------------- 4. pointwise class
def _two_arrays():
    rs = np.random.default_rng(0)
    a, b = rs.normal(1.0, 1.5, 70).astype(np.float32), rs.exponential(0.5, 33).astype(np.float32)

    def fn(p):
        return (B.ns.Normal(0, 5).log_prob(p["mu"]) + B.ns.Exponential(1.0).log_prob(p["rate"])
                + mx.sum(B.ns.Normal(p["mu"], 1.5).log_prob(mx.array(a)))
                + mx.sum(B.ns.Exponential(p["rate"]).log_prob(mx.array(b))))
    return fn, {"mu": 0.0, "rate": 1.0}, np.array([1.0, 2.0]), [1]


def _lin_bernoulli():
    rs = np.random.default_rng(1)
    x = rs.normal(size=300).astype(np.float32)
    y = (rs.uniform(size=300) < 1 / (1 + np.exp(-(0.3 + 1.2 * x)))).astype(np.float32)

    def fn(p):
        return (B.ns.Normal(0, 5).log_prob(p["a"]) + B.ns.Normal(0, 5).log_prob(p["b"])
                + mx.sum(B.ns.Bernoulli(logits=p["a"] + p["b"] * mx.array(x)).log_prob(mx.array(y))))
    return fn, {"a": 0.0, "b": 0.0}, np.array([0.3, 1.2]), None


def test_pointwise_class_against_float64(cuda):
    got = []
    for style in ("vector", "unrolled", "stack"):
        fn, init, _ = W.c1_normal(B.ns, style=style)
        model = compile_model(fn, init, cache=False)
        draws = _draws(np.array([5.0, 2.0]), 0.2, 50, 91, seed=2, positive=[1])
        res = waic(model, draws)
        _check(res, _stats64(_ll64(model.traced, draws.reshape(-1, 2).double())))
        got.append(res)
    for r in got[1:]:
        for k in ("lppd", "mean", "p_waic"):
            np.testing.assert_array_equal(r["pointwise"][k], got[0]["pointwise"][k])
    fn, init, _ = W.c2_event_rate(B.ns)
    model = compile_model(fn, init, cache=False)
    draws = _draws(np.array([3.0]), 0.3, 40, 64, seed=3, positive=[0])
    _check(waic(model, draws), _stats64(_ll64(model.traced, draws.reshape(-1, 1).double())))
    for make in (_lin_bernoulli, _two_arrays):
        fn, init, center, pos = make()
        model = compile_model(fn, init, cache=False)
        draws = _draws(center, 0.1, 33, 70, seed=4, positive=pos)
        res = waic(model, draws)
        assert res["n_obs"] == sum(model.traced.terms[i].length for i in model.traced.observation_terms())
        _check(res, _stats64(_ll64(model.traced, draws.reshape(-1, model.D).double())))


def test_glm_with_extra_observed_term(cuda):
    fr, _, meta = W.regression(B.ns, 700, 20, seed=2)
    z = np.linspace(-1, 1, 45).astype(np.float32)

    def fn(p):
        return fr({"beta": p["beta"]}) + mx.sum(B.ns.Normal(p["m"], 2.0).log_prob(mx.array(z)))
    for path in ("simt", "tc16"):
        model = compile_model(fn, {"beta": np.zeros(20, np.float32), "m": 0.0}, cache=False, glm_path=path)
        draws = _draws(np.concatenate([meta.beta_true, [0.1]]), 0.05, 5, 77, seed=6)
        res = waic(model, draws)
        assert res["n_obs"] == 745
        _check(res, _stats64(_ll64(model.traced, draws.reshape(-1, model.D).double())))


# ----------------------------------------------------------------------------- 5. end to end
def _samples_to_theta(model, samples, single):
    parts = []
    for name, (off, n, shp) in model.layout.items():
        x = torch.as_tensor(samples[name]).cuda().double()
        if single:
            x = x[None]
        parts.append(x.reshape(x.shape[0], x.shape[1], n))
    return torch.cat(parts, 2).permute(1, 0, 2).reshape(-1, model.D)


@pytest.mark.parametrize("chains", [1, 256])
@pytest.mark.parametrize("torch_draws", [False, True])
def test_mcmc_waic_end_to_end(cuda, chains, torch_draws):
    fn, init, _ = W.t_regression_small(B.ns)
    m = B.MCMC(fn)
    m.run(init, num_samples=150, num_warmup=150, method="nuts", num_chains=chains, compat="correct",
          return_torch=torch_draws, verbose=False)
    res = m.waic()
    model = compile_model(fn, init)
    theta = _samples_to_theta(model, m.samples, chains == 1)
    assert res["n_draws"] == theta.shape[0] == 150 * chains
    _check(res, _stats64(_ll64(model.traced, theta)))


def test_mcmc_waic_with_transforms(cuda):
    fn, init, _ = W.t_regression_sigma(B.ns)
    m = B.MCMC(fn)
    m.run(init, num_samples=100, num_warmup=150, method="nuts", num_chains=64, compat="correct", transforms="auto",
          verbose=False)
    assert np.all(m.samples["sigma"] > 0)
    res = m.waic()
    model = compile_model(fn, init, transforms="auto")
    _check(res, _stats64(_ll64(model.traced, _samples_to_theta(model, m.samples, False))))


# ----------------------------------------------------------------------------- 6. model comparison
def test_model_comparison_prefers_the_true_model(cuda):
    rs = np.random.default_rng(7)
    n = 400
    X = rs.standard_normal((n, 3)).astype(np.float32)
    y = (X @ np.array([1.0, 0.8, -0.5]) + 0.7 * rs.standard_normal(n)).astype(np.float32)
    res = []
    for cols in ([0, 1, 2], [0, 2]):
        fn, init, meta = W.regression(B.ns, n, len(cols), noise=0.7)
        meta.X, meta.y = X[:, cols].copy(), y
        Xa, ya = mx.array(meta.X), mx.array(y)

        def f(p, Xa=Xa, ya=ya):
            return mx.sum(B.ns.Normal(0, 10.0).log_prob(p["beta"])) + mx.sum(B.ns.Normal(Xa @ p["beta"], 0.7).log_prob(ya))
        m, V = W.regression_posterior(meta)
        L = np.linalg.cholesky(V)
        th = (m[None, :] + rs.standard_normal((4000, len(cols))) @ L.T).astype(np.float32)
        model = compile_model(f, init, cache=False)
        res.append(waic(model, torch.from_numpy(th).cuda().reshape(1000, 4, len(cols))))
    cmp = waic_compare(res[0], res[1])
    assert cmp["elpd_diff"] > 4 * cmp["se_diff"], cmp


# ----------------------------------------------------------------------------- 7. determinism and refusals
def test_repeated_calls_are_bit_equal_and_sampling_is_unaffected(cuda):
    fn, init, meta = W.regression(B.ns, 3000, 70, seed=3)
    for path in ("tc16", "tc", "simt"):
        model = compile_model(fn, init, cache=False, glm_path=path)
        draws = _draws(meta.beta_true.astype(np.float64), 0.03, 7, 300, seed=8)
        theta = draws[0, :64].contiguous()
        lp0, g0 = model.logp_grad(theta)
        s0, _ = B.nuts(fn, init, num_samples=5, num_warmup=5, num_chains=64, model=model, key=mx.random.key(2),
                       return_torch=True)
        a, b = waic(model, draws), waic(model, draws)
        for k in ("lppd", "mean", "p_waic"):
            np.testing.assert_array_equal(a["pointwise"][k], b["pointwise"][k])
        lp1, g1 = model.logp_grad(theta)
        s1, _ = B.nuts(fn, init, num_samples=5, num_warmup=5, num_chains=64, model=model, key=mx.random.key(2),
                       return_torch=True)
        assert torch.equal(lp0, lp1) and torch.equal(g0, g1), path
        assert torch.equal(s0["beta"], s1["beta"]), path


def _raw(model, draws, obs, n_obs):
    out = torch.empty((max(n_obs, 1), 3), dtype=torch.float64, device="cuda")
    idx = (C.c_int32 * len(obs))(*obs)
    return model.lib.b2m_loglik_stats(model.handle, C.c_void_p(draws.data_ptr()), draws.shape[0] * draws.shape[1], idx,
                                      len(obs), C.c_void_p(out.data_ptr()), n_obs,
                                      C.c_void_p(torch.cuda.current_stream().cuda_stream))


def test_refusals(cuda):
    fn5, init5, _ = W.c5_ab_test(B.ns)
    m5 = compile_model(fn5, init5, cache=False)
    d5 = torch.full((4, 8, 2), 0.3, device="cuda")
    with pytest.raises(ValueError, match="no observation terms"):
        waic(m5, d5)
    assert _raw(m5, d5, [0], 1) != 0                     # a prior term
    fn, init, meta = W.regression(B.ns, 300, 6, seed=1)
    model = compile_model(fn, init, cache=False)
    obs = model.traced.observation_terms()
    draws = _draws(meta.beta_true.astype(np.float64), 0.05, 2, 40, seed=1)
    assert _raw(model, draws, obs, 300) == 0
    assert _raw(model, draws, [len(model.traced.terms)], 300) != 0     # out of range
    assert "out of range" in model.lib.b2m_last_error().decode()
    assert _raw(model, draws, [-1], 300) != 0
    prior = [i for i in range(len(model.traced.terms)) if i not in obs]
    assert _raw(model, draws, prior, 6) != 0                          # a prior term
    assert "not an observation term" in model.lib.b2m_last_error().decode()
    assert _raw(model, draws, obs, 299) != 0                          # wrong n_obs
    assert "n_obs" in model.lib.b2m_last_error().decode()
    bad = draws.clone()
    bad[1, 3, 2] = float("nan")
    with pytest.raises(ValueError, match="non-finite"):
        waic(model, bad)
    with pytest.raises(ValueError, match="D ="):
        waic(model, draws[:, :, :5].contiguous())
