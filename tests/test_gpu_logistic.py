"""GPU: logistic regression -- Bernoulli(logits = X @ beta) on the GLM contractions (SIMT, tcgen05 3xTF32, tcgen05
3xFP16 with the Bernoulli-logit epilogue of K5) and the pointwise Bernoulli density, against float64; cross-class
agreement; posterior checks of NUTS / HMC / Metropolis against float64 quadrature and importance sampling."""
import math

import numpy as np
import pytest
import torch

import mlx_mcmc_b200 as B
import mlx_mcmc_b200.core as mx
from mlx_mcmc_b200 import _cabi, workloads as W
from mlx_mcmc_b200.engine import ChainState, compile_model, launch_nuts

pytestmark = pytest.mark.gpu

PRIOR = 10.0


def _model(path, n, d, seed):
    fn, init, meta = W.logistic_regression(B.ns, n, d, seed=seed)
    return compile_model(fn, init, cache=False, glm_path=path), meta


def _float64(X64, y64, theta):
    """log p and gradient of the logistic model in float64 on the device (torch as a calculator)"""
    b = theta.double()
    d = X64.shape[1]
    eta = b @ X64.T
    lp = ((y64[None, :] * eta - torch.nn.functional.softplus(eta)).sum(1)
          - 0.5 * (b ** 2).sum(1) / PRIOR ** 2 - d * (0.5 * math.log(2 * math.pi) + math.log(PRIOR)))
    g = (y64[None, :] - torch.sigmoid(eta)) @ X64 - b / PRIOR ** 2
    return lp, g


def _errors(lp, g, lp64, g64, n):
    """relative log p per chain, norm-wise gradient over the batch, and gradient per chain.  A chain's gradient is
    measured against its own largest component, or against sqrt(n) / 2 if that is smaller: one posterior standard
    deviation from the mode the gradient is of that order (Fisher information ~ n / 4 per unit-variance column), and a
    chain that happens to sit closer to the mode has a gradient near zero that no floating-point sum over n terms
    resolves to a relative 1e-5."""
    e_lp = float(((lp.double() - lp64).abs() / lp64.abs()).max())
    e_g = float((g.double() - g64).abs().max() / g64.abs().max())
    e_chain = float(((g.double() - g64).abs().amax(1) / g64.abs().amax(1).clamp(min=0.5 * math.sqrt(n))).max())
    return e_lp, e_g, e_chain


# ------------------------------------------------------------------------------------------------ 1. GLM vs float64
@pytest.mark.parametrize("path", ["simt", "tc", "tc16"])
@pytest.mark.parametrize("n,d,c", [(257, 65, 1), (255, 63, 129), (513, 1, 300), (4097, 129, 257),
                                   (30000, 256, 512), (50000, 500, 1024), (26000, 200, 300)])
def test_glm_logistic_ragged_shapes_vs_float64(cuda, n, d, c, path):
    model, meta = _model(path, n, d, seed=n * 7 + d)
    assert model.model_class == 1 and model.glm_path == path
    gen = torch.Generator(device="cuda").manual_seed(2)
    beta = torch.from_numpy(meta.beta_true).cuda()
    theta = (beta[None, :] + 0.1 * torch.randn(c, d, device="cuda", generator=gen)).contiguous()
    lp, g = model.logp_grad(theta)
    lp64, g64 = _float64(torch.from_numpy(meta.X).cuda().double(), torch.from_numpy(meta.y).cuda().double(), theta)
    e = _errors(lp, g, lp64, g64, n)
    print(f"{path} n={n} d={d} c={c}: logp {e[0]:.2e} grad {e[1]:.2e} per-chain {e[2]:.2e}")
    # the fp32 SIMT path sums the n products of each gradient component in one sequential fp32 chain (K6 of the SIMT
    # path, shared with the Normal kind): at n >= 30000 its per-chain error reaches 1e-5 (measured 1.02e-5 at 50000)
    assert e[0] < 1e-5 and e[1] < 1e-5 and e[2] < (2e-5 if path == "simt" and n >= 30000 else 1e-5), e


@pytest.fixture(scope="module", params=["tc16", "tc"])
def c4(cuda, request):
    """the C4 shape in both tensor-core encodings (the SIMT path's single fp32 chain over 100,000 products per gradient
    component is not held to 1e-5 at this size, for either likelihood kind)"""
    model, meta = _model(request.param, 100000, 1000, seed=0)
    assert model.glm_path == request.param
    return model, meta, torch.from_numpy(meta.X).cuda().double(), torch.from_numpy(meta.y).cuda().double()


@pytest.mark.parametrize("where,spread", [("mode", 0.003), ("zero", 0.0), ("far", 3.0)])
def test_glm_logistic_c4_vs_float64(c4, where, spread):
    model, meta, X64, y64 = c4
    gen = torch.Generator(device="cuda").manual_seed(7)
    if where == "mode":      # a few Newton steps in float64 from beta*: the posterior mode
        b = torch.from_numpy(meta.beta_true).cuda().double()
        for _ in range(8):
            p = torch.sigmoid(X64 @ b)
            H = (X64 * (p * (1 - p))[:, None]).T @ X64 + torch.eye(1000, device="cuda", dtype=torch.float64) / PRIOR ** 2
            b = b + torch.linalg.solve(H, X64.T @ (y64 - p) - b / PRIOR ** 2)
        base = b.float()[None, :]
    else:
        base = torch.from_numpy(meta.beta_true).cuda()[None, :] if where == "far" else torch.zeros(1, 1000, device="cuda")
    theta = (base + spread * torch.randn(256, 1000, device="cuda", generator=gen)).contiguous()
    lp, g = model.logp_grad(theta)
    e = _errors(lp, g, *_float64(X64, y64, theta), 100000)
    print(f"C4 logistic {model.glm_path} {where} spread={spread}: logp {e[0]:.2e} grad {e[1]:.2e} per-chain {e[2]:.2e}")
    assert max(e) < 1e-5, e


# ------------------------------------------------------------------------------------------------ 2. repeats, labels
@pytest.mark.parametrize("path", ["simt", "tc", "tc16"])
def test_glm_logistic_repeatable_and_value_only(cuda, path):
    model, meta = _model(path, 3000, 40, seed=3)
    theta = torch.from_numpy(np.tile(meta.beta_true, (300, 1)).astype(np.float32)).cuda()
    a, ga = model.logp_grad(theta)
    b, _ = model.logp_grad(theta, want_grad=False)
    c, gc = model.logp_grad(theta)
    assert torch.equal(a, b) and torch.equal(a, c) and torch.equal(ga, gc)
    assert torch.equal(a, a[0].expand_as(a)) and torch.equal(ga, ga[0].expand_as(ga))


def test_glm_labels_outside_0_1_fail_model_creation(cuda):
    X = np.random.default_rng(0).standard_normal((500, 8)).astype(np.float32)
    y = (np.arange(500) % 2).astype(np.float32)
    y[123] = 0.5
    Xa, ya = mx.array(X), mx.array(y)

    def fn(p):
        return mx.sum(B.Normal(0, 10).log_prob(p["beta"])) + mx.sum(B.Bernoulli(logits=Xa @ p["beta"]).log_prob(ya))
    with pytest.raises(_cabi.B2MError, match="labels must all be 0 or 1"):
        compile_model(fn, {"beta": np.zeros(8, dtype=np.float32)}, cache=False)


# ------------------------------------------------------------------------------------------------ 3. pointwise Bernoulli
_Y = np.array([1, 0, 0, 1, 1, 1, 0, 1, 0, 1, 1], dtype=np.float32)


def _pointwise_fn(y):
    def fn(p):
        return (B.Normal(0, 2).log_prob(p["a"]) + B.Normal(0, 2).log_prob(p["b"])
                + mx.sum(B.Bernoulli(logits=p["a"]).log_prob(y)) + B.Bernoulli(logits=p["b"]).log_prob(0.0))
    return fn, {"a": 0.3, "b": -0.2}


def _pointwise64(y, th):
    a, b = th[:, 0], th[:, 1]
    ok = (y == 0) | (y == 1)
    yk = y[ok].astype(np.float64)
    prior = lambda v: -0.5 * math.log(2 * math.pi) - math.log(2.0) - v ** 2 / 8.0   # noqa: E731
    lp = prior(a) + prior(b) + (yk[None, :] * a[:, None] - np.logaddexp(0, a)[:, None]).sum(1) - np.logaddexp(0, b)
    if not ok.all():
        lp = np.full_like(lp, -np.inf)
    ga = -a / 4.0 + (yk[None, :] - 1 / (1 + np.exp(-a[:, None]))).sum(1)
    gb = -b / 4.0 - 1 / (1 + np.exp(-b))
    return lp, np.stack([ga, gb], 1)


def test_pointwise_bernoulli_vs_float64_and_paths_bit_identical(cuda):
    from mlx_mcmc_b200 import jit as J
    fn, init = _pointwise_fn(_Y)
    fast = compile_model(fn, init, cache=False)
    assert fast.model_class == 0
    slow = compile_model(fn, init, cache=False, pointwise_path="general")
    spec = compile_model(fn, init, cache=False)
    assert J.specialize(spec, True) and spec.lib.b2m_model_has_module(spec.handle) == 1
    rng = np.random.default_rng(5)
    th = np.concatenate([rng.uniform(-4, 4, (253, 2)), [[40.0, -40.0], [-90.0, 90.0], [0.0, 0.0], [100.0, -100.0]]])
    theta = torch.from_numpy(th.astype(np.float32)).cuda()
    lp64, g64 = _pointwise64(_Y, th.astype(np.float32).astype(np.float64))
    for lanes in (1, 4):
        a, ga = fast.logp_grad(theta, lanes=lanes)
        assert np.max(np.abs(a.cpu().numpy() - lp64) / np.maximum(1.0, np.abs(lp64))) < 1e-5
        assert np.max(np.abs(ga.cpu().numpy() - g64) / np.maximum(1.0, np.abs(g64))) < 1e-5
        for other in (slow, spec):
            b, gb = other.logp_grad(theta, lanes=lanes)
            assert torch.equal(a, b) and torch.equal(ga, gb)
    kw = dict(num_samples=30, num_warmup=30, num_chains=96, key=mx.random.key(3), compat="correct")
    na, _ = B.nuts(fn, init, model=fast, **kw)
    for other in (slow, spec):
        nb, _ = B.nuts(fn, init, model=other, **kw)
        assert all(np.array_equal(na[k], nb[k]) for k in na)


def test_pointwise_bernoulli_label_outside_support_is_minus_inf_with_zero_gradient(cuda):
    y = _Y.copy()
    y[4] = 0.5
    fn, init = _pointwise_fn(y)
    model = compile_model(fn, init, cache=False)
    th = np.array([[0.3, -0.2], [2.0, 1.0]], dtype=np.float32)
    lp, g = model.logp_grad(torch.from_numpy(th).cuda())
    assert torch.all(lp == -math.inf)
    _, g64 = _pointwise64(y, th.astype(np.float64))        # the element outside the support adds nothing to the gradient
    np.testing.assert_allclose(g.cpu().numpy(), g64, rtol=1e-5, atol=1e-5)


# ------------------------------------------------------------------------------------------------ 4. cross-class
def _cross_models(n=300, seed=4):
    X, y, _ = W.data_logistic(n, 3, seed)
    Xa, ya = mx.array(X), mx.array(y)
    cols = [mx.array(np.ascontiguousarray(X[:, j])) for j in range(3)]

    def glm(p):
        return mx.sum(B.Normal(0, PRIOR).log_prob(p["beta"])) + mx.sum(B.Bernoulli(logits=Xa @ p["beta"]).log_prob(ya))

    def pw(p):
        prior = B.Normal(0, PRIOR).log_prob(p["b0"]) + B.Normal(0, PRIOR).log_prob(p["b1"]) + B.Normal(0, PRIOR).log_prob(p["b2"])
        return prior + mx.sum(B.Bernoulli(logits=p["b0"] * cols[0] + p["b1"] * cols[1] + p["b2"] * cols[2]).log_prob(ya))

    mg = compile_model(glm, {"beta": np.zeros(3, dtype=np.float32)}, cache=False)
    mp = compile_model(pw, {"b0": 0.0, "b1": 0.0, "b2": 0.0}, cache=False)
    assert mg.model_class == 1 and mp.model_class == 0
    return mg, mp


def test_cross_class_logp_grad_and_first_nuts_transition(cuda):
    mg, mp = _cross_models()
    gen = torch.Generator(device="cuda").manual_seed(9)
    C = 512
    theta = (0.5 * torch.randn(C, 3, device="cuda", generator=gen)).contiguous()
    lg, gg = mg.logp_grad(theta)
    lq, gq = mp.logp_grad(theta)
    assert float(((lg - lq).abs() / lq.abs()).max()) < 1e-5
    assert float((gg - gq).abs().max() / gq.abs().max()) < 1e-5
    depths = []
    for m in (mg, mp):
        st = ChainState(m, theta.clone(), 0.05)
        dep = torch.empty((1, C), dtype=torch.int32, device="cuda")
        launch_nuts(st, 1, 10, _cabi.ADAPT_NONE, _cabi.COMPAT_CORRECT, 0.65, 1234, 0, depths=dep)
        depths.append(dep[0].cpu().numpy())
    same = float(np.mean(depths[0] == depths[1]))
    print(f"first NUTS transition: equal depths for {100 * same:.1f} % of {C} chains, mean depth {depths[0].mean():.2f}")
    assert same >= 0.95


# ------------------------------------------------------------------------------------------------ 5. posterior
def _chain_mean_and_mcse(x):
    """x [C, S, D] draws of independent chains -> mean [D], MCSE [D] from the spread of the per-chain means"""
    cm = x.reshape(x.shape[0], x.shape[1], -1).mean(1)
    return cm.mean(0), cm.std(0, ddof=1) / math.sqrt(cm.shape[0])


def test_posterior_d2_against_grid_quadrature(cuda):
    n, C = 400, 256
    fn, init, meta = W.logistic_regression(B.ns, n, 2, seed=11)
    X, y = meta.X.astype(np.float64), meta.y.astype(np.float64)
    # float64 grid quadrature around the mode (+-10 posterior sd)
    b = np.zeros(2)
    for _ in range(30):
        p = 1 / (1 + np.exp(-X @ b))
        H = (X * (p * (1 - p))[:, None]).T @ X + np.eye(2) / PRIOR ** 2
        b = b + np.linalg.solve(H, X.T @ (y - p) - b / PRIOR ** 2)
    sd = np.sqrt(np.diag(np.linalg.inv(H)))
    g0, g1 = (np.linspace(b[k] - 10 * sd[k], b[k] + 10 * sd[k], 401) for k in (0, 1))
    G = np.stack(np.meshgrid(g0, g1, indexing="ij"), -1).reshape(-1, 2)
    eta = G @ X.T
    lp = (y[None, :] * eta - np.logaddexp(0, eta)).sum(1) - 0.5 * (G ** 2).sum(1) / PRIOR ** 2
    w = np.exp(lp - lp.max())
    truth = (w[:, None] * G).sum(0) / w.sum()

    X32, cols = meta.X, [mx.array(np.ascontiguousarray(meta.X[:, j])) for j in range(2)]
    ya = mx.array(meta.y)

    def pw(p):
        return (B.Normal(0, PRIOR).log_prob(p["b0"]) + B.Normal(0, PRIOR).log_prob(p["b1"])
                + mx.sum(B.Bernoulli(logits=p["b0"] * cols[0] + p["b1"] * cols[1]).log_prob(ya)))

    runs = {}
    kw = dict(num_chains=C, key=mx.random.key(21))
    s, _ = B.nuts(fn, init, num_samples=200, num_warmup=200, compat="correct", **kw)
    runs["glm nuts"] = np.asarray(s["beta"])
    s, _ = B.nuts(fn, init, num_samples=200, num_warmup=200, compat="correct", schedule="sync", **kw)
    runs["glm nuts sync"] = np.asarray(s["beta"])
    s, _ = B.nuts(pw, {"b0": 0.0, "b1": 0.0}, num_samples=200, num_warmup=200, compat="correct", **kw)
    runs["pointwise nuts"] = np.stack([np.asarray(s["b0"]), np.asarray(s["b1"])], -1)
    s, _ = B.hmc(fn, init, num_samples=200, num_warmup=200, step_size=0.05, num_leapfrog_steps=8, **kw)
    runs["glm hmc"] = np.asarray(s["beta"])
    s, _ = B.metropolis_hastings(fn, init, num_samples=3000, proposal_scale=0.08, num_chains=C)
    runs["glm metropolis"] = np.asarray(s["beta"])[:, 1000:]
    for name, x in runs.items():
        assert x.shape[0] == C and x.shape[-1] == 2, (name, x.shape)
        m, se = _chain_mean_and_mcse(x)
        z = np.abs(m - truth) / se
        print(f"{name}: mean {m} truth {truth} |z| {z}")
        assert np.all(np.isfinite(x)) and np.all(z < 4.0), (name, m, truth, se)


def test_posterior_d20_against_laplace_importance_sampling(cuda):
    n, d, C = 20000, 20, 512
    fn, init, meta = W.logistic_regression(B.ns, n, d, seed=12)
    X64, y64 = torch.from_numpy(meta.X).cuda().double(), torch.from_numpy(meta.y).cuda().double()
    b = torch.zeros(d, device="cuda", dtype=torch.float64)
    I = torch.eye(d, device="cuda", dtype=torch.float64)
    for _ in range(30):
        p = torch.sigmoid(X64 @ b)
        H = (X64 * (p * (1 - p))[:, None]).T @ X64 + I / PRIOR ** 2
        b = b + torch.linalg.solve(H, X64.T @ (y64 - p) - b / PRIOR ** 2)
    L = torch.linalg.cholesky(torch.linalg.inv(H))
    gen = torch.Generator(device="cuda").manual_seed(5)
    M = 40000
    z = torch.randn(M, d, device="cuda", dtype=torch.float64, generator=gen)
    draws = b[None, :] + z @ L.T
    logq = -0.5 * (z ** 2).sum(1)
    logp = torch.zeros(M, device="cuda", dtype=torch.float64)
    for i in range(0, M, 4000):
        eta = draws[i:i + 4000] @ X64.T
        logp[i:i + 4000] = (y64[None, :] * eta - torch.nn.functional.softplus(eta)).sum(1)
    logp -= 0.5 * (draws ** 2).sum(1) / PRIOR ** 2
    lw = logp - logq
    w = torch.exp(lw - lw.max())
    w = w / w.sum()
    ess_w = float(1.0 / (w ** 2).sum())
    truth = (w[:, None] * draws).sum(0)
    se_is = torch.sqrt((w[:, None] ** 2 * (draws - truth[None, :]) ** 2).sum(0)).cpu().numpy()
    s, _ = B.nuts(fn, init, num_samples=150, num_warmup=150, num_chains=C, compat="correct",
                  step_size_adaptation="pooled", key=mx.random.key(8))
    x = np.asarray(s["beta"])
    m, se = _chain_mean_and_mcse(x)
    zs = np.abs(m - truth.cpu().numpy()) / np.sqrt(se ** 2 + se_is ** 2)
    print(f"D=20 N=20000: importance-weight ESS {ess_w:.0f} of {M}; max |z| {zs.max():.2f}")
    assert ess_w > 0.3 * M and np.all(np.isfinite(x)) and zs.max() < 4.5, (ess_w, zs)


# ------------------------------------------------------------------------------------------------ 6. C4 through MCMC.run
def test_c4_logistic_through_mcmc_run(cuda):
    fn, init, meta = W.logistic_regression(B.ns, 100000, 1000, seed=0)
    m = B.MCMC(fn)
    m.run(init, method="nuts", num_samples=40, num_warmup=150, adapt_mass_matrix=True, step_size=1e-3, num_chains=4096,
          compat="correct", step_size_adaptation="pooled", return_torch=True, return_info=True, verbose=False, random_seed=1)
    assert bool(torch.isfinite(m.samples["beta"]).all())
    diag = m.diagnostics(ess=False)["beta"]
    print(f"C4 logistic: max R-hat {np.nanmax(diag['rhat']):.4f}, mean depth {m.info.depths.mean():.2f}, "
          f"step size {float(m.info.step_size[0]):.3g}")
    assert np.all(np.isfinite(diag["rhat"])) and diag["rhat"].max() < 1.05
