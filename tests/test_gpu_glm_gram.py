"""GPU: the Gram form of the GLM Normal likelihood (one [C, D] x [D, D] contraction against X^T X precomputed in float64)
against float64 and against the streaming form (K5 + K6), in both tensor-core encodings."""
import math

import numpy as np
import pytest
import torch

import mlx_mcmc_b200 as B
from mlx_mcmc_b200 import _cabi, workloads as W
from mlx_mcmc_b200.engine import ChainState, compile_model, launch_nuts

pytestmark = pytest.mark.gpu


def _model(path, form, n, d, seed):
    fn, init, meta = W.regression(B.ns, n, d, seed=seed)
    m = compile_model(fn, init, cache=False, glm_path=path, glm_form=form)
    assert m.glm_path == path and m.glm_form == form
    return m, meta


def _float64(meta, theta):
    X, y, b = meta.X.astype(np.float64), meta.y.astype(np.float64), theta.astype(np.float64)
    n, d = X.shape
    r = y[None, :] - b @ X.T
    lp = (-0.5 * (r ** 2).sum(1) - n * 0.5 * math.log(2 * math.pi)
          - 0.5 * (b ** 2).sum(1) / 100.0 - d * (0.5 * math.log(2 * math.pi) + math.log(10.0)))
    return lp, r @ X - b / 100.0


def _errs(lp, g, lp64, g64):
    lp, g = lp.cpu().numpy().astype(np.float64), g.cpu().numpy().astype(np.float64)
    return np.max(np.abs(lp - lp64) / np.abs(lp64)), np.max(np.abs(g - g64)) / np.max(np.abs(g64))


SHAPES = [(200, 5, 7), (1000, 100, 130), (5000, 96, 300), (3000, 300, 1024), (40000, 64, 256),
          (257, 65, 1), (255, 63, 129), (513, 1, 300), (4097, 129, 257), (30000, 256, 512), (50000, 500, 1024)]


@pytest.mark.parametrize("path", ["tc", "tc16"])
@pytest.mark.parametrize("n,d,c", SHAPES)
def test_gram_and_stream_vs_float64(cuda, n, d, c, path):
    gram, meta = _model(path, "gram", n, d, seed=n + d)
    stream, _ = _model(path, "stream", n, d, seed=n + d)
    rng = np.random.default_rng(1)
    theta = (meta.beta_true[None, :] + 0.2 * rng.standard_normal((c, d))).astype(np.float32)
    t = torch.from_numpy(theta).cuda()
    lp_g, g_g = gram.logp_grad(t)
    lp_s, g_s = stream.logp_grad(t)
    lp64, g64 = _float64(meta, theta)
    e_lp_g, e_g_g = _errs(lp_g, g_g, lp64, g64)
    e_lp_s, e_g_s = _errs(lp_s, g_s, lp64, g64)
    print(f"{path} n={n} d={d} c={c}: gram lp {e_lp_g:.2e} g {e_g_g:.2e} | stream lp {e_lp_s:.2e} g {e_g_s:.2e}")
    assert e_lp_g < 1e-5 and e_lp_s < 1e-5
    assert e_g_g < 3e-6 and e_g_s < 1e-5
    # the two forms against each other: the same function summed in a different order
    gs = g_s.double()
    assert float((g_g.double() - gs).abs().max() / gs.abs().max()) < 1e-5


@pytest.mark.parametrize("path", ["tc", "tc16"])
def test_gram_value_only_repeats_and_identical_rows(cuda, path):
    model, meta = _model(path, "gram", 2000, 40, seed=3)
    theta = torch.from_numpy(np.tile(meta.beta_true, (64, 1)).astype(np.float32)).cuda()
    a, ga = model.logp_grad(theta)
    b, _ = model.logp_grad(theta, want_grad=False)
    c, gc = model.logp_grad(theta)
    assert torch.equal(a, b) and torch.equal(a, c) and torch.equal(ga, gc)
    assert torch.equal(a, a[0].expand_as(a)) and torch.equal(ga, ga[0:1].expand_as(ga))
    # a spread batch: value-only still runs the contraction and gets the same log p bit for bit
    rng = np.random.default_rng(4)
    th2 = torch.from_numpy((meta.beta_true[None, :] + 0.1 * rng.standard_normal((300, 40))).astype(np.float32)).cuda()
    l1, _ = model.logp_grad(th2)
    l2, _ = model.logp_grad(th2, want_grad=False)
    assert torch.equal(l1, l2)


def _sigma_model(X, y, form, path):
    mx, Normal, HalfNormal = B.ns.mx, B.ns.Normal, B.ns.HalfNormal
    Xa, ya = mx.array(X), mx.array(y)

    def log_prob(params):
        beta, sigma = params["beta"], params["sigma"]
        return (mx.sum(Normal(0, 10.0).log_prob(beta)) + HalfNormal(5.0).log_prob(sigma)
                + 0.5 * mx.sum(Normal(Xa @ beta + 2.5, sigma).log_prob(ya)))
    init = {"beta": np.zeros(X.shape[1], dtype=np.float32), "sigma": np.float32(1.0)}
    m = compile_model(log_prob, init, cache=False, glm_path=path, glm_form=form, transforms="auto")
    assert m.glm_form == form
    return m


@pytest.mark.parametrize("path", ["tc", "tc16"])
def test_gram_sigma_parameter_transforms_location_and_weight(cuda, path):
    """sigma as a parameter sampled in log coordinates, a constant location 2.5 and a likelihood weight 0.5: the Gram
    form gives the streaming form's log p and gradient (sigma's gradient included), and a value-only call agrees"""
    rng = np.random.default_rng(5)
    n, d, c = 8000, 70, 200
    X = rng.standard_normal((n, d)).astype(np.float32)
    beta = rng.standard_normal(d).astype(np.float32)
    y = (X.astype(np.float64) @ beta + 2.5 + 1.3 * rng.standard_normal(n)).astype(np.float32)
    gram, stream = _sigma_model(X, y, "gram", path), _sigma_model(X, y, "stream", path)
    theta = 0.02 * rng.standard_normal((c, d + 1))
    theta[:, :d] += beta                           # layout: beta then sigma (the order of the parameter dict)
    theta[:, d] = math.log(1.3) + 0.05 * rng.standard_normal(c)
    t = torch.from_numpy(theta.astype(np.float32)).cuda()
    lp_g, g_g = gram.logp_grad(t)
    lp_s, g_s = stream.logp_grad(t)
    e_lp = float(((lp_g.double() - lp_s.double()).abs() / lp_s.double().abs()).max())
    e_g = float(((g_g.double() - g_s.double()).abs() / g_s.double().abs().amax(0)).max())   # per coordinate
    print(f"{path} sigma model: lp {e_lp:.2e} grad {e_g:.2e}")
    assert e_lp < 1e-5 and e_g < 1e-5
    lv, _ = gram.logp_grad(t, want_grad=False)
    assert torch.equal(lv, lp_g)


def _custom_model(X, y, form):
    mx, Normal = B.ns.mx, B.ns.Normal
    Xa, ya = mx.array(X), mx.array(y)

    def log_prob(params):
        beta = params["beta"]
        return mx.sum(Normal(0, 10.0).log_prob(beta)) + mx.sum(Normal(Xa @ beta, 1.0).log_prob(ya))
    return compile_model(log_prob, {"beta": np.zeros(X.shape[1], dtype=np.float32)}, cache=False, glm_form=form)


def test_gram_column_scales_per_coefficient(cuda):
    """features on scales 1e-3 .. 1e3: each gradient component within 1e-5 of float64 against its own column's scale"""
    rng = np.random.default_rng(3)
    n, d, c = 6000, 48, 200
    colscale = 10.0 ** rng.uniform(-3, 3, d)
    X = (rng.standard_normal((n, d)) * colscale).astype(np.float32)
    beta = (rng.standard_normal(d) / colscale).astype(np.float32)
    y = (X.astype(np.float64) @ beta.astype(np.float64) + rng.standard_normal(n)).astype(np.float32)
    model = _custom_model(X, y, "gram")
    assert model.glm_path == "tc16" and model.glm_form == "gram"
    theta = (beta[None, :] * (1 + 0.01 * rng.standard_normal((c, d)))).astype(np.float32)
    lp, g = model.logp_grad(torch.from_numpy(theta).cuda())
    b = theta.astype(np.float64)
    r = y.astype(np.float64)[None, :] - b @ X.astype(np.float64).T
    g64 = r @ X.astype(np.float64) - b / 100.0
    lp64 = (-0.5 * (r ** 2).sum(1) - n * 0.5 * math.log(2 * math.pi) - 0.5 * (b ** 2).sum(1) / 100.0
            - d * (0.5 * math.log(2 * math.pi) + math.log(10.0)))
    assert np.max(np.abs(lp.cpu().numpy() - lp64) / np.abs(lp64)) < 1e-5
    err = np.max(np.abs(g.cpu().numpy() - g64), axis=0) / np.max(np.abs(g64), axis=0)
    print(f"column scales: worst coefficient {err.max():.2e}")
    assert err.max() < 1e-5


def test_auto_form_choice_and_refusals(cuda):
    fn, init, _ = W.regression(B.ns, 100000, 1000, seed=0)
    assert compile_model(fn, init, cache=False).glm_form == "gram"                       # C4
    fn, init, _ = W.regression(B.ns, 10000, 100, seed=0)
    assert compile_model(fn, init, cache=False).glm_form == "gram"                       # C3
    fn, init, _ = W.regression(B.ns, 100, 64, seed=0)
    assert compile_model(fn, init, cache=False).glm_form == "stream"                     # N < 2 Dp
    assert compile_model(fn, init, cache=False, glm_form="gram").glm_form == "gram"      # forced: allowed, slower
    assert compile_model(fn, init, cache=False, glm_path="simt").glm_form == "stream"    # the validation path
    with pytest.raises(RuntimeError, match="tensor-core"):
        compile_model(fn, init, cache=False, glm_path="simt", glm_form="gram")
    fl, il, _ = W.logistic_regression(B.ns, 5000, 20, seed=0)
    assert compile_model(fl, il, cache=False).glm_form == "stream"
    with pytest.raises(RuntimeError, match="Normal likelihood"):
        compile_model(fl, il, cache=False, glm_form="gram")


@pytest.fixture(scope="module")
def c4data(cuda):
    fn, init, meta = W.regression(B.ns, 100000, 1000, seed=0)
    X64 = torch.from_numpy(meta.X).cuda().double()
    y64 = torch.from_numpy(meta.y).cuda().double()
    return fn, init, meta, X64, y64


def _float64_gpu(X64, y64, theta):
    b = theta.double()
    n, d = X64.shape
    r = y64[None, :] - b @ X64.T
    lp = (-0.5 * (r ** 2).sum(1) - n * 0.5 * math.log(2 * math.pi)
          - 0.5 * (b ** 2).sum(1) / 100.0 - d * (0.5 * math.log(2 * math.pi) + math.log(10.0)))
    return lp, r @ X64 - b / 100.0


def test_c4_full_batch_streaming_form(c4data):
    """K5's Normal epilogue keeps full-size coverage now that auto picks the Gram form at C4: all 4096 chains of the
    streaming form within 1e-5 of float64, bit-repeatable"""
    fn, init, meta, X64, y64 = c4data
    model = compile_model(fn, init, cache=False, glm_form="stream")
    assert model.glm_form == "stream"
    gen = torch.Generator(device="cuda").manual_seed(13)
    theta = (torch.from_numpy(meta.beta_true).cuda()[None, :] + 0.003 * torch.randn(4096, 1000, device="cuda", generator=gen)).contiguous()
    lp, g = model.logp_grad(theta)
    lp2, g2 = model.logp_grad(theta)
    assert torch.equal(lp, lp2) and torch.equal(g, g2)
    e_lp = e_g = 0.0
    for i in range(0, 4096, 1024):
        lp64, g64 = _float64_gpu(X64, y64, theta[i:i + 1024])
        e_lp = max(e_lp, float(((lp[i:i + 1024].double() - lp64).abs() / lp64.abs()).max()))
        e_g = max(e_g, float(((g[i:i + 1024].double() - g64).abs().amax(1) / g64.abs().amax(1)).max()))
    print(f"C4 streaming, 4096 chains: logp {e_lp:.2e} per-chain grad {e_g:.2e}")
    assert e_lp < 1e-5 and e_g < 1e-5
    del model


def test_c4_nuts_first_transition_gram_vs_stream(c4data):
    """Both forms from identical states with identical draws: first-transition draws agree within 1e-2 posterior sd
    for >= 97 % of chains, with the same mean tree depth (the trajectories differ only by rounding).  The tail of the
    transition runs on compacted batches, so this also covers the Gram form on a compacted batch."""
    fn, init, meta, X64, y64 = c4data
    mean, cov = W.regression_posterior(meta)
    sd = torch.from_numpy(np.sqrt(np.diag(cov))).cuda()
    C, N = 4096, 100000
    gen = torch.Generator(device="cuda").manual_seed(21)
    theta0 = (torch.from_numpy(mean.astype(np.float32)).cuda()[None, :]
              + torch.randn(C, 1000, device="cuda", generator=gen) / N ** 0.5).contiguous()
    out = {}
    for form in ("gram", "stream"):
        model = compile_model(fn, init, cache=False, glm_form=form)
        st = ChainState(model, theta0.clone(), 0.002, 0)
        draws = torch.empty(1, C, 1000, device="cuda")
        depths = torch.empty(1, C, dtype=torch.int32, device="cuda")
        launch_nuts(st, 1, 10, _cabi.ADAPT_NONE, _cabi.COMPAT_CORRECT, 0.65, 77, 0, draws=draws, depths=depths)
        torch.cuda.synchronize()
        out[form] = (draws[0].double(), depths[0].double())
        del st, model
    dg, ds = out["gram"], out["stream"]
    close = ((dg[0] - ds[0]).abs() / sd[None, :]).amax(1) < 1e-2
    frac = float(close.double().mean())
    print(f"C4 NUTS first transition: {frac:.4f} of chains within 1e-2 sd; mean depth {float(dg[1].mean()):.3f} "
          f"vs {float(ds[1].mean()):.3f}")
    assert frac >= 0.97
    assert abs(float(dg[1].mean()) - float(ds[1].mean())) < 0.1
