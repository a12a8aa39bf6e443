"""GPU: the tcgen05 contractions (K5/K6) in both operand encodings -- 3xTF32 ("tc") and 3xFP16 with power-of-two
operand scaling ("tc16", the default when the data's dynamic range allows it) -- against float64 and against the
fp32 SIMT path."""
import math
import os

import numpy as np
import pytest
import torch

import mlx_mcmc_b200 as B
from mlx_mcmc_b200 import workloads as W
from mlx_mcmc_b200.engine import compile_model

pytestmark = pytest.mark.gpu


def _model(path, n, d, seed):
    fn, init, meta = W.regression(B.ns, n, d, seed=seed)
    return compile_model(fn, init, cache=False, glm_path=path), meta


def _float64(meta, theta):
    X, y, b = meta.X.astype(np.float64), meta.y.astype(np.float64), theta.astype(np.float64)
    n, d = X.shape
    r = y[None, :] - b @ X.T
    lp = (-0.5 * (r ** 2).sum(1) - n * 0.5 * math.log(2 * math.pi)
          - 0.5 * (b ** 2).sum(1) / 100.0 - d * (0.5 * math.log(2 * math.pi) + math.log(10.0)))
    return lp, r @ X - b / 100.0


@pytest.mark.parametrize("path", ["tc", "tc16"])
@pytest.mark.parametrize("n,d,c", [(200, 5, 7), (1000, 100, 130), (5000, 96, 300), (3000, 300, 1024), (40000, 64, 256)])
def test_tc_logp_grad_vs_float64_and_simt(cuda, n, d, c, path):
    tc, meta = _model(path, n, d, seed=n + d)
    assert tc.glm_path == path
    simt, _ = _model("simt", n, d, seed=n + d)
    rng = np.random.default_rng(1)
    theta = (meta.beta_true[None, :] + 0.2 * rng.standard_normal((c, d))).astype(np.float32)
    t = torch.from_numpy(theta).cuda()
    lp_tc, g_tc = tc.logp_grad(t)
    lp_s, g_s = simt.logp_grad(t)
    torch.cuda.synchronize()
    lp64, g64 = _float64(meta, theta)
    for lp, g, tol in ((lp_tc, g_tc, 1e-5), (lp_s, g_s, 1e-5)):
        assert np.max(np.abs(lp.cpu().numpy() - lp64) / np.abs(lp64)) < tol
        assert np.max(np.abs(g.cpu().numpy() - g64)) / np.max(np.abs(g64)) < tol
    # 3xTF32 with chunked promotion is as accurate as fp32 FMA tiles
    e_tc = np.max(np.abs(g_tc.cpu().numpy() - g64)) / np.max(np.abs(g64))
    e_s = np.max(np.abs(g_s.cpu().numpy() - g64)) / np.max(np.abs(g64))
    print(f"n={n} d={d} c={c}: grad err tc {e_tc:.2e} simt {e_s:.2e}; "
          f"logp err tc {np.max(np.abs(lp_tc.cpu().numpy() - lp64) / np.abs(lp64)):.2e}")
    assert e_tc < 3e-6


@pytest.mark.parametrize("path", ["tc", "tc16"])
def test_tc_value_only_and_repeatability(cuda, path):
    tc, meta = _model(path, 2000, 40, seed=3)
    theta = torch.from_numpy(np.tile(meta.beta_true, (64, 1)).astype(np.float32)).cuda()
    a, ga = tc.logp_grad(theta)
    b, _ = tc.logp_grad(theta, want_grad=False)
    c, gc = tc.logp_grad(theta)
    assert torch.equal(a, b) and torch.equal(a, c) and torch.equal(ga, gc)      # deterministic, bit for bit
    assert torch.equal(a, a[0].expand_as(a))                                     # identical rows -> identical results


# ------------------------------------------------------------------------------------------------ full size (C4)
@pytest.fixture(scope="module", params=["tc16", "tc"])
def c4(cuda, request):
    """BASELINE.json's Target configuration: 1000 coefficients x 100,000 observations (SURVEY.md 8d), both encodings."""
    model, meta = _model(request.param, 100000, 1000, seed=0)
    assert model.glm_path == request.param
    X64 = torch.from_numpy(meta.X).cuda().double()
    y64 = torch.from_numpy(meta.y).cuda().double()
    return model, meta, X64, y64


def _float64_gpu(X64, y64, theta):
    """float64 arbiter on the device (torch used as a calculator for the test, not by the product)"""
    b = theta.double()
    n, d = X64.shape
    r = y64[None, :] - b @ X64.T
    lp = (-0.5 * (r ** 2).sum(1) - n * 0.5 * math.log(2 * math.pi)
          - 0.5 * (b ** 2).sum(1) / 100.0 - d * (0.5 * math.log(2 * math.pi) + math.log(10.0)))
    return lp, r @ X64 - b / 100.0


@pytest.mark.parametrize("where,spread", [("mode", 0.003), ("mode", 0.2), ("zero", 0.0), ("far", 3.0)])
def test_c4_full_size_logp_grad_within_1e5_of_float64(c4, where, spread):
    """parity check 1 at full size: |lp - lp64| / |lp64| and max|g - g64| / max|g64| below 1e-5, per chain too"""
    model, meta, X64, y64 = c4
    gen = torch.Generator(device="cuda").manual_seed(7)
    base = torch.from_numpy(meta.beta_true).cuda()[None, :] if where != "zero" else torch.zeros(1, 1000, device="cuda")
    theta = (base + spread * torch.randn(256, 1000, device="cuda", generator=gen)).contiguous()
    lp, g = model.logp_grad(theta)
    lp64, g64 = _float64_gpu(X64, y64, theta)
    e_lp = float(((lp.double() - lp64).abs() / lp64.abs()).max())
    e_g = float((g.double() - g64).abs().max() / g64.abs().max())
    e_chain = float(((g.double() - g64).abs().amax(1) / g64.abs().amax(1)).max())
    print(f"C4 {where} spread={spread}: logp {e_lp:.2e} grad {e_g:.2e} per-chain {e_chain:.2e}")
    assert e_lp < 1e-5 and e_g < 1e-5 and e_chain < 1e-5


def test_c4_full_size_properties(c4):
    """size-independent properties at full size: the gradient is affine in beta with slope -(X'X + I/100); the
    value-only path, a repeat and a sub-batch give the same numbers."""
    model, meta, X64, y64 = c4
    gen = torch.Generator(device="cuda").manual_seed(11)
    b0 = torch.from_numpy(meta.beta_true).cuda()[None, :] + 0.003 * torch.randn(128, 1000, device="cuda", generator=gen)
    delta = 0.002 * torch.randn(128, 1000, device="cuda", generator=gen)
    both = torch.cat([b0, b0 + delta]).contiguous()            # one batch => one centring point for both halves
    lp, g = model.logp_grad(both)
    dg = (g[128:] - g[:128]).double()
    want = -((delta.double() @ X64.T) @ X64) - delta.double() / 100.0
    assert float((dg - want).abs().max() / want.abs().max()) < 2e-5
    lp2, _ = model.logp_grad(both, want_grad=False)
    lp3, g3 = model.logp_grad(both)
    assert torch.equal(lp, lp2) and torch.equal(lp, lp3) and torch.equal(g, g3)
    # energy-like check of the value: lp(b + d) - lp(b) = g(b).d - 0.5 d'(X'X + I/100)d  (exact for a quadratic)
    quad = (g[:128].double() * delta.double()).sum(1) + 0.5 * (want * delta.double()).sum(1)
    assert float(((lp[128:] - lp[:128]).double() - quad).abs().max()) < 2e-5 * float(lp.abs().max())


@pytest.mark.parametrize("path", ["tc", "tc16"])
@pytest.mark.parametrize("n,d,c", [(257, 65, 1), (255, 63, 129), (513, 1, 300), (4097, 129, 257),
                                   (30000, 256, 512), (50000, 500, 1024), (26000, 200, 300)])
def test_tc_ragged_shapes(cuda, n, d, c, path):
    """padding edges: N, D, C just off the 256 / 64 / 128 tile sizes, a single chain, a single coefficient; and mid-size
    shapes with several observation tiles per K split and several CTA-pair row tiles"""
    tc, meta = _model(path, n, d, seed=n * 7 + d)
    rng = np.random.default_rng(2)
    theta = (meta.beta_true[None, :] + 0.1 * rng.standard_normal((c, d))).astype(np.float32)
    lp, g = tc.logp_grad(torch.from_numpy(theta).cuda())
    lp64, g64 = _float64(meta, theta)
    assert np.max(np.abs(lp.cpu().numpy() - lp64) / np.abs(lp64)) < 1e-5
    assert np.max(np.abs(g.cpu().numpy() - g64)) / np.max(np.abs(g64)) < 1e-5


def _custom_model(X, y):
    mx, Normal = B.ns.mx, B.ns.Normal
    Xa, ya = mx.array(X), mx.array(y)

    def log_prob(params):
        beta = params["beta"]
        return mx.sum(Normal(0, 10.0).log_prob(beta)) + mx.sum(Normal(Xa @ beta, 1.0).log_prob(ya))
    return compile_model(log_prob, {"beta": np.zeros(X.shape[1], dtype=np.float32)}, cache=False)


def test_fp16_encoding_handles_column_scales_and_falls_back_on_outliers(cuda):
    """Features on wildly different scales (1e-3 .. 1e3) keep the fp16 encoding -- every column gets its own power-of-two
    scale -- and the 1e-5 gate; a column dominated by one outlier (max / rms > 4096) makes the model fall back to the
    tf32 encoding at build time."""
    rng = np.random.default_rng(3)
    n, d, c = 6000, 48, 200
    colscale = 10.0 ** rng.uniform(-3, 3, d)
    X = (rng.standard_normal((n, d)) * colscale).astype(np.float32)
    beta = (rng.standard_normal(d) / colscale).astype(np.float32)
    y = (X.astype(np.float64) @ beta.astype(np.float64) + rng.standard_normal(n)).astype(np.float32)
    model = _custom_model(X, y)
    assert model.glm_path == "tc16"
    theta = (beta[None, :] * (1 + 0.01 * rng.standard_normal((c, d)))).astype(np.float32)
    lp, g = model.logp_grad(torch.from_numpy(theta).cuda())
    b = theta.astype(np.float64)
    r = y.astype(np.float64)[None, :] - b @ X.astype(np.float64).T
    g64 = r @ X.astype(np.float64) - b / 100.0
    lp64 = (-0.5 * (r ** 2).sum(1) - n * 0.5 * math.log(2 * math.pi) - 0.5 * (b ** 2).sum(1) / 100.0
            - d * (0.5 * math.log(2 * math.pi) + math.log(10.0)))
    assert np.max(np.abs(lp.cpu().numpy() - lp64) / np.abs(lp64)) < 1e-5
    # per coefficient: each gradient component against the scale of ITS column (a norm-wise test over all columns
    # would only see the largest-scale feature)
    err = np.max(np.abs(g.cpu().numpy() - g64), axis=0) / np.max(np.abs(g64), axis=0)
    assert err.max() < 1e-5, err.max()
    X2 = X.copy()
    X2[17, 5] = 3e5 * np.abs(X2[:, 5]).mean()              # one wild entry
    wide = _custom_model(X2, y)
    assert wide.glm_path == "tc"
    lp2, g2 = wide.logp_grad(torch.from_numpy(theta).cuda())
    assert torch.isfinite(lp2).all() and torch.isfinite(g2).all()


def test_c4_full_batch_within_1e5_of_float64(c4):
    """All 4096 chains of BASELINE.json's Target configuration (residual operand 1.6 GB): repeatable bit for bit and
    within 1e-5 of float64 on the device."""
    model, meta, X64, y64 = c4
    gen = torch.Generator(device="cuda").manual_seed(13)
    base = torch.from_numpy(meta.beta_true).cuda()[None, :]
    theta = (base + 0.003 * torch.randn(4096, 1000, device="cuda", generator=gen)).contiguous()
    lp, g = model.logp_grad(theta)
    lp2, g2 = model.logp_grad(theta)
    assert torch.equal(lp, lp2) and torch.equal(g, g2)
    e_lp = e_g = e_chain = 0.0
    for i in range(0, 4096, 1024):                      # float64 arbiter in four slices (3.3 GB of residuals each)
        lp64, g64 = _float64_gpu(X64, y64, theta[i:i + 1024])
        e_lp = max(e_lp, float(((lp[i:i + 1024].double() - lp64).abs() / lp64.abs()).max()))
        e_g = max(e_g, float((g[i:i + 1024].double() - g64).abs().max() / g64.abs().max()))
        e_chain = max(e_chain, float(((g[i:i + 1024].double() - g64).abs().amax(1) / g64.abs().amax(1)).max()))
    print(f"C4 4096 chains ({model.glm_path}): logp {e_lp:.2e} grad {e_g:.2e} per-chain {e_chain:.2e}")
    assert e_lp < 1e-5 and e_g < 1e-5 and e_chain < 1e-5
