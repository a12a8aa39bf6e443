"""GLM class: every non-likelihood term (hierarchical and affine priors, extra observed terms, every prior density,
Bernoulli side terms, constants, fractional and negative weights), every parameter layout and constraint transforms,
checked coordinate by coordinate against a float64 evaluation of the traced term table.

The bound of coordinate j is 1e-5 * max(|g64_j|, S_j), S_j = sum over terms, slots and elements of |w df/dop_n| *
|dop_n/dtheta_j|: the sum of the absolute contributions the kernels add into g_j.  |df/dop_n| is taken as the sum of the
absolute summands of the partial as the device evaluates it: the Beta partial (a-1)/x - (b-1)/(1-x) cancels at the mode
and carries the float32 rounding of both parts (measured 1.8e-5 of |df/dx| on every path when only the partial itself
was counted).  A coordinate whose contributions are dropped has a ratio near 1; a norm-wise check over the batch would not see it, because the likelihood gradient of beta
is of order sqrt(N) or larger.  The float64 evaluator itself is checked against the oracle's float64 autograd on the
CPU (no gpu mark)."""
import math

import numpy as np
import pytest
import torch

import mlx_mcmc_b200 as B
from mlx_mcmc_b200 import _cabi, tracer as T

TOL = 1e-5
_POS = ("tau", "s", "r", "g", "sigma")   # names of positive scalars (HalfNormal / Exponential / Gamma values)


# ----------------------------------------------------------------------------- float64 reference
def _tf64(u, codes):
    """theta = T(u), log-Jacobian [C], d theta / du and d logjac / du (float64)"""
    codes = torch.as_tensor(np.asarray(codes), device=u.device)
    log, logit = codes == _cabi.TF_LOG, codes == _cabi.TF_LOGIT
    sg = torch.sigmoid(u)
    theta = torch.where(log, u.exp(), torch.where(logit, sg, u))
    lj = torch.where(log, u, torch.where(logit, torch.nn.functional.logsigmoid(u) + torch.nn.functional.logsigmoid(-u),
                                         torch.zeros_like(u))).sum(1)
    jac = torch.where(log, theta, torch.where(logit, sg * (1 - sg), torch.ones_like(u)))
    dlj = torch.where(log, torch.ones_like(u), torch.where(logit, 1 - 2 * sg, torch.zeros_like(u)))
    return theta, lj, jac, dlj


def _density(t, x, p0, p1):
    """elementwise float64 log density of term t (broadcast [C, n])"""
    ninf = torch.tensor(-math.inf, dtype=torch.float64, device=x.device)
    if t.dist == T.NORMAL:
        return -0.5 * math.log(2 * math.pi) - torch.log(p1) - 0.5 * ((x - p0) / p1) ** 2
    if t.dist == T.HALFNORMAL:
        return torch.where(x >= 0, math.log(2) - 0.5 * math.log(2 * math.pi) - torch.log(p0) - 0.5 * (x / p0) ** 2, ninf)
    if t.dist == T.EXPONENTIAL:
        return torch.where(x >= 0, torch.log(p0) - p0 * x, ninf)
    if t.dist == T.GAMMA:
        a = t.k[0]
        return torch.where(x > 0, a * torch.log(p0) - math.lgamma(a) + (a - 1) * torch.log(x) - p0 * x, ninf)
    if t.dist == T.BETA:
        a, b = t.k[0], t.k[1]
        lb = math.lgamma(a) + math.lgamma(b) - math.lgamma(a + b)
        return torch.where((x > 0) & (x < 1), (a - 1) * torch.log(x) + (b - 1) * torch.log1p(-x) - lb, ninf)
    if t.dist == T.BERNOULLI:
        return x * p0 - torch.nn.functional.softplus(p0)
    if t.dist == T.CONSTANT:
        return torch.full_like(x + p0 + p1, t.k[0])
    raise AssertionError(t.dist)


def _summands(t, x, p0, p1):
    """per slot, the sum of the absolute values of the summands of d f / d slot as the device evaluates it
    (model.cuh dist_eval): e.g. d/dx of Beta is (a - 1) / x - (b - 1) / (1 - x), two terms that cancel at the mode, so
    the float32 partial carries the rounding of both.  None: the slot is not differentiated"""
    if t.dist == T.NORMAL:
        z = (x - p0).abs()
        return z / p1 ** 2, z / p1 ** 2, z ** 2 / p1.abs() ** 3 + 1 / p1.abs()
    if t.dist == T.HALFNORMAL:
        return x.abs() / p0 ** 2, x ** 2 / p0.abs() ** 3 + 1 / p0.abs(), None
    if t.dist == T.EXPONENTIAL:
        return p0.abs(), 1 / p0.abs() + x.abs(), None
    if t.dist == T.GAMMA:
        return abs(t.k[0] - 1) / x.abs() + p0.abs(), t.k[0] / p0.abs() + x.abs(), None
    if t.dist == T.BETA:
        return abs(t.k[0] - 1) / x.abs() + abs(t.k[1] - 1) / (1 - x).abs(), None, None
    if t.dist == T.BERNOULLI:
        return None, (x - torch.sigmoid(p0)).abs(), None
    return None, None, None


def eval64(tm, u, codes=None):
    """float64 log p [C], gradient [C, D] (with respect to u through theta = T(u), log-Jacobian included), the
    per-coordinate sums S [C, D] of absolute gradient contributions and the per-chain sums L [C] of |w f_n|, of traced
    model `tm` at u [C, D].  The contributions to S are the summands of the element partials (_summands); each is
    checked to bound the autograd partial of its element."""
    dev = u.device
    u = u.detach().double().clone().requires_grad_(True)
    C, D = u.shape
    if codes is not None and np.any(np.asarray(codes) != 0):
        theta, lj, jac, dlj = _tf64(u, codes)
    else:
        theta, lj, jac, dlj = u, torch.zeros(C, dtype=torch.float64, device=dev), None, None
    arr = [torch.as_tensor(np.asarray(a, dtype=np.float64), device=dev) for a in tm.arrays]
    S = torch.zeros(C, D, dtype=torch.float64, device=dev)
    L = torch.zeros(C, dtype=torch.float64, device=dev)
    total = lj
    for t in tm.terms:
        n = t.length

        def op(o):
            if o.kind == T.OP_CONST:
                return torch.full((1, 1), o.c, dtype=torch.float64, device=dev)
            if o.kind == T.OP_PARAM:
                return theta[:, o.a:o.a + 1]
            if o.kind == T.OP_DATA:
                return arr[o.a][:n][None, :]
            if o.kind == T.OP_PARAMVEC:
                return theta[:, o.a:o.a + n]
            if o.kind == T.OP_LIN:
                v = torch.full((1, 1), o.c, dtype=torch.float64, device=dev)
                for p, a, coef in o.lin:
                    e = coef * (arr[a][:n][None, :] if a >= 0 else 1.0)
                    v = v + e * (theta[:, p:p + 1] if p >= 0 else 1.0)
                return v
            X = arr[o.a][:n]
            return theta[:, o.b:o.b + X.shape[1]] @ X.T + o.c
        ops = [op(o) for o in (t.x, t.p0, t.p1)]
        f = _density(t, *ops).expand(C, n)
        total = total + t.weight * f.sum(1)
        # per-element partials with respect to the operand values (the densities are elementwise)
        leaf = [o.detach().expand(C, n).clone().requires_grad_(True) for o in ops]
        fl = t.weight * _density(t, *leaf).expand(C, n)
        L = L + fl.detach().abs().sum(1)
        if t.dist == T.CONSTANT:
            continue
        parts = torch.autograd.grad(fl.sum(), leaf, allow_unused=True)
        bounds = _summands(t, *(o.detach().expand(C, n) for o in ops))
        for o, g, b in zip((t.x, t.p0, t.p1), parts, bounds):
            if g is None or o.kind in (T.OP_CONST, T.OP_DATA):
                continue
            g = g.abs()
            b = abs(t.weight) * b
            assert torch.all(b >= g * (1 - 1e-12)), (T.DIST_NAMES[t.dist], float((g - b).max()))
            g = b
            if o.kind == T.OP_PARAM:
                S[:, o.a] += g.sum(1)
            elif o.kind == T.OP_PARAMVEC:
                S[:, o.a:o.a + n] += g
            elif o.kind == T.OP_LIN:
                for p, a, coef in o.lin:
                    if p >= 0:
                        S[:, p] += (g * abs(coef) * (arr[a][:n].abs()[None, :] if a >= 0 else 1.0)).sum(1)
            elif o.kind == T.OP_MATVEC:
                X = arr[o.a][:n]
                S[:, o.b:o.b + X.shape[1]] += g @ X.abs()
    grad, = torch.autograd.grad(total.sum(), u)
    if jac is not None:   # g_u = g_theta jac + dlogjac, the kernels' chain rule
        S = S * jac.detach().abs() + dlj.detach().abs()
    return total.detach(), grad.detach(), S, L


def _ratios(lp, g, ref):
    """worst |lp - lp64| / sum|w f| and |g - g64| / max(|g64|, S) over chains and coordinates"""
    lp64, g64, S, L = ref
    r_lp = float(((lp.double() - lp64).abs() / L).max())
    r_g = ((g.double() - g64).abs() / torch.maximum(g64.abs(), S))
    return r_lp, float(r_g.max()), tuple(int(i) for i in np.unravel_index(int(r_g.argmax()), r_g.shape))


# ----------------------------------------------------------------------------- catalogue
AFFINE = ("mu", "tau", "a", "b", "m")
DENSITIES = ("mu", "s", "r", "g", "q", "c")


def _data(kind, N, D, seed, positive=False):
    rs = np.random.default_rng(seed)
    X = rs.standard_normal((N, D)).astype(np.float32)
    beta = (rs.standard_normal(D) / np.sqrt(D)).astype(np.float32)
    if positive:   # coefficients with a HalfNormal prior
        beta = np.abs(beta) + np.float32(0.3)
    if kind == "logit":
        y = (rs.uniform(size=N) < 1 / (1 + np.exp(-(X.astype(np.float64) @ beta)))).astype(np.float32)
    elif kind == "normal_cw":
        y = (X @ beta + 1.5 + 0.9 * rs.standard_normal(N)).astype(np.float32)
    else:
        y = (X @ beta + 0.8 * rs.standard_normal(N)).astype(np.float32)
    t = np.linspace(-1, 1, 200).astype(np.float32)
    z = (0.3 + 0.7 * t + 0.5 * rs.standard_normal(200)).astype(np.float32)
    labels = (rs.uniform(size=50) < 0.4).astype(np.float32)
    return dict(X=X, y=y, beta=beta, t=t, z=z, labels=labels)


def _lik(ns, kind, Xb, ya, p):
    mx = ns.mx
    if kind == "normal_const":
        return mx.sum(ns.Normal(Xb, 0.8).log_prob(ya))
    if kind == "normal_sigma":
        return mx.sum(ns.Normal(Xb, p["sigma"]).log_prob(ya)) + ns.HalfNormal(1.0).log_prob(p["sigma"])
    if kind == "normal_cw":
        return 0.7 * mx.sum(ns.Normal(Xb + 1.5, 0.9).log_prob(ya))
    return mx.sum(ns.Bernoulli(logits=Xb).log_prob(ya))


def build(ns, model, kind, dat, order, bernoulli=True, pointwise=False):
    """(log_prob, init) of catalogue `model` with likelihood `kind`; `order` = parameter names in layout order
    ('beta' the coefficient vector, 'pad<k>' extra scalars with a Normal prior, 'sigma' the likelihood scale).
    `pointwise`: the same model with scalar coefficients b0.. in place of beta (pointwise class)"""
    mx = ns.mx
    D = dat["X"].shape[1]
    Xa, ya, ta, za, la = (mx.array(dat[k]) for k in ("X", "y", "t", "z", "labels"))
    cols = [mx.array(np.ascontiguousarray(dat["X"][:, j])) for j in range(D)] if pointwise else None

    def fn(p):
        if pointwise:
            Xb = p["b0"] * cols[0]
            for j in range(1, D):
                Xb = Xb + p[f"b{j}"] * cols[j]
            bv = None
        else:
            Xb, bv = Xa @ p["beta"], p["beta"]

        def coef_prior(dist):   # sum over the coefficients of one prior
            if bv is not None:
                return mx.sum(dist.log_prob(bv))
            out = dist.log_prob(p["b0"])
            for j in range(1, D):
                out = out + dist.log_prob(p[f"b{j}"])
            return out
        lp = _lik(ns, kind, Xb, ya, p)
        for name in order:
            if name.startswith("pad"):
                lp = lp + ns.Normal(0.3, 1.0).log_prob(p[name])
        if model == "affine":
            lp = (lp + coef_prior(ns.Normal(2.0 * p["mu"] + 1.0, p["tau"]))            # p0 affine, p1 parameter
                  + coef_prior(ns.Normal(p["m"], p["tau"]))                            # hierarchical: both parameters
                  + ns.Normal(0, 1).log_prob(p["mu"] - p["a"])                         # x affine
                  + ns.HalfNormal(1.0).log_prob(p["tau"])
                  + ns.Normal(0, 0.5 * p["tau"] + 1.0).log_prob(p["m"])                # p1 affine
                  + mx.sum(ns.Normal(p["a"] + p["b"] * ta, 0.5).log_prob(za)))         # affine with a data coefficient
        elif model == "densities":
            lp = (lp + ns.Normal(0.5, 2.0).log_prob(p["mu"])
                  + ns.HalfNormal(1.5).log_prob(p["s"])
                  + ns.Exponential(2.0).log_prob(p["r"])
                  + 0.5 * ns.Gamma(3.0, p["r"]).log_prob(p["g"])
                  + ns.Beta(2.0, 3.0).log_prob(p["q"])
                  + ns.Normal(p["mu"], p["s"]).log_prob(p["c"])
                  + coef_prior(ns.Normal(0, 2.0))
                  - 0.25 * coef_prior(ns.Normal(0.1, 3.0))
                  + 1.7)
            if bernoulli:
                lp = lp + mx.sum(ns.Bernoulli(logits=p["c"]).log_prob(la))
        elif model == "constrained":
            lp = lp + coef_prior(ns.HalfNormal(1.0))
        return lp
    init = {}
    for name in order:
        if name == "beta" and pointwise:
            init.update({f"b{j}": 0.5 for j in range(D)})
        elif name == "beta":
            init["beta"] = np.full(D, 0.5, np.float32)
        else:
            init[name] = 0.5
    return fn, init


def _points(tm, codes, dat, C, seed, spread=0.05):
    """[C, D] float32 test points in the sampler's coordinates: coefficients near the data's beta, scalars inside
    their supports"""
    rs = np.random.default_rng(seed)
    th = np.zeros((C, tm.D))
    for name, (off, n, _) in tm.layout.items():
        if name == "beta":
            th[:, off:off + n] = dat["beta"][None, :n] + spread * rs.standard_normal((C, n))
        elif name.startswith("b") and name[1:].isdigit():
            th[:, off] = dat["beta"][int(name[1:])] + spread * rs.standard_normal(C)
        elif name in _POS:
            th[:, off] = rs.uniform(0.6, 1.4, C)
        elif name == "q":
            th[:, off] = rs.uniform(0.2, 0.8, C)
        else:
            th[:, off] = 0.5 * rs.standard_normal(C)
    if codes is not None:
        pos, unit = codes == _cabi.TF_LOG, codes == _cabi.TF_LOGIT
        th[:, pos] = np.log(th[:, pos])
        th[:, unit] = np.log(th[:, unit]) - np.log1p(-th[:, unit])
    return th.astype(np.float32)


def _order(model, beta_off, D, sigma=None, pads=0):
    names = list(AFFINE if model == "affine" else DENSITIES if model == "densities" else ()) + \
        [f"pad{k}" for k in range(pads)]
    order = names[:beta_off] + ["beta"] + names[beta_off:]
    if sigma is not None:
        order.insert(sigma, "sigma")
    return order


# ----------------------------------------------------------------------------- 1. the reference (CPU)
ORACLE_CASES = [("affine", "normal_const", _order("affine", 3, 5)),
                ("affine", "normal_sigma", _order("affine", 0, 4, sigma=6)),
                ("affine", "normal_cw", _order("affine", 5, 3)),
                ("densities", "normal_const", _order("densities", 4, 8, pads=1)),
                ("densities", "normal_sigma", _order("densities", 2, 5, sigma=0)),
                ("constrained", "normal_const", ["beta"])]


@pytest.mark.parametrize("tf", [None, "auto"])
@pytest.mark.parametrize("model,kind,order", ORACLE_CASES)
def test_float64_reference_against_oracle(model, kind, order, tf):
    from oracle import ns as oracle
    D = 5 if model != "densities" else 8
    dat = _data(kind, 60, D, seed=3, positive=model == "constrained")
    fn, init = build(B.ns, model, kind, dat, order, bernoulli=False)
    fo, _ = build(oracle.ns, model, kind, dat, order, bernoulli=False)
    tm = T.trace(fn, init)
    codes = tm.transform_codes() if tf else np.zeros(tm.D, np.int32)
    assert tf is None or np.any(codes != 0)
    u = _points(tm, codes, dat, 4, seed=1)
    lp, g, S, L = eval64(tm, torch.from_numpy(u), codes)
    for c in range(u.shape[0]):
        uc = u[c].astype(np.float64)
        theta = uc.copy()
        theta[codes == _cabi.TF_LOG] = np.exp(uc[codes == _cabi.TF_LOG])
        theta[codes == _cabi.TF_LOGIT] = 1 / (1 + np.exp(-uc[codes == _cabi.TF_LOGIT]))
        params = {name: theta[off:off + n].reshape(shp) if shp else theta[off] for name, (off, n, shp) in tm.layout.items()}
        lo, go = oracle.value_and_grad(fo, params, "float64")
        gv = np.zeros(tm.D)
        for name, (off, n, shp) in tm.layout.items():
            gv[off:off + n] = np.asarray(go[name]).reshape(-1)
        # chain rule and log-Jacobian of the transforms on the oracle's side
        lj = 0.0
        for d in range(tm.D):
            if codes[d] == _cabi.TF_LOG:
                lj += uc[d]
                gv[d] = gv[d] * theta[d] + 1.0
            elif codes[d] == _cabi.TF_LOGIT:
                lj += math.log(theta[d]) + math.log1p(-theta[d])
                gv[d] = gv[d] * theta[d] * (1 - theta[d]) + 1 - 2 * theta[d]
        # the traced constants are float32 (as on the device), the oracle's float64: agreement to ~1e-8 relative
        assert abs(float(lp[c]) - (float(lo) + lj)) <= 1e-7 * float(L[c]), (c, float(lp[c]), float(lo) + lj)
        err = np.abs(g[c].numpy() - gv) / np.maximum(np.abs(gv), S[c].numpy())
        assert np.all(err <= 1e-7), (c, float(err.max()), int(err.argmax()))
        assert torch.all(S[c] >= g[c].abs() - 1e-9 * S[c].max())   # S bounds the gradient it is the sum for


def test_float64_reference_sees_a_dropped_affine_gradient():
    """the bound is tight enough to see the defect it is for: a gradient without the contributions of the affine
    operands is far outside it"""
    dat = _data("normal_const", 60, 5, seed=3)
    fn, init = build(B.ns, "affine", "normal_const", dat, _order("affine", 3, 5))
    tm = T.trace(fn, init)
    u = torch.from_numpy(_points(tm, None, dat, 3, seed=2))
    ref = eval64(tm, u)
    lin_free = T.TracedModel(tm.D, tm.layout, [t for t in tm.terms if T.OP_LIN not in (t.x.kind, t.p0.kind, t.p1.kind)],
                             tm.arrays, tm.lin)
    _, r, _ = _ratios(ref[0].float(), eval64(lin_free, u)[1].float(), ref)
    assert r > 0.1, r


# ----------------------------------------------------------------------------- 2. GLM class on the device
def _compile(fn, init, path, form, tf, **kw):
    from mlx_mcmc_b200.engine import compile_model
    m = compile_model(fn, init, cache=False, glm_path=path, glm_form=form or "auto", transforms=tf, **kw)
    assert m.model_class == 1 and m.glm_path == path and (form is None or m.glm_form == form), (m.glm_path, m.glm_form)
    assert tf is None or m.has_transforms
    return m


def _check(model, u, label, tol=TOL):
    """log p and gradient of `model` at u [C, D] (sampler coordinates) against eval64, per chain and coordinate; a
    value-only call and a repeated call bit for bit"""
    theta = torch.from_numpy(u).cuda()
    lp, g = model.logp_grad(theta)
    ref = eval64(model.traced, theta.double(), model.tf_codes if model.has_transforms else None)
    r_lp, r_g, (wc, wj) = _ratios(lp, g, ref)
    name = next(k for k, (off, n, _) in model.layout.items() if off <= wj < off + n)
    print(f"{label}: worst logp {r_lp:.2e}, worst grad {r_g:.2e} (chain {wc}, coordinate {wj} = {name})")
    assert torch.isfinite(lp).all() and torch.isfinite(g).all()
    lp_v, _ = model.logp_grad(theta, want_grad=False)
    lp2, g2 = model.logp_grad(theta)
    assert torch.equal(lp_v, lp), "value-only log p differs"
    assert torch.equal(lp2, lp) and torch.equal(g2, g), "repeated call differs"
    assert r_lp <= tol and r_g <= tol, (label, r_lp, r_g, name)


NORMAL_KINDS = ("normal_const", "normal_sigma", "normal_cw")
PATH_FORMS = [(k, p, f) for k in NORMAL_KINDS
              for p, f in (("simt", "stream"), ("tc", "stream"), ("tc", "gram"), ("tc16", "stream"), ("tc16", "gram"))] + \
             [("logit", p, None) for p in ("simt", "tc", "tc16")]


def _case_order(model, kind, beta_off, D, sigma=None, pads=0):
    if kind != "normal_sigma":
        sigma = None
    elif sigma is None:
        sigma = beta_off + 1          # right after beta
    return _order(model, beta_off, D, sigma=sigma, pads=pads)


@pytest.mark.gpu
@pytest.mark.parametrize("tf", [None, "auto"])
@pytest.mark.parametrize("kind,path,form", PATH_FORMS)
@pytest.mark.parametrize("model", ["affine", "densities"])
def test_prior_terms_every_path(cuda, model, kind, path, form, tf):
    """every operand kind and prior density next to every likelihood kind, on every path and form"""
    D = 5 if model == "affine" else 8
    order = _case_order(model, kind, 3, 5) if model == "affine" else _case_order(model, kind, 4, 8, pads=1)
    dat = _data(kind, 500, D, seed=11)
    fn, init = build(B.ns, model, kind, dat, order)
    m = _compile(fn, init, path, form, tf)
    _check(m, _points(m.traced, m.tf_codes if tf else None, dat, 129, seed=5), f"{model} {kind} {path}/{form} tf={tf}")


# (model, beta_off, D, sigma position or None, padding scalars, kind)
LAYOUTS = [("affine", 0, 5, None, 0, "normal_const"),           # beta first
           ("affine", 5, 1, None, 0, "normal_const"),           # beta last, D = 1
           ("affine", 3, 129, None, 0, "normal_const"),         # beta in the middle at offset 3
           ("densities", 4, 8, None, 2, "normal_const"),        # Dtot 16, offset 4, D 8: the float4 finish loop
           ("densities", 4, 8, None, 1, "normal_const"),        # Dtot 15: float4 coefficient prior on every 4th row
           ("densities", 3, 8, 0, 0, "normal_sigma"),           # sigma before beta (offset 4)
           ("affine", 0, 8, 1, 0, "normal_sigma")]              # sigma right after beta


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 129, 300])
@pytest.mark.parametrize("path,form", [("simt", "stream"), ("tc", "gram"), ("tc16", "stream"), ("tc16", "gram")])
@pytest.mark.parametrize("layout", LAYOUTS, ids=lambda c: f"{c[0]}-off{c[1]}-D{c[2]}-sig{c[3]}-pad{c[4]}")
def test_layouts_and_batches(cuda, layout, path, form, C):
    model, off, D, sig, pads, kind = layout
    order = _case_order(model, kind, off, D, sigma=sig, pads=pads)
    dat = _data(kind, 300, D, seed=D + off)
    fn, init = build(B.ns, model, kind, dat, order)
    m = _compile(fn, init, path, form, None)
    assert m.layout["beta"][0] == (off if sig is None or sig > off else off + 1)
    _check(m, _points(m.traced, None, dat, C, seed=C), f"{order} {path}/{form} C={C}")


@pytest.mark.gpu
@pytest.mark.parametrize("tf", [None, "auto"])
@pytest.mark.parametrize("path,form", [("simt", "stream"), ("tc", "stream"), ("tc16", "stream"), ("tc16", "gram")])
@pytest.mark.parametrize("N", [6000, 12000])
def test_affine_prior_staged_and_unstaged(cuda, N, path, form, tf):
    """the prior's 1-D arrays (y, t, z) are staged in shared memory up to 32 KB: y alone is 24 KB at N = 6000 and
    48 KB at N = 12000"""
    dat = _data("normal_sigma", N, 5, seed=N)
    fn, init = build(B.ns, "affine", "normal_sigma", dat, _case_order("affine", "normal_sigma", 3, 5))
    m = _compile(fn, init, path, form, tf)
    _check(m, _points(m.traced, m.tf_codes if tf else None, dat, 129, seed=3), f"affine N={N} {path}/{form} tf={tf}")


def _halfnormal_mode(dat, sigma=0.8):
    """posterior mode of the constrained-coefficient model in u = log beta (float64 Newton steps)"""
    X, y = dat["X"].astype(np.float64), dat["y"].astype(np.float64)
    XtX, Xty = X.T @ X, X.T @ y
    u = np.log(np.clip(np.linalg.solve(XtX, Xty), 0.05, None))
    for _ in range(50):
        b = np.exp(u)
        gb = -b + (Xty - XtX @ b) / sigma ** 2
        gu = gb * b + 1.0
        H = (b[:, None] * (-np.eye(len(b)) - XtX / sigma ** 2) * b[None, :]) + np.diag(gb * b)
        step = np.linalg.solve(H, gu)
        u = u - step
        if np.max(np.abs(step)) < 1e-12:
            break
    return u, np.sqrt(np.diag(np.linalg.inv(-H)))


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["stream", "gram"])
def test_constrained_coefficients_at_c3_size(cuda, form):
    """HalfNormal prior on the coefficient vector under transforms='auto' (beta sampled as log beta), chains around the
    posterior mode, N = 10,000 and D = 100: the centring must use the constrained coefficients"""
    dat = _data("normal_const", 10000, 100, seed=21, positive=True)
    fn, init = build(B.ns, "constrained", "normal_const", dat, ["beta"])
    from mlx_mcmc_b200.engine import compile_model
    m = compile_model(fn, init, cache=False, transforms="auto", glm_form=form)
    assert m.model_class == 1 and m.glm_form == form and np.all(m.tf_codes == _cabi.TF_LOG)
    mode, sd = _halfnormal_mode(dat)
    rs = np.random.default_rng(4)
    u = (mode[None, :] + sd[None, :] * rs.standard_normal((256, 100))).astype(np.float32)
    _check(m, u, f"constrained beta N=10000 D=100 {m.glm_path}/{form}")


# ----------------------------------------------------------------------------- 3. sampler path, across the classes
def _cross(path, tf, N=300):
    dat = _data("normal_const", N, 5, seed=8)
    order = _order("affine", 3, 5)
    fg, ig = build(B.ns, "affine", "normal_const", dat, order)
    fp, ip = build(B.ns, "affine", "normal_const", dat, order, pointwise=True)
    mg = _compile(fg, ig, path, None, tf)
    from mlx_mcmc_b200.engine import compile_model
    mp = compile_model(fp, ip, cache=False, transforms=tf)
    assert mp.model_class == 0 and mg.D == mp.D
    assert [mp.layout[f"b{j}"][0] for j in range(5)] == list(range(mg.layout["beta"][0], mg.layout["beta"][0] + 5))
    assert np.array_equal(mg.tf_codes, mp.tf_codes)
    return dat, mg, mp


@pytest.mark.gpu
@pytest.mark.parametrize("tf", [None, "auto"])
def test_pointwise_comparator_against_float64(cuda, tf):
    """the pointwise form of the affine model (coefficients as scalars, X @ beta as an affine expression with data
    coefficients) on 1, 4 and 32 lanes per chain and on the general path"""
    from mlx_mcmc_b200.engine import compile_model
    dat, mg, mp = _cross("tc16", tf)
    u = _points(mp.traced, mp.tf_codes if tf else None, dat, 200, seed=6)
    for lanes in (1, 4, 32):
        theta = torch.from_numpy(u).cuda()
        lp, g = mp.logp_grad(theta, lanes=lanes)
        r = _ratios(lp, g, eval64(mp.traced, theta.double(), mp.tf_codes if tf else None))
        print(f"pointwise lanes={lanes} tf={tf}: worst logp {r[0]:.2e}, worst grad {r[1]:.2e} at {r[2]}")
        assert r[0] <= TOL and r[1] <= TOL, (lanes, r)
    fp, ip = build(B.ns, "affine", "normal_const", dat, _order("affine", 3, 5), pointwise=True)
    mgen = compile_model(fp, ip, cache=False, transforms=tf, pointwise_path="general")
    _check(mgen, u, f"pointwise general tf={tf}")


@pytest.mark.gpu
@pytest.mark.parametrize("tf", [None, "auto"])
@pytest.mark.parametrize("path", ["tc16", "tc", "simt"])
def test_cross_class_first_nuts_transition(cuda, path, tf):
    """tc16 runs NUTS on the fused state kernel (its own inlined finish), tc / simt on the unfused loop: the first
    transition of the GLM form must follow the pointwise form of the same model"""
    from mlx_mcmc_b200.engine import ChainState, launch_nuts
    dat, mg, mp = _cross(path, tf)
    C = 512
    theta = torch.from_numpy(_points(mg.traced, mg.tf_codes if tf else None, dat, C, seed=9)).cuda()
    lg, gg = mg.logp_grad(theta)
    lq, gq = mp.logp_grad(theta)
    ref = eval64(mg.traced, theta.double(), mg.tf_codes if tf else None)
    for lab, lp, g in (("glm", lg, gg), ("pointwise", lq, gq)):
        r = _ratios(lp, g, ref)
        print(f"{path} tf={tf} {lab}: worst logp {r[0]:.2e}, worst grad {r[1]:.2e} at {r[2]}")
        assert r[0] <= TOL and r[1] <= TOL, (lab, r)
    depths = []
    for m in (mg, mp):
        st = ChainState(m, theta.clone(), 0.05)
        dep = torch.empty((1, C), dtype=torch.int32, device="cuda")
        launch_nuts(st, 1, 10, _cabi.ADAPT_NONE, _cabi.COMPAT_CORRECT, 0.65, 1234, 0, depths=dep)
        depths.append(dep[0].cpu().numpy())
    same = float(np.mean(depths[0] == depths[1]))
    print(f"{path} tf={tf} first NUTS transition: equal depths for {100 * same:.1f} % of {C} chains, "
          f"mean depth {depths[0].mean():.2f}")
    assert same >= 0.95
