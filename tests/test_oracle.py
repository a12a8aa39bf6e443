"""CPU: the oracle restatement against the golden vectors produced from the unmodified reference
(oracle/make_golden.py), plus the reference's own known-answer log_prob tests run on the oracle."""
import json
import math
import os

import numpy as np
import pytest

from oracle.ns import Tape, ns, samplers, value_and_grad
from mlx_mcmc_b200 import workloads as W
from util import RUN_FIXTURES, golden

mx = ns.mx


def test_logp_grad_matches_reference_fixtures():
    g = golden("logp_grad")
    for model, rows in g.items():
        fn, _, _ = W.ALL_SMALL[model](ns)
        for row in rows:
            lp, grad = value_and_grad(fn, row["params"], "float32")
            assert np.array_equal(np.float32(lp), np.float32(row["logp32"]), equal_nan=True), (model, row["params"])
            for n, gv in row["grad32"].items():
                assert np.array_equal(grad[n].astype(np.float32), np.asarray(gv, dtype=np.float32), equal_nan=True)
            lp64, grad64 = value_and_grad(fn, row["params"], "float64")
            if math.isfinite(row["logp64"]):
                assert abs(lp64 - row["logp64"]) <= 1e-12 * max(1.0, abs(row["logp64"]))


def test_survey_golden_values():
    """fp64 values quoted in SURVEY.md 8(c) for the benchmark models"""
    fn, init, _ = W.c1_normal(ns)
    lp, g = value_and_grad(fn, init, "float64")
    assert abs(lp - (-1408.585347591399)) < 2e-4 and abs(g["mu"] - 479.2306965211812) < 2e-5 and abs(g["sigma"] - 2523.1894827593087) < 2e-4
    fn, init, _ = W.c2_event_rate(ns)
    lp, g = value_and_grad(fn, init, "float64")
    assert abs(lp - 5.152357277683324) < 2e-6 and abs(g["rate"] - 10.400925534563058) < 2e-6
    fn, init, _ = W.c5_ab_test(ns)
    lp, _ = value_and_grad(fn, init, "float64")
    assert abs(lp - (-7.136865754315352)) < 2e-4   # logB constants are float32 in the reference


@pytest.mark.parametrize("name", RUN_FIXTURES)
def test_port_reproduces_reference_draws(name):
    """Same stand-in keys => the restatement's draws equal the reference's, bit for bit, and it ends on the committed
    step size having consumed the committed random numbers (the slots the GPU parity tests inject)."""
    g = golden(name)
    fn, init, _ = W.ALL_SMALL[g["model"]](ns)
    kw = dict(g["kwargs"])
    tape, eps = Tape(), None
    if g["method"] == "hmc":
        s, a, eps = samplers.hmc_port(fn, init, key=mx.random.key(g["seed"]), tape=tape, **kw)
    elif g["method"] == "nuts":
        s, a, eps = samplers.nuts_port(fn, init, key=mx.random.key(g["seed"]), tape=tape, **kw)
    else:
        s, a = samplers.run_port(fn, init, method="metropolis", random_seed=g["seed"], tape=tape, **kw)
    assert a == g["accept_rate"]
    for k, v in g["draws"].items():
        assert np.array_equal(np.asarray(s[k], dtype=np.float32), np.asarray(v, dtype=np.float32))
    assert json.loads(json.dumps(eps)) == g["final_step_size"]
    normals = [{"it": k[0], "param": k[1], "z": np.asarray(v, dtype=np.float64).tolist()} for k, v in tape.normals.items()]
    uniforms = [{"slot": list(k), "u": float(v)} for k, v in tape.uniforms.items()]
    assert json.loads(json.dumps(normals)) == g["tape"]["normals"]
    assert json.loads(json.dumps(uniforms)) == g["tape"]["uniforms"]


# --- the reference's known-answer tests (tests/test_distributions.py, tests/test_new_distributions.py) ---
def test_known_answers_on_oracle():
    f = lambda a: float(a)  # noqa: E731
    assert abs(f(ns.Normal(0, 1).log_prob(0.0)) - (-0.5 * math.log(2 * math.pi))) < 1e-5
    assert f(ns.Normal(0, 1).log_prob(1.0)) == f(ns.Normal(0, 1).log_prob(-1.0))
    assert abs(f(ns.HalfNormal(1).log_prob(0.0)) - (math.log(2) - 0.5 * math.log(2 * math.pi))) < 1e-5
    assert f(ns.HalfNormal(1).log_prob(-1.0)) == -math.inf
    for x in (-0.1, 1.5, 0.0, 1.0):
        assert f(ns.Beta(2, 2).log_prob(x)) == -math.inf
    assert math.isfinite(f(ns.Beta(2, 2).log_prob(0.5)))
    assert f(ns.Gamma(2, 1).log_prob(-1.0)) == -math.inf and f(ns.Gamma(2, 1).log_prob(1.5)) < 0
    assert abs(f(ns.Exponential(2).log_prob(0.0)) - math.log(2)) < 1e-6 and f(ns.Exponential(2).log_prob(-1.0)) == -math.inf
    c = ns.Categorical(probs=[0.2, 0.5, 0.3])
    assert abs(f(c.log_prob(0)) - math.log(0.2)) < 1e-2 and abs(f(c.log_prob(1)) - math.log(0.5)) < 1e-2
    assert f(c.log_prob(-1)) == -math.inf and f(c.log_prob(3)) == -math.inf
    with pytest.raises(ValueError):
        ns.Categorical()
    with pytest.raises(ValueError):
        ns.Categorical(probs=[0.5, 0.5], logits=[0.0, 0.0])


def test_diagnostics_restatement_matches_reference_fixture():
    """oracle/refport/diagnostics.py against the answers the reference's own function bodies gave
    (tests/golden/diagnostics.json, written by oracle/make_golden_diag.py)."""
    from oracle.refport import diagnostics as D
    g = golden("diagnostics")
    for row in g["ess"]:
        x = np.asarray(row["x"], dtype=np.float32)
        assert float(D.compute_ess(x)) == row["ess06"], (row["kind"], row["n"])
        if row["ess02"] is not None:
            assert float(D.compute_ess_example02(x)) == row["ess02"], (row["kind"], row["n"])
    smp = {"mu": np.asarray(g["summary"]["samples"]["mu"], dtype=np.float32),
           "beta": np.asarray(g["summary"]["samples"]["beta"], dtype=np.float32)}
    assert D.summary(smp, g["summary"]["credible_interval"]) == g["summary"]["table"]
    # the product's host-side estimator is the same function
    from mlx_mcmc_b200.diagnostics import compute_ess
    for row in g["ess"]:
        x = np.asarray(row["x"], dtype=np.float32)
        assert abs(compute_ess(x) - row["ess06"]) <= 1e-4 * abs(row["ess06"])


@pytest.mark.skipif(not os.path.isdir(os.environ.get("B2M_REFERENCE", "")),
                    reason="set B2M_REFERENCE to a checkout of the upstream korentomas/mlx-mcmc source to run it")
def test_committed_fixtures_reproduce_from_the_unmodified_reference():
    """The pin itself, re-checked where the reference is at hand: oracle/make_golden.py --check runs the UNMODIFIED
    reference samplers on the mlx.core stand-in and compares draws, acceptance rate and consumed random numbers with
    the committed JSON (one fixture per sampler keeps the CPU suite short; the generator asserts all of them)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "oracle", "make_golden.py"), "--check", "hmc_c2", "mh_c5",
                          "nuts_c2"], capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stdout[-1500:] + out.stderr[-1500:]
    assert out.stdout.count("committed fixture reproduces") == 3
