"""GPU: the GLM NUTS tree keeps its saved states (edges, candidate, parked subtrees) in per-chain slots addressed by
index.  These runs push the slot bookkeeping to its limits on every schedule: trees that reach the depth cap of 12
(the most parked subtrees, hence the most live slots) and divergence-heavy trees whose subtrees end in the middle of a
doubling (stack entries abandoned mid-way).  The schedules must agree on every tree and deliver every draw."""
import numpy as np
import pytest
import torch

import mlx_mcmc_b200 as B
from mlx_mcmc_b200 import _cabi, workloads as W
from mlx_mcmc_b200.engine import ChainState, compile_model, launch_nuts

pytestmark = pytest.mark.gpu

# (schedule name, glm_path, b2m schedule): tc16 takes the fused state kernel, tc (tf32) the unfused asynchronous loop
SCHEDULES = [("fused", "tc16", _cabi.SCHED_ASYNC), ("async", "tc", _cabi.SCHED_ASYNC), ("sync", "tc16", _cabi.SCHED_SYNC)]


def _run(d, step_sizes, n_iter, max_tree_depth):
    fn, init, meta = W.regression(B.ns, 512, d, seed=11)
    m, V = W.regression_posterior(meta)
    C = len(step_sizes)
    rng = np.random.default_rng(5)
    theta0 = (m[None, :] + rng.standard_normal((C, d)) @ np.linalg.cholesky(V).T).astype(np.float32)
    out = {}
    for name, path, schedule in SCHEDULES:
        model = compile_model(fn, init, cache=False, glm_path=path)
        assert model.glm_path == path
        st = ChainState(model, torch.from_numpy(theta0).cuda(), 1.0)
        st.step_size.copy_(torch.from_numpy(np.asarray(step_sizes, dtype=np.float64)))
        draws = torch.full((n_iter, C, d), float("nan"), device="cuda")
        depths = torch.full((n_iter, C), -1, dtype=torch.int32, device="cuda")
        launch_nuts(st, n_iter, max_tree_depth, _cabi.ADAPT_NONE, _cabi.COMPAT_CORRECT, 0.8, 123, 0, draws=draws,
                    depths=depths, schedule=schedule)
        torch.cuda.synchronize()
        out[name] = (draws.cpu().numpy(), depths.cpu().numpy(), st.n_leaves.cpu().numpy(), st.n_diverge.cpu().numpy())
    return out, V


@pytest.mark.parametrize("d", [8, 13])   # D % 4 == 0 takes the float4 leaf passes, the other the scalar ones
def test_slots_trees_at_the_depth_cap(cuda, d):
    """A step size far below the posterior scale: no U-turn and no divergence before depth 12, so every transition
    builds all 4095 leaves and parks a subtree on each of the 11 lower levels."""
    n_iter, md = 2, 12
    out, V = _run(d, [2e-6] * 16, n_iter, md)
    for name, (draws, depths, leaves, div) in out.items():
        assert np.isfinite(draws).all(), name
        assert (depths == md).all(), (name, np.unique(depths))
        assert (leaves == n_iter * ((1 << md) - 1)).all() and (div == 0).all(), name


@pytest.mark.parametrize("d", [8, 13])
def test_slots_divergent_subtrees(cuda, d):
    """Step sizes from half to eight times the smallest posterior scale: the unstable chains diverge after a few
    leaves, often inside a subtree of depth >= 2, which ends the doubling with parked subtrees still on the stack."""
    n_iter, md = 8, 10
    fn, init, meta = W.regression(B.ns, 512, d, seed=11)
    sd_min = float(np.sqrt(np.linalg.eigvalsh(W.regression_posterior(meta)[1]).min()))
    steps = sd_min * np.geomspace(0.5, 8.0, 128)
    out, _ = _run(d, steps, n_iter, md)
    ref_depths = out["sync"][1]
    for name, (draws, depths, leaves, div) in out.items():
        assert np.isfinite(draws).all(), name
        assert ((depths >= 1) & (depths <= md)).all(), name
        assert (depths == ref_depths).mean() > 0.95, (name, (depths == ref_depths).mean())
        full = ((1 << depths.astype(np.int64)) - 1).sum(0)   # leaves of trees whose last subtree ran to completion
        assert div.sum() > 0 and (leaves < full).any(), (name, int(div.sum()))
        assert (depths >= 3).any(), name
