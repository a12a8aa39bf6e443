"""High-level MCMC interface with the reference's call convention (mlx_mcmc/inference/mcmc.py:10-246)."""
from __future__ import annotations

import numpy as np

from .. import core as mx
from ..kernels.hmc import hmc
from ..kernels.metropolis import metropolis_hastings
from ..kernels.nuts import nuts

_RULE = "=" * 70


class MCMC:
    """``MCMC(log_prob_fn).run(initial_params, ...)`` -> dict of numpy draws; ``self.samples`` and
    ``self.acceptance_rate`` are set as in the reference (mcmc.py:33-36,99-100,187).

    ``log_prob_fn(params)`` is traced once per ``run`` configuration into a term table and executed by
    the CUDA kernels; it must be written against ``mlx_mcmc_b200.core`` (as ``mx``) and the library
    distributions.  Unsupported operations raise ``UnsupportedOpError``.
    """

    def __init__(self, log_prob_fn):
        self.log_prob_fn = log_prob_fn
        self.samples = None
        self.acceptance_rate = None
        self.info = None
        self._single_chain = True
        self._waic_source = None

    def run(self, initial_params, num_samples=1000, num_warmup=1000, method='metropolis', proposal_scale=0.1,
            random_seed=0, verbose=True, **kwargs):
        """Same positional/keyword arguments as the reference (mcmc.py:38-48); ``**kwargs`` go to the
        sampler verbatim (mcmc.py:96,122,156,177), so e.g. ``step_size`` with ``method='metropolis'``
        raises TypeError exactly as there.  Extra keyword-only sampler options (``num_chains``,
        ``adapt``, ``compat``, ``return_torch`` ...) ride in ``kwargs`` too."""
        # keyword-only extensions for one-process-per-GPU runs under torchrun (the reference is single device):
        #   device=i          run on cuda:i (default: the current device)
        #   shard='chains'    this rank runs its block of the `num_chains` global chains; draws of all ranks are gathered
        #   shard='obs'       GLM-class models: every rank holds a row shard of (X, y) and all chains (dist.py);
        #                     with slice_state='peer' | 'nccl' the per-chain work is sliced over the ranks too
        device = kwargs.pop("device", kwargs.pop("devices", None))
        shard = kwargs.pop("shard", None)
        if isinstance(device, (list, tuple)):
            if len(device) != 1:
                raise ValueError("one process drives one GPU: pass device=i (launch one process per GPU with torchrun)")
            device = device[0]
        if device is not None:
            import torch
            torch.cuda.set_device(int(device))
        if shard not in (None, "chains", "obs"):
            raise ValueError(f"Unknown shard mode: {shard}")
        gather = None
        if shard is not None:
            from .. import dist as D_
            rank, world = D_.rank_world()
            total = int(kwargs.get("num_chains", 1))
            if shard == "chains" and world > 1:
                count, offset = D_.shard_chains(total, rank, world)
                if count == 0:
                    raise ValueError(f"rank {rank} would own no chains (num_chains={total}, world={world})")
                kwargs["num_chains"], kwargs["chain_offset"] = count, offset
                gather = (D_, count)
            elif shard == "obs" and world > 1:
                peer = total if kwargs.get("slice_state") in (True, "peer") else None
                kwargs["model"] = D_.compile_obs_sharded(self.log_prob_fn, initial_params, peer_chains=peer)
        self._single_chain = int(kwargs.get("num_chains", 1)) == 1 and gather is None
        # what waic() needs to find the same device model again (compile_model's cache) after the run
        self._waic_source = dict(initial_params=initial_params, shard=shard, model=kwargs.get("model"),
                                 transforms=kwargs.get("transforms"), cache=kwargs.get("cache", True))
        out = self._run_local(initial_params, num_samples, num_warmup, method, proposal_scale, random_seed, verbose, kwargs)
        if gather is not None:
            D_, count = gather
            local = self.samples if count > 1 else {k: v[None] for k, v in self.samples.items()}
            self.samples = D_.gather_draws(local, count)
            import torch
            dev = torch.device("cuda") if D_.td.get_backend() == "nccl" else None
            tot = D_.reduce_stats({"acc": self.acceptance_rate * count, "n": count}, "sum", None, dev)
            self.acceptance_rate = tot["acc"] / max(tot["n"], 1.0)
            out = self.samples
        return out

    def _run_local(self, initial_params, num_samples, num_warmup, method, proposal_scale, random_seed, verbose, kwargs):
        if method in ('hmc', 'nuts'):
            if verbose:
                print(f"\n{_RULE}\nB200-MCMC: {method.upper()} Sampling\n{_RULE}\n")
            sampler = hmc if method == 'hmc' else nuts
            out = sampler(self.log_prob_fn, initial_params, num_samples=num_samples, num_warmup=num_warmup,
                          key=mx.random.key(random_seed), **kwargs)
            samples, accept_rate = out[0], out[1]
            self.info = out[2] if len(out) > 2 else None
            self.samples = samples if kwargs.get("return_torch") else {k: np.array(v) for k, v in samples.items()}
            self.acceptance_rate = accept_rate
            if verbose:
                print(f"Sampling acceptance rate: {accept_rate:.2%}\n{_RULE}\nSampling complete!\n{_RULE}\n")
            return self.samples
        elif method == 'metropolis':
            sampler = metropolis_hastings
        else:
            raise ValueError(f"Unknown sampling method: {method}")

        if verbose:
            print(f"\n{_RULE}\nB200-MCMC: {method.upper()} Sampling\n{_RULE}\n")
        # warm-up is a separate sampler call with `random_seed`; sampling restarts from its last draw
        # with `random_seed + 1` (mcmc.py:146-178)
        extra = {}
        if num_warmup > 0:
            wkw = dict(kwargs)
            wkw.update(return_info=True, return_torch=True)
            _, warm_accept, winfo = sampler(self.log_prob_fn, initial_params, num_samples=num_warmup,
                                            proposal_scale=proposal_scale, random_seed=random_seed, verbose=False, **wkw)
            if verbose:
                print(f"Warmup phase: {num_warmup} samples, acceptance rate: {warm_accept:.2%}\n")
            # the last warm-up draw of every chain is the chain's final position (mcmc.py:162)
            extra = dict(theta0=winfo.state.theta, model=winfo.model)
        out = sampler(self.log_prob_fn, initial_params, num_samples=num_samples, proposal_scale=proposal_scale,
                      random_seed=random_seed + 1 if num_warmup > 0 else random_seed, verbose=False, **kwargs, **extra)
        self.samples, self.acceptance_rate = out[0], out[1]
        self.info = out[2] if len(out) > 2 else None
        if verbose:
            print(f"Sampling phase: {num_samples} samples\nSampling acceptance rate: {self.acceptance_rate:.2%}")
            print(f"\n{_RULE}\nSampling complete!\n{_RULE}\n")
        if not kwargs.get("return_torch"):
            self.samples = {k: np.array(v) for k, v in self.samples.items()}
        return self.samples

    def summary(self, credible_interval=0.95):
        """mean / std / median / lower / upper percentile per parameter, keys as in mcmc.py:219-225.
        Multi-chain draws are pooled over chains."""
        if self.samples is None:
            raise ValueError("Must run sampling first. Call run() method.")
        alpha = 1 - credible_interval
        lo, hi = 100 * alpha / 2, 100 * (1 - alpha / 2)
        table = {}
        for name, draws in self.samples.items():
            if hasattr(draws, "is_cuda") and draws.is_cuda:
                # device draws (return_torch=True): moments from the diagnostics kernels, the three order statistics from
                # ONE radix-select pass set over the pooled draws (b2m_quantiles) -- the draws never travel to the host
                from ..diagnostics import device_quantiles, device_summary
                x = draws.reshape(1, -1, 1).permute(1, 0, 2).contiguous().float()      # one pooled series [S*, 1, 1]
                cols = device_summary(x, None, ess=False)
                med, q_lo, q_hi = device_quantiles(draws.reshape(-1).float(), [0.5, lo / 100.0, hi / 100.0])
                table[name] = {'mean': float(cols["mean"][0]), 'std': float(cols["std"][0]), 'median': med,
                               f'{lo:.1f}%': q_lo, f'{hi:.1f}%': q_hi}
                continue
            x = np.asarray(draws.detach().cpu() if hasattr(draws, "detach") else draws)
            table[name] = {
                'mean': float(np.mean(x)), 'std': float(np.std(x)), 'median': float(np.median(x)),
                f'{lo:.1f}%': float(np.percentile(x, lo)), f'{hi:.1f}%': float(np.percentile(x, hi)),
            }
        return table

    def diagnostics(self, ess=True):
        """Per-parameter `mean`, `std`, `rhat`, `ess` (the reference examples' estimator summed over chains) and
        `ess_geyer`, computed on the device from the draws of the last ``run(..., return_torch=True)`` -- nothing but
        the table travels to the host.  (Not in the reference: README.md:212-216 lists R-hat / ESS as planned; the
        ESS definition is examples/06_nuts_comparison.py:22-41.)  Vector parameters give arrays."""
        import torch
        from ..diagnostics import device_summary
        if self.samples is None:
            raise ValueError("Must run sampling first. Call run() method.")
        table = {}
        for name, x in self.samples.items():
            if not (hasattr(x, "is_cuda") and x.is_cuda):
                raise ValueError("diagnostics() works on device draws: call run(..., return_torch=True)")
            if self._single_chain:
                x = x[None]                                   # (S,) | (S, n) -> (1, S[, n])
            d = x.reshape(x.shape[0], x.shape[1], -1).permute(1, 0, 2).contiguous().float()   # [S, C, n]
            cols = device_summary(d, None, ess)
            table[name] = {k: (float(v[0]) if x.dim() == 2 else v.copy()) for k, v in cols.items()}
        return table

    def waic(self):
        """WAIC of the model over the draws of the last ``run`` (numpy or ``return_torch=True``, any number of chains),
        from the pointwise log-likelihood of every observation of the model's observation terms, reduced on the device
        (``diagnostics.waic``).  Not in the reference.  Runs with ``shard='obs'`` are refused: each rank holds only its
        rows of the observations."""
        import torch
        from ..diagnostics import waic
        from ..engine import DeviceModel, compile_model
        if self.samples is None or self._waic_source is None:
            raise ValueError("Must run sampling first. Call run() method.")
        src = self._waic_source
        if src["shard"] == "obs":
            raise ValueError("waic() is not supported for observation-sharded runs (shard='obs')")
        model = src["model"] if isinstance(src["model"], DeviceModel) else compile_model(
            self.log_prob_fn, src["initial_params"], cache=src["cache"], transforms=src["transforms"])
        # the inverse of DeviceModel.unpack: {name: (S,) | (S, n) | (C, S) | (C, S, n)} -> [S, C, D] in model coordinates
        parts = []
        for name, (off, n, shp) in model.layout.items():
            x = torch.as_tensor(self.samples[name]).to(device=model.device, dtype=torch.float32)
            if self._single_chain:
                x = x[None]
            parts.append(x.reshape(x.shape[0], x.shape[1], n))
        draws = torch.cat(parts, dim=2).permute(1, 0, 2).contiguous()
        return waic(model, draws)

    def print_summary(self, credible_interval=0.95):
        table = self.summary(credible_interval)
        ci = f"{int(credible_interval * 100)}% CI"
        print("\nPosterior Summary:")
        print("=" * 80)
        print(f"{'Parameter':<15} {'Mean':<10} {'Std':<10} {'Median':<10} {ci:<20}")
        print("-" * 80)
        for name, row in table.items():
            vals = list(row.values())
            span = f"[{vals[3]:.3f}, {vals[4]:.3f}]"
            print(f"{name:<15} {row['mean']:<10.3f} {row['std']:<10.3f} {row['median']:<10.3f} {span:<20}")
        print("=" * 80)
