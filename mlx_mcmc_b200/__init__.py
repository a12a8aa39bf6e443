"""b200-mcmc: the sampling hot path of korentomas/mlx-mcmc, rebuilt for NVIDIA B200 (sm_100a).

Same public surface as ``mlx_mcmc`` (mlx_mcmc/__init__.py:24-46)::

    import mlx_mcmc_b200.core as mx
    from mlx_mcmc_b200 import Normal, HalfNormal, MCMC

    def log_prob(params):
        return Normal(0, 10).log_prob(params['mu']) + HalfNormal(5).log_prob(params['sigma'])

    samples = MCMC(log_prob).run({'mu': 0.0, 'sigma': 1.0}, num_samples=1000, method='nuts')

``run()`` traces ``log_prob`` once into a term table of library distributions and executes it with
hand-written CUDA kernels through a C ABI (include/b200mcmc.h); there is no CPU or MLX fallback.
"""
from types import SimpleNamespace as _NS

__version__ = "0.1.0"

from . import core
from .distributions import Bernoulli, Beta, Categorical, Distribution, Exponential, Gamma, HalfNormal, Normal
from .inference.mcmc import MCMC
from .kernels.hmc import hmc
from .kernels.metropolis import metropolis_hastings
from .kernels.nuts import nuts
from .tracer import UnsupportedOpError, trace

# namespace object accepted by the model factories in mlx_mcmc_b200.workloads
ns = _NS(mx=core, Normal=Normal, HalfNormal=HalfNormal, Beta=Beta, Gamma=Gamma, Exponential=Exponential,
         Categorical=Categorical, Bernoulli=Bernoulli)

__all__ = ["Normal", "HalfNormal", "Beta", "Gamma", "Exponential", "Categorical", "Bernoulli", "metropolis_hastings", "hmc",
           "nuts", "MCMC", "core", "trace", "UnsupportedOpError", "ns"]
