"""Probability distributions (the six classes and export list of mlx_mcmc/distributions/__init__.py, plus Bernoulli)."""
from .base import Distribution
from .normal import Normal
from .halfnormal import HalfNormal
from .beta import Beta
from .gamma import Gamma
from .exponential import Exponential
from .categorical import Categorical
from .bernoulli import Bernoulli

__all__ = ["Distribution", "Normal", "HalfNormal", "Beta", "Gamma", "Exponential", "Categorical", "Bernoulli"]
