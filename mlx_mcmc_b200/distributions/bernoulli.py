"""Bernoulli distribution over labels in {0, 1} (no reference counterpart; the binary-outcome likelihood of logistic
regression)."""
from __future__ import annotations

import numpy as np

from .. import core as mx
from ..tracer import BERNOULLI, Sym, UnsupportedOpError
from .base import Distribution, context, f32, require_concrete, traced


def _has_sym(v) -> bool:
    return isinstance(v, Sym) or (isinstance(v, (list, tuple)) and any(isinstance(e, Sym) for e in v))


class Bernoulli(Distribution):
    """Bernoulli from `probs` (probability of 1) or `logits` (log-odds); exactly one of the two, as for Categorical.

        log p(y) = y logits - softplus(logits) = y log p + (1 - y) log(1 - p)      for y in {0, 1}, -inf otherwise

    `logits` may be traced -- a constant, a scalar parameter, a vector parameter, an affine expression, or
    ``X @ beta (+ c)``, which makes the model a logistic regression on the GLM (tensor-core) path.  Traced `probs`
    are not lowered, and the value must be observed data."""

    def __init__(self, probs=None, logits=None):
        if probs is None and logits is None:
            raise ValueError("Either probs or logits must be specified")
        if probs is not None and logits is not None:
            raise ValueError("Only one of probs or logits can be specified")
        self._from_probs = probs is not None
        if _has_sym(probs):
            raise UnsupportedOpError("unsupported op: Bernoulli with traced probs (write the model with logits=, "
                                     "e.g. Bernoulli(logits=X @ beta))")
        if logits is not None and traced(logits):
            self.logits, self.probs = logits, None
        elif _has_sym(logits):
            raise UnsupportedOpError("unsupported op: Bernoulli logits given as a list of traced values "
                                     "(use one traced expression, e.g. a + b * x or X @ beta)")
        elif probs is not None:
            self.probs = f32(probs)
            with np.errstate(divide="ignore"):
                self.logits = (np.log(self.probs) - np.log1p(-self.probs)).astype(np.float32)
        else:
            self.logits = f32(logits)
            with np.errstate(over="ignore"):
                self.probs = (1.0 / (1.0 + np.exp(-self.logits))).astype(np.float32)

    def log_prob(self, value):
        if isinstance(value, Sym):
            raise UnsupportedOpError("unsupported op: Bernoulli.log_prob of a traced value (the labels must be "
                                     "observed data)")
        if traced(self.logits):
            return context().log_density(BERNOULLI, value, self.logits)
        y = f32(value)
        ok = (y == 0) | (y == 1)
        one = y == 1
        with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
            if self._from_probs:
                lp = np.where(one, np.log(self.probs), np.log1p(-self.probs))
            else:
                # y l - softplus(l) = (0 if the label agrees with the sign of l else -|l|) - log1p(exp(-|l|)):
                # no overflow and no cancellation at any |l|
                t = self.logits
                match = one == (t >= 0)
                lp = np.where(match, np.float32(0.0), -np.abs(t)) - np.log1p(np.exp(-np.abs(t)))
        return np.where(ok, lp, np.float32(-np.inf)).astype(np.float32)

    def _device_sample_spec(self):
        require_concrete("Bernoulli logits", self.logits)
        if np.size(self.probs) != 1:
            raise ValueError("sample_device needs a scalar Bernoulli probability")
        return BERNOULLI, float(np.reshape(self.probs, -1)[0]), 0.0, None

    def sample(self, key, shape=()):
        if self.probs is None:
            require_concrete("Bernoulli logits", self.logits)
        u = mx.random.uniform(shape=shape, key=key)
        return (np.asarray(u) < self.probs).astype(np.float32)

    def mean(self):
        return self.probs

    def variance(self):
        return self.probs * (1 - self.probs)

    def __repr__(self):
        if self.probs is None:
            return "Bernoulli(<traced logits>)"
        if np.ndim(self.probs) == 0:
            return f"Bernoulli(probs={float(self.probs):.3f})"
        return f"Bernoulli(shape={np.shape(self.probs)})"
