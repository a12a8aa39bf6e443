"""Trace a user ``log_prob(params)`` once against symbolic parameters into a term table.

The reference differentiates the user's Python function with ``mx.grad`` on every gradient call
(mlx_mcmc/kernels/hmc.py:53-67, nuts.py:76-87), re-running the Python each time.  Here the function
is called ONCE with symbolic parameters; what comes back is a sum of library-distribution terms whose
operands are affine in the parameters with observed-data coefficients:

    log p(theta) = sum_t  w_t * sum_n  logpdf_t( x_t[n] ; p0_t[n], p1_t[n] )

    operand[n] = c  +  sum_e coef_e * data_e[n] * theta[i_e]     (or theta[a+n], or (X @ theta[a:a+d])[n])

which is exactly what the CUDA kernels evaluate with analytic gradients (include/b200mcmc.h).
Anything outside this family raises :class:`UnsupportedOpError` at trace time -- there is no
fallback evaluation path.

Python idioms of the reference's models that are recognised (SURVEY.md section 7 "tracer coverage"):
  * ``mx.sum(Dist(mu, sigma).log_prob(mx.array(data)))``                 examples/02:50
  * ``lp = lp + Dist(...).log_prob(mx.array(y_i))`` unrolled over data    examples/01:46-48, 04:51-53
  * ``mx.sum(mx.array([Dist(...).log_prob(mx.array(y)) for y in ys]))``   tests/test_nuts.py:205-207
  * parameter in the scale slot, constant in the value slot               tests/test_nuts.py:93
  * ``X @ beta`` / ``mx.matmul`` with a vector parameter                  (north-star regression model)
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple, Union

import numpy as np


class UnsupportedOpError(TypeError):
    """The traced log_prob used an operation the B200 term table cannot express."""


# distribution / operand tags: keep in sync with include/b200mcmc.h
NORMAL, HALFNORMAL, EXPONENTIAL, GAMMA, BETA, CONSTANT = range(6)
BERNOULLI = 7   # not 6: b2m_sample's B2M_SAMPLE_CATEGORICAL is 6, and 6 stays an unknown term tag
OP_CONST, OP_PARAM, OP_DATA, OP_PARAMVEC, OP_LIN, OP_MATVEC = range(6)
DIST_NAMES = {NORMAL: "Normal", HALFNORMAL: "HalfNormal", EXPONENTIAL: "Exponential", GAMMA: "Gamma",
              BETA: "Beta", CONSTANT: "const", BERNOULLI: "Bernoulli"}


def _is_number(x) -> bool:
    return isinstance(x, (int, float, np.integer, np.floating)) or (isinstance(x, np.ndarray) and x.ndim == 0)


def _concrete(x):
    """python / numpy value -> float scalar or 1-D/2-D float32 array; None if not concrete."""
    if isinstance(x, Sym):
        return None
    if _is_number(x):
        return float(x)
    if isinstance(x, np.ndarray):
        return x.astype(np.float32, copy=False)
    if isinstance(x, (list, tuple)) and not any(isinstance(e, Sym) for e in x):
        return np.asarray(x, dtype=np.float32)
    return None


class Sym:
    """Base of every traced value.  ``__array_ufunc__ = None`` makes numpy defer to our reflected
    operators instead of trying to broadcast over the symbol."""

    __array_ufunc__ = None
    shape: Tuple[int, ...] = ()

    @property
    def size(self):
        return int(np.prod(self.shape)) if self.shape else 1

    @property
    def ndim(self):
        return len(self.shape)

    def _concretise(self, what):
        raise UnsupportedOpError(
            f"unsupported op: {what} needs the concrete value of a traced parameter "
            "(data-dependent Python control flow cannot be traced; examples/05_categorical_model.py does this)")

    def __float__(self):
        self._concretise("float()")

    def __int__(self):
        self._concretise("int()")

    def __bool__(self):
        self._concretise("bool() / if / comparison result")

    def __len__(self):
        if not self.shape:
            raise TypeError("len() of a traced scalar")
        return self.shape[0]

    def item(self):
        self._concretise(".item()")

    def tolist(self):
        self._concretise(".tolist()")


# --------------------------------------------------------------------------------------
# affine expressions in the parameters
@dataclass(frozen=True)
class Atom:
    kind: str      # 'elem' theta[i] | 'vec' theta[a:a+n] elementwise | 'matvec' X @ theta[a:a+n]
    a: int
    n: int = 1
    array: int = -1  # matvec: id of the [N, n] matrix


@dataclass(frozen=True)
class Coef:
    scale: float = 1.0
    array: int = -1  # id of a 1-D data vector multiplying elementwise, or -1

    def times(self, other: "Coef", ctx) -> "Coef":
        if self.array >= 0 and other.array >= 0:
            prod = ctx.arrays[self.array] * ctx.arrays[other.array]
            return Coef(self.scale * other.scale, ctx.add_array(prod))
        return Coef(self.scale * other.scale, max(self.array, other.array))


class Lin(Sym):
    """c + sum_e coef_e * atom_e  with shape () or (N,)."""

    def __init__(self, ctx, shape, const: List[Coef], entries: List[Tuple[Coef, Atom]]):
        self.ctx, self.shape = ctx, tuple(shape)
        self.const = [c for c in const if c.scale != 0.0]
        self.entries = [(c, a) for c, a in entries if c.scale != 0.0]

    # -- construction helpers
    @staticmethod
    def lift(ctx, x) -> "Lin":
        if isinstance(x, Lin):
            return x
        if isinstance(x, Sym):
            raise UnsupportedOpError(f"unsupported op: arithmetic on a {type(x).__name__} value "
                                     "(log-probabilities can only be added, scaled and summed)")
        c = _concrete(x)
        if c is None:
            raise UnsupportedOpError(f"unsupported operand type {type(x).__name__}")
        if isinstance(c, float):
            return Lin(ctx, (), [Coef(c)], [])
        if c.ndim != 1:
            raise UnsupportedOpError("only scalars and 1-D observed arrays may be combined with traced values")
        return Lin(ctx, c.shape, [Coef(1.0, ctx.add_array(c))], [])

    def _shape_with(self, o: "Lin"):
        if self.shape == o.shape or not o.shape:
            return self.shape
        if not self.shape:
            return o.shape
        raise UnsupportedOpError(f"shape mismatch {self.shape} vs {o.shape}")

    def is_constant(self):
        return not self.entries

    # -- linear algebra over the symbols
    def __add__(self, o):
        if isinstance(o, LogProb):
            return o.__radd__(self)
        o = Lin.lift(self.ctx, o)
        return Lin(self.ctx, self._shape_with(o), self.const + o.const, self.entries + o.entries)

    __radd__ = __add__

    def __neg__(self):
        return self._scaled(Coef(-1.0))

    def __sub__(self, o):
        return self + (-Lin.lift(self.ctx, o))

    def __rsub__(self, o):
        return Lin.lift(self.ctx, o) + (-self)

    def _scaled(self, k: Coef, shape=None):
        return Lin(self.ctx, self.shape if shape is None else shape,
                   [c.times(k, self.ctx) for c in self.const],
                   [(c.times(k, self.ctx), a) for c, a in self.entries])

    def __mul__(self, o):
        o = Lin.lift(self.ctx, o)
        if o.is_constant():
            lin, k = self, o
        elif self.is_constant():
            lin, k = o, self
        else:
            raise UnsupportedOpError("unsupported op: product of two traced values (only affine operands "
                                     "are lowered; put the nonlinearity inside a distribution)")
        shape = lin._shape_with(k)
        out = Lin(self.ctx, shape, [], [])
        for kc in (k.const or [Coef(0.0)]):
            part = lin._scaled(kc, shape)
            out = Lin(self.ctx, shape, out.const + part.const, out.entries + part.entries)
        return out

    __rmul__ = __mul__

    def __truediv__(self, o):
        c = _concrete(o)
        if c is None:
            raise UnsupportedOpError("unsupported op: division by a traced value")
        return self * (1.0 / c if isinstance(c, float) else (1.0 / c).astype(np.float32))

    def __rtruediv__(self, o):
        raise UnsupportedOpError("unsupported op: division by a traced value")

    def __pow__(self, o):
        if _is_number(o) and float(o) == 1.0:
            return self
        raise UnsupportedOpError("unsupported op: power of a traced value outside a distribution")

    def __matmul__(self, o):
        raise UnsupportedOpError("unsupported op: traced @ value (only observed_matrix @ vector_parameter)")

    def __rmatmul__(self, X):
        X = _concrete(X)
        if X is None or isinstance(X, float) or X.ndim != 2:
            raise UnsupportedOpError("unsupported op: matmul needs a concrete 2-D observed matrix on the left")
        if not (len(self.entries) == 1 and not self.const and self.entries[0][1].kind == "vec"
                and self.entries[0][0] == Coef(1.0)):
            raise UnsupportedOpError("unsupported op: matmul right operand must be a plain vector parameter")
        atom = self.entries[0][1]
        if X.shape[1] != atom.n:
            raise UnsupportedOpError(f"matmul shape mismatch {X.shape} @ ({atom.n},)")
        mid = self.ctx.add_array(X)
        return Lin(self.ctx, (X.shape[0],), [], [(Coef(1.0), Atom("matvec", atom.a, atom.n, mid))])

    def __getitem__(self, idx):
        if len(self.entries) == 1 and not self.const and self.entries[0][1].kind == "vec" \
                and self.entries[0][0] == Coef(1.0) and isinstance(idx, (int, np.integer)):
            atom = self.entries[0][1]
            i = int(idx) + (atom.n if idx < 0 else 0)
            if not 0 <= i < atom.n:
                raise IndexError(idx)
            return Lin(self.ctx, (), [], [(Coef(1.0), Atom("elem", atom.a + i))])
        raise UnsupportedOpError("unsupported op: indexing a traced value (only vector_param[int])")

    def _cmp(self, *_):
        raise UnsupportedOpError("unsupported op: comparison on a traced value outside a distribution "
                                 "(support masks live inside the library distributions)")

    __lt__ = __le__ = __gt__ = __ge__ = _cmp

    def __repr__(self):
        return f"Lin(shape={self.shape}, const={self.const}, entries={self.entries})"


# --------------------------------------------------------------------------------------
# log-probability values
@dataclass
class Operand:
    kind: int
    a: int = 0
    b: int = 0
    c: float = 0.0
    lin: Tuple[Tuple[int, int, float], ...] = ()   # (param, array, coef) for OP_LIN

    def key(self):
        return (self.kind, self.a, self.b, self.c, self.lin)


@dataclass
class Term:
    dist: int
    length: int
    x: Operand
    p0: Operand
    p1: Operand
    k: Tuple[float, float, float] = (0.0, 0.0, 0.0)
    weight: float = 1.0
    natural_shape: Tuple[int, ...] = ()   # () scalar term, (N,) elementwise term not yet summed


@dataclass
class Part:
    """Terms sharing one natural shape.  `const` is a scalar addend when shape == (), or the already
    summed total of a constant vector when shape == (N,)."""
    terms: List[Term]
    shape: Tuple[int, ...]
    const: float = 0.0


class LogProb(Sym):
    """A (possibly not yet reduced) sum of log-density terms plus constants."""

    def __init__(self, ctx, parts: List[Part]):
        self.ctx, self.parts = ctx, parts
        shapes = {p.shape for p in parts if p.shape}
        if len(shapes) > 1:
            raise UnsupportedOpError(f"shape mismatch between log-probability terms: {sorted(shapes)}")
        self.shape = shapes.pop() if shapes else ()

    @property
    def terms(self):
        return [t for p in self.parts for t in p.terms]

    @property
    def const(self):
        return sum(p.const for p in self.parts)

    def _coerce(self, o) -> "LogProb":
        if isinstance(o, LogProb):
            return o
        if isinstance(o, Lin):
            if o.is_constant() and all(c.array < 0 for c in o.const):
                return LogProb(self.ctx, [Part([], (), sum(c.scale for c in o.const))])
            raise UnsupportedOpError("unsupported op: adding a raw traced parameter expression to a log-probability "
                                     "(express it through a library distribution)")
        c = _concrete(o)
        if isinstance(c, float):
            return LogProb(self.ctx, [Part([], (), c)])
        if isinstance(c, np.ndarray) and c.ndim <= 1:
            if c.ndim == 0 or c.shape[0] == 1:
                return LogProb(self.ctx, [Part([], (), float(c.reshape(-1)[0]))])
            return LogProb(self.ctx, [Part([], c.shape, float(np.sum(c.astype(np.float64))))])
        raise UnsupportedOpError(f"unsupported op: log-probability + {type(o).__name__}")

    def __add__(self, o):
        return LogProb(self.ctx, self.parts + self._coerce(o).parts)

    __radd__ = __add__

    def __neg__(self):
        return self * -1.0

    def __sub__(self, o):
        return self + (-self._coerce(o))

    def __rsub__(self, o):
        return self._coerce(o) + (-self)

    def __mul__(self, k):
        if not _is_number(k):
            raise UnsupportedOpError("unsupported op: a log-probability may only be scaled by a python number")
        k = float(k)
        return LogProb(self.ctx, [
            Part([Term(t.dist, t.length, t.x, t.p0, t.p1, t.k, t.weight * k, t.natural_shape) for t in p.terms],
                 p.shape, p.const * k) for p in self.parts])

    __rmul__ = __mul__

    def __truediv__(self, k):
        if not _is_number(k):
            raise UnsupportedOpError("unsupported op: a log-probability may only be divided by a python number")
        return self * (1.0 / float(k))

    def total(self) -> "LogProb":
        """mx.sum: reduce to a scalar.  Scalar parts broadcast into a vector count once per element."""
        n = self.shape[0] if self.shape else 1
        terms, const = [], 0.0
        for p in self.parts:
            rep = float(n) if (self.shape and not p.shape) else 1.0
            const += p.const * rep
            for t in p.terms:
                terms.append(Term(t.dist, t.length, t.x, t.p0, t.p1, t.k, t.weight * rep, ()))
        return LogProb(self.ctx, [Part(terms, (), const)])

    def __getitem__(self, idx):
        raise UnsupportedOpError("unsupported op: indexing a traced log-probability")

    def _cmp(self, *_):
        raise UnsupportedOpError("unsupported op: comparison on a traced log-probability")

    __lt__ = __le__ = __gt__ = __ge__ = _cmp


class LogProbStack(Sym):
    """``mx.array([lp_1, ..., lp_K])`` of traced scalar log-probabilities (tests/test_nuts.py:205-207)."""

    def __init__(self, ctx, items: Sequence[LogProb]):
        self.ctx, self.items, self.shape = ctx, list(items), (len(items),)

    def total(self) -> LogProb:
        out = LogProb(self.ctx, [])
        for it in self.items:
            out = out + it.total()
        return out.total()


# --------------------------------------------------------------------------------------
class TraceContext:
    """Owns the observed-array table and the parameter layout of one trace."""

    def __init__(self, param_shapes: Dict[str, Tuple[int, ...]]):
        self.arrays: List[np.ndarray] = []
        self._array_ids: Dict[tuple, int] = {}
        self.layout: Dict[str, Tuple[int, int, Tuple[int, ...]]] = {}
        off = 0
        for name, shp in param_shapes.items():
            n = int(np.prod(shp)) if shp else 1
            if len(shp) > 1:
                raise UnsupportedOpError(f"parameter {name!r}: only scalar and 1-D parameters are supported")
            self.layout[name] = (off, n, tuple(shp))
            off += n
        self.D = off

    def add_array(self, a: np.ndarray) -> int:
        a = np.ascontiguousarray(a, dtype=np.float32)
        key = (a.shape, a.tobytes() if a.size <= 4096 else (id(a), a.ctypes.data, float(a.reshape(-1)[0])))
        if key in self._array_ids:
            return self._array_ids[key]
        self.arrays.append(a)
        self._array_ids[key] = len(self.arrays) - 1
        return len(self.arrays) - 1

    def symbols(self) -> Dict[str, Lin]:
        out = {}
        for name, (off, n, shp) in self.layout.items():
            atom = Atom("elem", off) if not shp else Atom("vec", off, n)
            out[name] = Lin(self, shp, [], [(Coef(1.0), atom)])
        return out

    # -- operand lowering
    def operand(self, v, length: int) -> Operand:
        if isinstance(v, LogProb) or isinstance(v, LogProbStack):
            raise UnsupportedOpError("unsupported op: a log-probability used as a distribution argument")
        if not isinstance(v, Lin):
            c = _concrete(v)
            if c is None:
                raise UnsupportedOpError(f"unsupported distribution argument of type {type(v).__name__}")
            if isinstance(c, float):
                return Operand(OP_CONST, c=c)
            if c.ndim == 0 or c.size == 1:
                return Operand(OP_CONST, c=float(c.reshape(-1)[0]))
            if c.ndim != 1:
                raise UnsupportedOpError("distribution arguments must be scalars or 1-D arrays")
            if c.shape[0] != length:
                raise UnsupportedOpError(f"cannot broadcast an observed array of length {c.shape[0]} against a term of "
                                         f"length {length}")
            return Operand(OP_DATA, a=self.add_array(c))
        const_scalar = sum(c.scale for c in v.const if c.array < 0)
        const_arrays = [c for c in v.const if c.array >= 0]
        if not v.entries:
            if not const_arrays:
                return Operand(OP_CONST, c=const_scalar)
            if len(const_arrays) == 1 and const_scalar == 0.0 and const_arrays[0].scale == 1.0:
                return Operand(OP_DATA, a=const_arrays[0].array)
        if len(v.entries) == 1 and not const_arrays:
            coef, atom = v.entries[0]
            if coef == Coef(1.0):
                if atom.kind == "elem" and const_scalar == 0.0:
                    return Operand(OP_PARAM, a=atom.a)
                if atom.kind == "vec" and const_scalar == 0.0:
                    return Operand(OP_PARAMVEC, a=atom.a, b=atom.n)
                if atom.kind == "matvec":
                    return Operand(OP_MATVEC, a=atom.array, b=atom.a, c=const_scalar)
        lin = []
        for c in const_arrays:
            lin.append((-1, c.array, c.scale))
        for coef, atom in v.entries:
            if atom.kind != "elem":
                raise UnsupportedOpError("unsupported op: a vector parameter or X @ beta combined with other traced "
                                         "terms inside one distribution argument")
            lin.append((atom.a, coef.array, coef.scale))
        return Operand(OP_LIN, c=const_scalar, lin=tuple(lin))

    def log_density(self, dist: int, value, p0=None, p1=None, k=(0.0, 0.0, 0.0)) -> LogProb:
        """Called by the distribution classes when any argument is traced."""
        # python lists / tuples are data like numpy arrays (the reference does `value = mx.array(value)`)
        value, p0, p1 = (np.asarray(v, dtype=np.float32) if isinstance(v, (list, tuple)) and _concrete(v) is not None else v
                         for v in (value, p0, p1))
        length = 1
        for v in (value, p0, p1):
            if v is None:
                continue
            shp = v.shape if isinstance(v, (Sym, np.ndarray)) else ()
            if len(shp) > 1:
                raise UnsupportedOpError("distribution arguments must be scalars or 1-D")
            n = shp[0] if shp else 1
            if n != 1 and length != 1 and n != length:
                raise UnsupportedOpError(f"cannot broadcast distribution arguments of lengths {length} and {n}")
            length = max(length, n)
        ox = self.operand(value, length)
        o0 = self.operand(p0, length) if p0 is not None else Operand(OP_CONST)
        o1 = self.operand(p1, length) if p1 is not None else Operand(OP_CONST)
        shape = (length,) if length > 1 else ()
        for o in (ox, o0, o1):      # a length-1 array argument was folded to a constant above
            if o.kind == OP_PARAMVEC and o.b != length:
                raise UnsupportedOpError("vector parameter length does not match the other arguments")
        if OP_MATVEC in (o0.kind, o1.kind) and ox.kind == OP_CONST:
            # a single observation next to X @ beta: the contraction kernels read y from an observed array
            ox = Operand(OP_DATA, a=self.add_array(np.full(length, ox.c, dtype=np.float32)))
        t = Term(dist, length, ox, o0, o1, tuple(float(v) for v in k), 1.0, shape)
        return LogProb(self, [Part([t], shape)])


_ACTIVE: List[TraceContext] = []


def active_context() -> Optional[TraceContext]:
    return _ACTIVE[-1] if _ACTIVE else None


# --------------------------------------------------------------------------------------
@dataclass
class TracedModel:
    """Result of a trace: everything b2m_model_create needs, still on the host."""

    D: int
    layout: Dict[str, Tuple[int, int, Tuple[int, ...]]]
    terms: List[Term]
    arrays: List[np.ndarray]
    lin: List[Tuple[int, int, float]] = field(default_factory=list)

    @property
    def is_glm(self):
        return any(o.kind == OP_MATVEC for t in self.terms for o in (t.x, t.p0, t.p1))

    def transform_codes(self) -> np.ndarray:
        """Per flat parameter index: 0 none, 1 log, 2 logit (include/b200mcmc.h B2M_TF_*), chosen from the support of
        the library distribution the parameter is the VALUE of: HalfNormal / Exponential / Gamma => positive => log;
        Beta => unit interval => logit.  A parameter claimed by both kinds keeps its own coordinate."""
        want = {HALFNORMAL: 1, EXPONENTIAL: 1, GAMMA: 1, BETA: 2}
        codes = np.zeros(self.D, dtype=np.int32)
        clash = np.zeros(self.D, dtype=bool)
        for t in self.terms:
            code = want.get(t.dist)
            if code is None:
                continue
            if t.x.kind == OP_PARAM:
                idx = [t.x.a]
            elif t.x.kind == OP_PARAMVEC:
                idx = range(t.x.a, t.x.a + t.length)
            else:
                continue
            for i in idx:
                if codes[i] not in (0, code):
                    clash[i] = True
                codes[i] = code
        codes[clash] = 0
        return codes

    @staticmethod
    def _involves_param(o: Operand) -> bool:
        if o.kind in (OP_PARAM, OP_PARAMVEC, OP_MATVEC):
            return True
        return o.kind == OP_LIN and any(p >= 0 for p, _, _ in o.lin)

    def observation_terms(self) -> List[int]:
        """Indices of the observation terms, in term order: the value operand involves no parameter (a constant, data,
        or an affine expression of data) and p0 or p1 does.  Every element of such a term is one observation, numbered
        in term order and by element within a term -- the columns of the pointwise log-likelihood that WAIC is
        computed from (diagnostics.waic, b2m_loglik_stats, which checks this choice).  Constant terms never count."""
        return [i for i, t in enumerate(self.terms)
                if t.dist != CONSTANT and not self._involves_param(t.x)
                and (self._involves_param(t.p0) or self._involves_param(t.p1))]

    def describe(self) -> str:
        rows = []
        for t in self.terms:
            rows.append(f"{t.weight:+g} * sum_{t.length} {DIST_NAMES[t.dist]}(x={t.x.key()[:4]}, p0={t.p0.key()[:4]}, "
                        f"p1={t.p1.key()[:4]}, k={t.k})")
        return "\n".join(rows)


def _merge_unrolled(terms: List[Term], ctx: TraceContext) -> List[Term]:
    """Fold runs of scalar terms that differ only in a constant value operand (a Python loop over the
    observations, examples/01:46-48) into one vector term over a new observation array."""
    groups: Dict[tuple, List[Term]] = {}
    order: List[tuple] = []
    for t in terms:
        if t.length == 1 and t.x.kind == OP_CONST and t.dist != CONSTANT and \
                (t.p0.kind != OP_CONST or t.p1.kind != OP_CONST):
            key = ("m", t.dist, t.p0.key(), t.p1.key(), t.k, t.weight)
        else:
            key = ("u", id(t))
        if key not in groups:
            groups[key] = []
            order.append(key)
        groups[key].append(t)
    out = []
    for key in order:
        g = groups[key]
        if key[0] == "u" or len(g) == 1:
            out.extend(g)
            continue
        data = np.asarray([t.x.c for t in g], dtype=np.float32)
        aid = ctx.add_array(data)
        t0 = g[0]
        out.append(Term(t0.dist, len(g), Operand(OP_DATA, a=aid), t0.p0, t0.p1, t0.k, t0.weight, ()))
    return out


def trace(log_prob_fn, initial_params: Dict[str, object]) -> TracedModel:
    """Call `log_prob_fn` once with symbolic parameters and lower the result to a term table."""
    shapes = {}
    for name, v in initial_params.items():
        a = np.asarray(v)
        if a.dtype.kind not in "fiu":
            raise TypeError(f"initial value of {name!r} must be numeric")
        shapes[name] = tuple(a.shape)
    ctx = TraceContext(shapes)
    _ACTIVE.append(ctx)
    try:
        out = log_prob_fn(ctx.symbols())
    finally:
        _ACTIVE.pop()
    if isinstance(out, LogProbStack):
        raise UnsupportedOpError("log_prob must return a scalar (did you forget mx.sum?)")
    if not isinstance(out, LogProb):
        if isinstance(out, Lin):
            raise UnsupportedOpError("unsupported op: log_prob returned a raw expression of the parameters; only sums of "
                                     "library-distribution log_prob terms are lowered to CUDA")
        raise UnsupportedOpError("log_prob does not depend on the parameters through any library distribution")
    if out.shape:
        raise UnsupportedOpError("log_prob must return a scalar (did you forget mx.sum?)")
    out = out.total()
    terms = [t for t in out.terms if t.weight != 0.0 and t.length > 0]
    if out.const != 0.0:
        terms.append(Term(CONSTANT, 1, Operand(OP_CONST), Operand(OP_CONST), Operand(OP_CONST), (out.const, 0.0, 0.0)))
    terms = _merge_unrolled(terms, ctx)
    if not terms:
        raise UnsupportedOpError("log_prob has no terms")
    # flatten OP_LIN entry lists into one table
    lin: List[Tuple[int, int, float]] = []
    for t in terms:
        for o in (t.x, t.p0, t.p1):
            if o.kind == OP_LIN:
                o.a, o.b = len(lin), len(o.lin)
                lin.extend(o.lin)
    return TracedModel(ctx.D, ctx.layout, terms, ctx.arrays, lin)
