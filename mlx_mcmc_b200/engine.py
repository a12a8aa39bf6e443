"""Host-side engine: device model handle + thin launch wrappers around the C ABI.

torch is used for device memory, streams and (in dist.py) torch.distributed -- plumbing only.  Every
number on the sampling path is produced by the kernels in csrc/ through libb200mcmc.so.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import numpy as np
import torch

from . import _cabi
from .tracer import OP_LIN, TracedModel, trace


def _require_cuda() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("mlx_mcmc_b200: no CUDA device visible -- the sampling path runs only on the GPU "
                           "(there is deliberately no CPU fallback)")
    return torch.device("cuda", torch.cuda.current_device())


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class DeviceModel:
    """A traced model resident on one GPU (observed arrays in HBM, term table inside the C handle).

    ``glm_path`` ('auto' | 'simt' | 'tc' | 'tc16') and ``pointwise_path`` ('auto' | 'general') choose the arithmetic /
    evaluation path (b2m_model_options; they were environment variables in ABI 1).  ``transforms``: None (the
    reference: the sampler moves in the model's own coordinates) or 'auto' -- positive / unit-interval parameters,
    recognised from the support of the distribution they are the value of, are sampled in log / logit coordinates.
    ``glm_form`` ('auto' | 'stream' | 'gram') chooses how a GLM-class Normal likelihood is evaluated: two contractions
    over X per evaluation, or one against X^T X precomputed in float64 (DESIGN.md 4.2); ``self.glm_form`` is the form
    in use ('stream' | 'gram', None for pointwise models)."""

    def __init__(self, traced: TracedModel, device: Optional[torch.device] = None, glm_path: str = "auto",
                 pointwise_path: str = "auto", transforms=None, glm_form: str = "auto"):
        self.lib = _cabi.load()
        self.device = device or _require_cuda()
        self.traced = traced
        self.D = traced.D
        self.layout = traced.layout
        if glm_path not in _cabi.GLM_PATHS:
            raise ValueError(f"Unknown glm_path: {glm_path}")
        if glm_form not in _cabi.GLM_FORMS:
            raise ValueError(f"Unknown glm_form: {glm_form}")
        if pointwise_path not in ("auto", "general"):
            raise ValueError(f"Unknown pointwise_path: {pointwise_path}")
        if transforms not in (None, "auto"):
            raise ValueError(f"Unknown transforms option: {transforms}")
        self.tf_codes = traced.transform_codes() if transforms == "auto" else np.zeros(traced.D, dtype=np.int32)
        self.has_transforms = bool(np.any(self.tf_codes != 0))
        # observed arrays: uploaded once, kept alive by this object (the library never owns them)
        self._arrays = [torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(self.device) for a in traced.arrays]
        n_t, n_a, n_l = len(traced.terms), len(traced.arrays), len(traced.lin)
        terms = (_cabi.Term * n_t)()
        for i, t in enumerate(traced.terms):
            terms[i].dist, terms[i].length, terms[i].weight = t.dist, t.length, t.weight
            terms[i].k0, terms[i].k1, terms[i].k2 = t.k
            for slot, o in (("x", t.x), ("p0", t.p0), ("p1", t.p1)):
                dst = getattr(terms[i], slot)
                dst.kind, dst.a, dst.b, dst.c = o.kind, o.a, o.b, o.c
        lin = (_cabi.LinEntry * max(n_l, 1))()
        for i, (p, a, c) in enumerate(traced.lin):
            lin[i].param, lin[i].array, lin[i].coef = p, a, c
        arrays = (_cabi.Array * max(n_a, 1))()
        for i, a in enumerate(self._arrays):
            arrays[i].data = a.data_ptr()
            arrays[i].rows = a.shape[0]
            arrays[i].cols = a.shape[1] if a.dim() == 2 else 1
        handle = C.c_void_p()
        opt = _cabi.ModelOptions()
        opt.glm_path = _cabi.GLM_PATHS[glm_path]
        opt.glm_form = _cabi.GLM_FORMS[glm_form]
        opt.pointwise_path = _cabi.POINTWISE_GENERAL if pointwise_path == "general" else _cabi.POINTWISE_AUTO
        tf_arr = (C.c_int32 * self.D)(*[int(v) for v in self.tf_codes])
        opt.transforms = tf_arr if self.has_transforms else None
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.b2m_model_create(terms, n_t, lin, n_l, arrays, n_a, self.D, C.byref(opt), C.byref(handle)))
        self.handle = handle
        self.jit = False            # set by jit.specialize once a specialised module is attached
        self.model_class = self.lib.b2m_model_class(handle)
        self.glm_path = {0: "simt", 1: "tc", 2: "tc16"}.get(self.lib.b2m_model_glm_path(handle))
        self.glm_form = {1: "stream", 2: "gram"}.get(self.lib.b2m_model_glm_form(handle))

    def __del__(self):
        h, self.handle = getattr(self, "handle", None), None
        if h:
            try:
                self.lib.b2m_model_destroy(h)
            except Exception:
                pass

    # -- parameter packing ----------------------------------------------------------------
    def pack(self, params: Dict[str, object], n_chains: int) -> torch.Tensor:
        """dict of initial values -> theta [n_chains, D] float32 on the device.  A value with a leading
        axis of length n_chains gives per-chain starting points; otherwise every chain starts at it."""
        flat = np.zeros((n_chains, self.D), dtype=np.float32)
        for name, (off, n, shp) in self.layout.items():
            v = np.asarray(params[name], dtype=np.float32)
            if v.shape == tuple(shp):
                flat[:, off:off + n] = v.reshape(1, n)
            elif v.shape == (n_chains,) + tuple(shp):
                flat[:, off:off + n] = v.reshape(n_chains, n)
            else:
                raise ValueError(f"initial value of {name!r} has shape {v.shape}, expected {shp} or ({n_chains},)+{shp}")
        if self.has_transforms:
            flat = self.unconstrain(flat)
        return torch.from_numpy(flat).to(self.device)

    def unconstrain(self, theta: np.ndarray) -> np.ndarray:
        """model coordinates -> the sampler's coordinates (log / logit of the transformed parameters), float32 [.., D]"""
        out = np.array(theta, dtype=np.float64, copy=True)
        pos, unit = self.tf_codes == _cabi.TF_LOG, self.tf_codes == _cabi.TF_LOGIT
        with np.errstate(divide="ignore", invalid="ignore"):
            bad = (out[..., pos] <= 0).any() or (out[..., unit] <= 0).any() or (out[..., unit] >= 1).any()
            if bad:
                raise ValueError("transforms='auto': an initial value lies outside the support of its parameter")
            out[..., pos] = np.log(out[..., pos])
            out[..., unit] = np.log(out[..., unit]) - np.log1p(-out[..., unit])
        return out.astype(np.float32)

    def constrain(self, u: torch.Tensor) -> torch.Tensor:
        """the sampler's coordinates -> model coordinates (device tensor [.., D]); identity without transforms"""
        if not self.has_transforms:
            return u
        codes = torch.from_numpy(self.tf_codes).to(u.device)
        return torch.where(codes == _cabi.TF_LOG, u.exp(), torch.where(codes == _cabi.TF_LOGIT, torch.sigmoid(u), u))

    def unpack(self, draws: torch.Tensor, squeeze_chain: bool, to_numpy: bool = True):
        """draws [S, C, D] -> {name: (S,) | (S, n) | (C, S) | (C, S, n)} in the reference's shapes.

        The chain-major transposition happens on the device (one strided copy per parameter); with ``to_numpy`` each
        result is then copied once into pinned host memory from torch's caching host allocator and returned as the
        numpy view of that buffer -- no host-side transposition or second copy (those dominated the end-to-end time
        of the 1M-chain Metropolis configuration)."""
        out = {}
        staged = []
        for name, (off, n, shp) in self.layout.items():
            part = draws[:, :, off:off + n].permute(1, 0, 2)          # [C, S, n] view
            if not shp:
                part = part[:, :, 0]
            if squeeze_chain:
                part = part[0]
            part = part.contiguous()                                  # device-side transpose
            if to_numpy:
                host = torch.empty(part.shape, dtype=part.dtype, pin_memory=True)
                host.copy_(part, non_blocking=True)
                staged.append((name, host))
            else:
                out[name] = part
        if to_numpy:
            torch.cuda.current_stream().synchronize()
            for name, host in staged:
                out[name] = host.numpy()
        return out

    # -- K1 -------------------------------------------------------------------------------
    def logp_grad(self, theta: torch.Tensor, want_grad: bool = True, lanes: int = 0):
        """log p and gradient for theta [C, D] (device float32).  Parity-check-1 entry point."""
        assert theta.is_cuda and theta.dtype == torch.float32 and theta.dim() == 2 and theta.shape[1] == self.D
        theta = theta.contiguous()
        Cn = theta.shape[0]
        logp = torch.empty(Cn, dtype=torch.float32, device=self.device)
        grad = torch.empty(Cn, self.D, dtype=torch.float32, device=self.device) if want_grad else None
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.b2m_logp_grad(self.handle, _ptr(theta), Cn, _ptr(logp), _ptr(grad), lanes, _stream()))
        return logp, grad


class ChainState:
    """Per-chain sampler state in HBM (positions, step sizes, counters)."""

    def __init__(self, model: DeviceModel, theta: torch.Tensor, step_size: float, chain_offset: int = 0):
        dev = model.device
        self.model = model
        self.n_chains = theta.shape[0]
        self.chain_offset = int(chain_offset)
        self.theta = theta.contiguous()
        self.step_size = torch.full((self.n_chains,), float(step_size), dtype=torch.float64, device=dev)
        self.n_accept = torch.zeros(self.n_chains, dtype=torch.int64, device=dev)
        self.n_total = torch.zeros(self.n_chains, dtype=torch.int64, device=dev)
        self.n_leaves = torch.zeros(self.n_chains, dtype=torch.int64, device=dev)
        self.n_diverge = torch.zeros(self.n_chains, dtype=torch.int64, device=dev)
        self.da_state = torch.zeros(self.n_chains, 3, dtype=torch.float64, device=dev)
        self.logp = torch.full((self.n_chains,), float("nan"), dtype=torch.float32, device=dev)

    def reset_counters(self):
        self.n_accept.zero_()
        self.n_total.zero_()


def launch_hmc(st: ChainState, n_iter: int, n_leapfrog: int, adapt: int, target_accept: float, seed: int,
               iter_offset: int, draws: Optional[torch.Tensor] = None, lanes: int = 0, inj_normal=None,
               inj_uniform=None, trace_energy=None, trace_accept=None, inv_mass=None, draws_unconstrained: bool = False,
               adapt_origin: int = 0):
    m = st.model
    a = _cabi.HmcArgs()
    a.n_chains, a.chain_offset, a.iter_offset = st.n_chains, st.chain_offset, iter_offset
    a.n_iter, a.n_leapfrog, a.adapt, a.lanes = n_iter, n_leapfrog, adapt, lanes
    a.target_accept, a.seed = target_accept, seed & 0xFFFFFFFFFFFFFFFF
    a.theta, a.step_size, a.n_accept, a.n_total = _ptr(st.theta), _ptr(st.step_size), _ptr(st.n_accept), _ptr(st.n_total)
    a.da_state, a.draws = _ptr(st.da_state), _ptr(draws)
    a.inj_normal, a.inj_uniform = _ptr(inj_normal), _ptr(inj_uniform)
    a.trace_energy, a.trace_accept = _ptr(trace_energy), _ptr(trace_accept)
    a.inv_mass, a.draws_unconstrained = _ptr(inv_mass), int(bool(draws_unconstrained))
    a.adapt_origin = int(adapt_origin)
    with torch.cuda.device(m.device):
        _cabi.check(m.lib.b2m_hmc_run(m.handle, C.byref(a), _stream()))


def launch_mh(st: ChainState, n_iter: int, proposal_scale: float, seed: int, iter_offset: int,
              draws: Optional[torch.Tensor] = None, lanes: int = 0, inj_normal=None, inj_uniform=None,
              trace_accept=None):
    m = st.model
    a = _cabi.MhArgs()
    a.n_chains, a.chain_offset, a.iter_offset = st.n_chains, st.chain_offset, iter_offset
    a.n_iter, a.lanes, a.proposal_scale, a.seed = n_iter, lanes, proposal_scale, seed & 0xFFFFFFFFFFFFFFFF
    a.theta, a.logp, a.n_accept, a.draws = _ptr(st.theta), _ptr(st.logp), _ptr(st.n_accept), _ptr(draws)
    a.inj_normal, a.inj_uniform, a.trace_accept = _ptr(inj_normal), _ptr(inj_uniform), _ptr(trace_accept)
    with torch.cuda.device(m.device):
        _cabi.check(m.lib.b2m_mh_run(m.handle, C.byref(a), _stream()))


def launch_nuts(st: ChainState, n_iter: int, max_tree_depth: int, adapt: int, compat: int, target_accept: float,
                seed: int, iter_offset: int, draws=None, depths=None, alphas=None, lanes: int = 0, inj=None,
                trace_doubling=None, trace_energy=None, step_size_jitter: float = 0.0, inv_mass=None,
                schedule: int = 0, slice_state: int = 0, draws_unconstrained: bool = False, adapt_origin: int = 0):
    m = st.model
    inj = inj or {}
    a = _cabi.NutsArgs()
    a.n_chains, a.chain_offset, a.iter_offset = st.n_chains, st.chain_offset, iter_offset
    a.n_iter, a.max_tree_depth, a.adapt, a.compat, a.lanes = n_iter, max_tree_depth, adapt, compat, lanes
    a.target_accept, a.seed = target_accept, seed & 0xFFFFFFFFFFFFFFFF
    a.step_size_jitter = float(step_size_jitter)
    a.theta, a.step_size, a.da_state = _ptr(st.theta), _ptr(st.step_size), _ptr(st.da_state)
    a.n_accept, a.n_leaves, a.n_diverge = _ptr(st.n_accept), _ptr(st.n_leaves), _ptr(st.n_diverge)
    a.draws, a.depths, a.alphas = _ptr(draws), _ptr(depths), _ptr(alphas)
    a.inj_normal, a.inj_slice = _ptr(inj.get("normal")), _ptr(inj.get("slice"))
    a.inj_dir, a.inj_take, a.inj_merge = _ptr(inj.get("dir")), _ptr(inj.get("take")), _ptr(inj.get("merge"))
    a.trace_doubling, a.trace_energy = _ptr(trace_doubling), _ptr(trace_energy)
    a.inv_mass, a.schedule, a.slice_state = _ptr(inv_mass), int(schedule), int(slice_state)
    a.draws_unconstrained = int(bool(draws_unconstrained))
    a.adapt_origin = int(adapt_origin)
    with torch.cuda.device(m.device):
        _cabi.check(m.lib.b2m_nuts_run(m.handle, C.byref(a), _stream()))


# ---------------------------------------------------------------------------------------- model cache
# The reference evaluates the user's log_prob afresh on every call (hmc.py:53-67), so data the function closes over may
# change between run() calls.  Here every compile_model call RE-TRACES the function on the host (cheap: one Python call)
# and the cache is keyed by a fingerprint of what the trace produced -- term table, parameter layout and the contents of
# every observed array -- never by the function object.  Same trace => the resident device model is reused (no
# re-upload of the observations); anything else builds a new one.  Least-recently-used models beyond `_CACHE_SIZE` are
# dropped, so a `make_log_prob(y)` factory pattern cannot pile up device models.
_MODEL_CACHE: "Dict[tuple, DeviceModel]" = {}
_CACHE_SIZE = 4


_FULL_FINGERPRINT_BYTES = 64 << 20


def _array_fingerprint(a: np.ndarray) -> tuple:
    """Content fingerprint of an observed array: 64 position-dependent wrapping sums over its 64-bit words (contiguous
    chunks, one memory-bound pass, no dtype conversion).  Arrays up to 64 MB are summed completely; larger ones (the 400 MB
    design matrix: a full pass would cost a tenth of a sampler call) through 1024 evenly spaced contiguous runs covering a
    sixteenth of the words, plus the first and last megabyte and the buffer address -- new data, re-generated data,
    rescaling and shuffles are all seen, an in-place edit of a handful of elements of a > 64 MB array may not be (pass
    cache=False, or clear_model_cache(), after such an edit)."""
    b = np.ascontiguousarray(a)
    raw = b.view(np.uint8).reshape(-1)
    n8 = raw.size // 8
    w = raw[: n8 * 8].view(np.uint64)
    tail = bytes(raw[n8 * 8:])
    extra = ()
    if raw.size > _FULL_FINGERPRINT_BYTES:
        extra = (int(b.ctypes.data), int(w[: 1 << 17].sum()), int(w[-(1 << 17):].sum()))
        blk = w.size // 1024
        runs = w[: blk * 1024].reshape(1024, blk)[:, : max(blk // 16, 1)].sum(axis=1)      # contiguous runs: no strided gather
        return (b.shape, str(b.dtype), tuple(int(v) for v in runs), extra, tail)
    if w.size == 0:
        return (b.shape, str(b.dtype), tail)
    bounds = np.linspace(0, w.size, 65).astype(np.int64)
    sums = tuple(int(w[bounds[i]:bounds[i + 1]].sum()) for i in range(64))
    return (b.shape, str(b.dtype), sums, extra, tail)


def _trace_fingerprint(traced: TracedModel, extra: tuple) -> tuple:
    terms = tuple((t.dist, t.length, t.weight, t.k, t.x.key(), t.p0.key(), t.p1.key()) for t in traced.terms)
    layout = tuple((k, v) for k, v in traced.layout.items())
    return (traced.D, layout, terms, tuple(traced.lin), tuple(_array_fingerprint(a) for a in traced.arrays), extra)


def clear_model_cache() -> None:
    """Drop every cached device model (their HBM is released when the last reference goes)."""
    _MODEL_CACHE.clear()


def compile_model(log_prob_fn, initial_params, cache: bool = True, glm_path: str = "auto", pointwise_path: str = "auto",
                  transforms=None, glm_form: str = "auto") -> DeviceModel:
    """Trace `log_prob_fn` (always) and return its device model: a cached one when the trace -- terms, layout and the
    contents of the observed arrays -- is identical to one already resident on this device, else a new one.
    ``cache=False`` neither looks up nor stores."""
    dev = _require_cuda()
    traced = trace(log_prob_fn, initial_params)
    key = None
    if cache:
        key = _trace_fingerprint(traced, (dev.index, glm_path, pointwise_path, transforms, glm_form))
        hit = _MODEL_CACHE.pop(key, None)
        if hit is not None:
            _MODEL_CACHE[key] = hit          # most recently used goes last
            return hit
    model = DeviceModel(traced, dev, glm_path=glm_path, pointwise_path=pointwise_path, transforms=transforms,
                        glm_form=glm_form)
    model._fn = log_prob_fn
    if cache:
        _MODEL_CACHE[key] = model
        while len(_MODEL_CACHE) > _CACHE_SIZE:
            _MODEL_CACHE.pop(next(iter(_MODEL_CACHE)))
    return model
