"""Multi-GPU plumbing (SURVEY.md 8e): one process per GPU under ``torchrun``; ``torch.distributed`` carries the
small control messages and the final gather, the data path stays inside libb200mcmc.so.

Two ways to partition a run over the ranks of one box:

* **chain sharding** -- rank g owns global chains ``[offset_g, offset_g + count_g)``.  Chains are independent and
  the Philox streams are keyed by the *global* chain id, so a chain's draws do not depend on the number of ranks.
  No data-path collective; one gather of draws / diagnostics at the end (`gather_draws`).
* **observation sharding** (GLM-class models, the 100K-observation regression) -- every rank holds every chain and a
  row shard of (X, y); each value+gradient sums the ``[C, D]`` gradient partial and the ``[C]`` sum of squared
  residuals over ranks with one NCCL all-reduce on the compute stream (`ObsComm`, csrc/comm.cu).  All ranks then
  hold identical results and take identical accept / U-turn decisions.  With ``slice_state=True`` (NUTS sampling
  phase) the per-chain work is sliced too: rank r finishes and advances chains ``[r C/G, (r+1) C/G)`` only; the
  all-reduce becomes a reduce-scatter and the new leaf positions are all-gathered (csrc/glm_samplers.cu,
  `glm_nuts_run_async`), which removes the replicated per-chain kernels from every rank's critical path.

The reference is single device, single chain (README.md:33-36,212-213): nothing here has a counterpart there.
"""
from __future__ import annotations

import copy
import ctypes as C
import os
from typing import Dict, Optional, Tuple

import numpy as np
import torch
import torch.distributed as td

from .tracer import NORMAL, OP_DATA, OP_MATVEC, TracedModel


# ------------------------------------------------------------------------------------------ partitions
def rank_world(group=None) -> Tuple[int, int]:
    """(rank, world size) of the initialised process group, or (0, 1) in a single process."""
    if td.is_available() and td.is_initialized():
        return td.get_rank(group), td.get_world_size(group)
    return 0, 1


def shard_chains(num_chains: int, rank: int, world: int) -> Tuple[int, int]:
    """(count, offset) of the contiguous block of global chain ids owned by `rank`; the remainder goes to the
    low ranks, so counts differ by at most one and the blocks tile [0, num_chains) in rank order."""
    if num_chains < 0 or world < 1 or not 0 <= rank < world:
        raise ValueError(f"bad partition request: num_chains={num_chains}, rank={rank}, world={world}")
    base, rem = divmod(num_chains, world)
    count = base + (1 if rank < rem else 0)
    offset = rank * base + min(rank, rem)
    return count, offset


def shard_rows(n_rows: int, rank: int, world: int, multiple: int = 1) -> Tuple[int, int]:
    """[r0, r1) of the observation rows owned by `rank`.  Boundaries are rounded to `multiple` rows (except the
    last) so every shard but the last keeps a tile-aligned length."""
    if n_rows < 0 or world < 1 or not 0 <= rank < world:
        raise ValueError(f"bad partition request: n_rows={n_rows}, rank={rank}, world={world}")
    per = -(-n_rows // world)
    per = -(-per // multiple) * multiple
    r0, r1 = min(rank * per, n_rows), min((rank + 1) * per, n_rows)
    return r0, r1


def shard_observations(traced: TracedModel, rank: int, world: int) -> TracedModel:
    """Row-shard the GLM likelihood of a traced model: the rank keeps rows [r0, r1) of X and y and the likelihood
    term's length becomes r1 - r0; priors are untouched (they are added once, after the all-reduce, on every
    rank).  Pure host logic -- no device needed."""
    if world == 1:
        return traced
    if not traced.is_glm:
        raise ValueError("observation sharding needs a GLM-class model (a Normal likelihood over X @ beta); "
                         "use chain sharding for pointwise models")
    out = copy.copy(traced)
    out.terms = [copy.copy(t) for t in traced.terms]
    out.arrays = list(traced.arrays)
    lik = [i for i, t in enumerate(out.terms) if any(o.kind == OP_MATVEC for o in (t.x, t.p0, t.p1))]
    if len(lik) != 1:
        raise ValueError("observation sharding supports exactly one X @ beta term")
    t = out.terms[lik[0]]
    if t.dist != NORMAL:
        raise ValueError("observation sharding supports the Normal likelihood of the GLM class only; shard the chains "
                         "(shard='chains') of a Bernoulli (logistic) model instead")
    if t.p0.kind != OP_MATVEC or t.x.kind != OP_DATA:
        raise ValueError("observation sharding needs the form Normal(X @ beta, sigma).log_prob(y)")
    xi, yi = t.p0.a, t.x.a
    for j, other in enumerate(out.terms):
        if j == lik[0]:
            continue
        for o in (other.x, other.p0, other.p1):
            if o.kind in (OP_DATA, OP_MATVEC) and o.a in (xi, yi):
                raise ValueError("observation sharding: X / y are also used by another term")
            if any(arr in (xi, yi) for (_, arr, _) in o.lin):
                raise ValueError("observation sharding: X / y are also used by another term")
    r0, r1 = shard_rows(t.length, rank, world)
    if r1 <= r0:
        raise ValueError(f"rank {rank} of {world} would own no observation rows (N = {t.length})")
    out.arrays[xi] = np.ascontiguousarray(traced.arrays[xi][r0:r1])
    out.arrays[yi] = np.ascontiguousarray(traced.arrays[yi][r0:r1])
    t.length = r1 - r0
    return out


# ------------------------------------------------------------------------------------------ final gather
def gather_draws(samples: Dict[str, object], num_chains_local: int, group=None, squeeze_single: bool = False):
    """Concatenate per-rank draws along the chain axis, in rank order, on every rank.

    `samples[name]` has a leading chain axis of length `num_chains_local` (numpy array or torch tensor, CPU or
    CUDA -- CUDA tensors need an NCCL group, CPU data a gloo group).  Ranks may own different chain counts.
    Returns the same container type as the input."""
    rank, world = rank_world(group)
    if world == 1:
        return samples
    out = {}
    for name, v in samples.items():
        as_numpy = isinstance(v, np.ndarray)
        t = torch.from_numpy(np.ascontiguousarray(v)) if as_numpy else v.contiguous()
        if t.shape[0] != num_chains_local:
            raise ValueError(f"{name}: leading axis {t.shape[0]} is not the local chain count {num_chains_local}")
        home = t.device
        if td.get_backend(group) == "nccl" and not t.is_cuda:
            t = t.cuda()                       # NCCL moves device memory only
        counts = [torch.zeros(1, dtype=torch.int64, device=t.device) for _ in range(world)]
        td.all_gather(counts, torch.tensor([t.shape[0]], dtype=torch.int64, device=t.device), group=group)
        counts = [int(c.item()) for c in counts]
        cmax = max(counts)
        pad = torch.zeros((cmax,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        pad[: t.shape[0]] = t
        parts = [torch.empty_like(pad) for _ in range(world)]
        td.all_gather(parts, pad, group=group)
        full = torch.cat([p[:n] for p, n in zip(parts, counts)], dim=0).to(home)
        out[name] = full.numpy() if as_numpy else full
    return out


def reduce_stats(values: Dict[str, float], op: str = "sum", group=None, device: Optional[torch.device] = None):
    """All-reduce a small dict of python numbers (accept counts, gradient-evaluation counts, timings)."""
    rank, world = rank_world(group)
    if world == 1:
        return dict(values)
    keys = sorted(values)
    t = torch.tensor([float(values[k]) for k in keys], dtype=torch.float64, device=device or "cpu")
    td.all_reduce(t, op={"sum": td.ReduceOp.SUM, "max": td.ReduceOp.MAX, "min": td.ReduceOp.MIN}[op], group=group)
    return {k: float(x) for k, x in zip(keys, t.tolist())}


def merge_slices(zero_based, accumulators=(), group=None) -> None:
    """Merge per-chain outputs of a sliced observation-sharded call, in place, on every rank.

    `zero_based`: tensors that were zero before the call and that only the owning rank wrote (draws, depths, accept
    counts) -- summed over ranks.  `accumulators`: pairs ``(tensor, value_before_the_call)`` of running per-chain counters
    that every rank held identically before the call and only the owner advanced -- the increments are summed."""
    if rank_world(group)[1] == 1:
        return
    for t, before in accumulators:
        inc = t - before
        td.all_reduce(inc, group=group)
        t.copy_(before + inc)
    for t in zero_based:
        td.all_reduce(t, group=group)


# ------------------------------------------------------------------------------------------ observation sharding
class ObsComm:
    """The library-side communicator for observation sharding.  Rank 0 asks the library for a 128-byte NCCL id, the
    id travels over `torch.distributed` (any backend), every rank calls `b2m_comm_init` (collective)."""

    def __init__(self, group=None, device: Optional[torch.device] = None):
        from . import _cabi
        self.lib = _cabi.load()
        self.rank, self.world = rank_world(group)
        self.handle = C.c_void_p()
        ident = torch.zeros(128, dtype=torch.uint8)
        if self.rank == 0:
            buf = (C.c_uint8 * 128)()
            _cabi.check(self.lib.b2m_comm_unique_id(buf))
            ident = torch.tensor(list(buf), dtype=torch.uint8)
        if self.world > 1:
            backend = td.get_backend(group)
            carrier = ident.cuda() if backend == "nccl" else ident
            td.broadcast(carrier, src=0, group=group)
            ident = carrier.cpu()
        raw = (C.c_uint8 * 128)(*ident.tolist())
        dev = device or torch.device("cuda", torch.cuda.current_device())
        with torch.cuda.device(dev):
            _cabi.check(self.lib.b2m_comm_init(raw, self.world, self.rank, C.byref(self.handle)))

    def attach(self, model) -> None:
        """Collective: sums the shard row counts and makes every later value+gradient of `model` all-reduce."""
        from . import _cabi
        with torch.cuda.device(model.device):
            _cabi.check(self.lib.b2m_model_set_comm(model.handle, self.handle,
                                                    C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        model._comm = self      # keep the communicator alive as long as the model uses it

    def all_reduce_(self, t: torch.Tensor) -> torch.Tensor:
        from . import _cabi
        assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()
        _cabi.check(self.lib.b2m_comm_allreduce_f32(self.handle, C.c_void_p(t.data_ptr()), t.numel(),
                                                    C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        return t

    def close(self):
        h, self.handle = self.handle, C.c_void_p()
        if h:
            self.lib.b2m_comm_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PeerWindow:
    """The peer window of the fused gradient exchange (include/b200mcmc.h, B2M_SLICE_PEER): one cudaMalloc'd window per
    rank, shared through CUDA IPC handles that travel over `torch.distributed`; collective over the group.  After
    construction `nuts(..., slice_state='peer')` on `model` exchanges gradients through plain NVLink stores issued by
    the kernels themselves -- K6's epilogue pushes every finished tile into its owner's window."""

    def __init__(self, model, num_chains: int, group=None):
        from . import _cabi
        self.lib = _cabi.load()
        self.rank, self.world = rank_world(group)
        self.group = group
        self.num_chains = int(num_chains)
        self.own = C.c_void_p()
        self.mapped = {}
        nccl = td.get_backend(group) == "nccl"
        dev = model.device

        def agree(ok: bool, what: str, err=None):
            """every rank learns whether the step worked everywhere: a failure is an error on ALL ranks, never a hang"""
            flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev if nccl else "cpu")
            td.all_reduce(flag, op=td.ReduceOp.MIN, group=group)
            if int(flag) == 0:
                self.close(barrier=False)
                raise RuntimeError(f"peer window: {what} failed on {'this rank: ' + str(err) if not ok else 'another rank'}")

        nbytes, handle, err = C.c_int64(), (C.c_uint8 * 64)(), None
        try:
            with torch.cuda.device(dev):
                _cabi.check(self.lib.b2m_model_peer_bytes(model.handle, self.num_chains, self.world, C.byref(nbytes)))
                _cabi.check(self.lib.b2m_peer_alloc(nbytes.value, C.byref(self.own), handle))
        except Exception as e:      # noqa: BLE001 -- reported on every rank by agree()
            err = e
        agree(err is None, "allocating the window / its CUDA IPC handle", err)
        self.bytes = nbytes.value
        mine = torch.tensor(list(handle), dtype=torch.uint8)
        carrier = mine.to(dev) if nccl else mine
        parts = [torch.zeros_like(carrier) for _ in range(self.world)]
        td.all_gather(parts, carrier, group=group)
        ptrs = (C.c_void_p * self.world)()
        try:
            with torch.cuda.device(dev):
                for s in range(self.world):
                    if s == self.rank:
                        ptrs[s] = self.own.value
                        continue
                    raw = (C.c_uint8 * 64)(*parts[s].cpu().tolist())
                    p = C.c_void_p()
                    _cabi.check(self.lib.b2m_peer_open(raw, C.byref(p)))
                    self.mapped[s] = p
                    ptrs[s] = p.value
        except Exception as e:      # noqa: BLE001
            err = e
        agree(err is None, "mapping the peers' windows (CUDA IPC / peer access)", err)    # also: every window exists and is zeroed
        try:
            with torch.cuda.device(dev):
                _cabi.check(self.lib.b2m_model_peer_attach(model.handle, ptrs, self.world, self.rank, self.num_chains, self.bytes))
        except Exception as e:      # noqa: BLE001
            err = e
        agree(err is None, "attaching the window to the model", err)
        model._peer = self

    def close(self, barrier: bool = True):
        mapped, self.mapped = self.mapped, {}
        for p in mapped.values():
            try:
                self.lib.b2m_peer_close(p)
            except Exception:
                pass
        own, self.own = self.own, C.c_void_p()
        if own:
            try:
                if barrier and td.is_initialized():
                    td.barrier(group=self.group)     # nobody still maps this window
                self.lib.b2m_peer_free(own)
            except Exception:
                pass


def compile_obs_sharded(log_prob_fn, initial_params, group=None, comm: Optional[ObsComm] = None,
                        peer_chains: Optional[int] = None, glm_path: str = "auto"):
    """Trace once, keep this rank's rows, build the device model and attach the communicator.  `peer_chains`: also set
    up the peer window for sliced NUTS runs of that many chains (`nuts(..., slice_state='peer')`)."""
    from .engine import DeviceModel, _require_cuda
    from .tracer import trace
    rank, world = rank_world(group)
    traced = shard_observations(trace(log_prob_fn, initial_params), rank, world)
    model = DeviceModel(traced, _require_cuda(), glm_path=glm_path)
    model._fn = log_prob_fn
    if world > 1:
        # every rank must have chosen the same arithmetic (a shard with wild outliers falls back to the tf32 encoding):
        # agree before the collective calls, so that a mismatch is an error on every rank and not a hang
        flag = torch.tensor([1 if model.glm_path == "tc16" else 0], dtype=torch.int32,
                            device=model.device if td.get_backend(group) == "nccl" else "cpu")
        lo, hi = flag.clone(), flag.clone()
        td.all_reduce(lo, op=td.ReduceOp.MIN, group=group)
        td.all_reduce(hi, op=td.ReduceOp.MAX, group=group)
        if int(lo) != int(hi):
            raise ValueError("observation sharding: the ranks chose different GLM arithmetic paths for their shards; "
                             "pass glm_path='tc' (or 'simt') explicitly")
        (comm or ObsComm(group, model.device)).attach(model)
        if peer_chains:
            if int(lo) != 1:
                raise ValueError("the peer window needs the fp16-encoded tensor-core path on every rank")
            PeerWindow(model, peer_chains, group)
    return model


# ------------------------------------------------------------------------------------------ one call for a sharded run
def run_sharded(log_prob_fn, initial_params, method: str = "nuts", num_chains: int = 1, shard: str = "chains",
                gather: bool = True, group=None, **kwargs):
    """Run `method` ('hmc' | 'nuts' | 'metropolis') over all ranks of the process group.

    shard='chains': this rank runs its block of the `num_chains` global chains (global ids key the random streams).
    shard='obs'   : every rank runs all `num_chains` chains on its row shard of the observations.
    Returns ``(samples, rate, info)``; with ``gather`` the chain axis of `samples` covers all `num_chains` chains
    on every rank (chains) or is the locally held full set (obs -- already identical on every rank)."""
    from .kernels.hmc import hmc
    from .kernels.metropolis import metropolis_hastings
    from .kernels.nuts import nuts
    samplers = {"hmc": hmc, "nuts": nuts, "metropolis": metropolis_hastings}
    if method not in samplers:
        raise ValueError(f"Unknown sampling method: {method}")
    if shard not in ("chains", "obs"):
        raise ValueError(f"Unknown shard mode: {shard}")
    rank, world = rank_world(group)
    kwargs = dict(kwargs)
    kwargs["return_info"] = True
    if shard == "chains":
        count, offset = shard_chains(num_chains, rank, world)
        if count == 0:
            raise ValueError(f"rank {rank} would own no chains (num_chains={num_chains}, world={world})")
        out = samplers[method](log_prob_fn, initial_params, num_chains=count, chain_offset=offset, **kwargs)
        samples, rate, info = out
        if count == 1:       # the single-chain return shape has no chain axis (reference shapes)
            samples = {k: v[None] for k, v in samples.items()}
        if gather and world > 1:
            samples = gather_draws(samples, count, group)
            dev = None if not (td.is_initialized() and td.get_backend(group) == "nccl") else torch.device("cuda")
            tot = reduce_stats({"acc": rate * count, "n": count}, "sum", group, dev)
            rate = tot["acc"] / max(tot["n"], 1.0)
        return samples, rate, info
    if kwargs.get("slice_state") and method != "nuts":
        raise ValueError("slice_state is a NUTS option")
    peer = num_chains if kwargs.get("slice_state") in (True, "peer") and world > 1 else None
    model = compile_obs_sharded(log_prob_fn, initial_params, group, peer_chains=peer)
    samples, rate, info = samplers[method](log_prob_fn, initial_params, num_chains=num_chains, model=model, **kwargs)
    if num_chains == 1:
        samples = {k: v[None] for k, v in samples.items()}
    return samples, rate, info
