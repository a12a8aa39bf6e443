"""ctypes binding of libb200mcmc.so (include/b200mcmc.h).  The structures below mirror the header
field for field; `load()` verifies their sizes against b2m_struct_sizes() so a drifted mirror fails
loudly instead of corrupting memory.  There is no fallback: if the library is missing or the CUDA
device is absent, the product path raises.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

c_f = C.c_float
c_p = C.c_void_p


class Operand(C.Structure):
    _fields_ = [("kind", C.c_int32), ("a", C.c_int32), ("b", C.c_int32), ("c", c_f)]


class LinEntry(C.Structure):
    _fields_ = [("param", C.c_int32), ("array", C.c_int32), ("coef", c_f)]


class Term(C.Structure):
    _fields_ = [("dist", C.c_int32), ("length", C.c_int32), ("weight", c_f), ("k0", c_f), ("k1", c_f), ("k2", c_f),
                ("x", Operand), ("p0", Operand), ("p1", Operand)]


class Array(C.Structure):
    _fields_ = [("data", c_p), ("rows", C.c_int64), ("cols", C.c_int64)]


class ModelOptions(C.Structure):
    _fields_ = [("glm_path", C.c_int32), ("pointwise_path", C.c_int32), ("transforms", C.POINTER(C.c_int32)),
                ("glm_form", C.c_int32), ("reserved", C.c_int32 * 3)]


class HmcArgs(C.Structure):
    _fields_ = [("n_chains", C.c_int64), ("chain_offset", C.c_int64), ("iter_offset", C.c_int64),
                ("n_iter", C.c_int32), ("n_leapfrog", C.c_int32), ("adapt", C.c_int32), ("lanes", C.c_int32),
                ("target_accept", C.c_double), ("seed", C.c_uint64),
                ("theta", c_p), ("step_size", c_p), ("n_accept", c_p), ("n_total", c_p), ("da_state", c_p),
                ("draws", c_p), ("inj_normal", c_p), ("inj_uniform", c_p), ("trace_energy", c_p), ("trace_accept", c_p),
                ("inv_mass", c_p), ("draws_unconstrained", C.c_int32), ("_pad2", C.c_int32), ("adapt_origin", C.c_int64)]


class MhArgs(C.Structure):
    _fields_ = [("n_chains", C.c_int64), ("chain_offset", C.c_int64), ("iter_offset", C.c_int64),
                ("n_iter", C.c_int32), ("lanes", C.c_int32), ("proposal_scale", c_f), ("_pad", C.c_int32),
                ("seed", C.c_uint64),
                ("theta", c_p), ("logp", c_p), ("n_accept", c_p), ("draws", c_p),
                ("inj_normal", c_p), ("inj_uniform", c_p), ("trace_accept", c_p)]


class NutsArgs(C.Structure):
    _fields_ = [("n_chains", C.c_int64), ("chain_offset", C.c_int64), ("iter_offset", C.c_int64),
                ("n_iter", C.c_int32), ("max_tree_depth", C.c_int32), ("adapt", C.c_int32), ("compat", C.c_int32),
                ("lanes", C.c_int32), ("step_size_jitter", c_f), ("target_accept", C.c_double), ("seed", C.c_uint64),
                ("theta", c_p), ("step_size", c_p), ("da_state", c_p), ("n_accept", c_p), ("n_leaves", c_p),
                ("n_diverge", c_p), ("draws", c_p), ("depths", c_p), ("alphas", c_p),
                ("inj_normal", c_p), ("inj_slice", c_p), ("inj_dir", c_p), ("inj_take", c_p), ("inj_merge", c_p),
                ("trace_doubling", c_p), ("trace_energy", c_p),
                ("inv_mass", c_p), ("schedule", C.c_int32), ("slice_state", C.c_int32),
                ("draws_unconstrained", C.c_int32), ("_pad2", C.c_int32), ("adapt_origin", C.c_int64)]


ADAPT_NONE, ADAPT_REFERENCE, ADAPT_DUAL_AVERAGING, ADAPT_POOLED = 0, 1, 2, 3
COMPAT_REFERENCE, COMPAT_CORRECT = 0, 1
SCHED_ASYNC, SCHED_SYNC = 0, 1
SLICE_OFF, SLICE_NCCL, SLICE_PEER = 0, 1, 2
TF_NONE, TF_LOG, TF_LOGIT = 0, 1, 2
GLM_AUTO, GLM_SIMT, GLM_TC, GLM_TC16 = 0, 1, 2, 3
GLM_PATHS = {"auto": GLM_AUTO, "simt": GLM_SIMT, "tc": GLM_TC, "tc16": GLM_TC16}
POINTWISE_AUTO, POINTWISE_GENERAL = 0, 1
FORM_AUTO, FORM_STREAM, FORM_GRAM = 0, 1, 2
GLM_FORMS = {"auto": FORM_AUTO, "stream": FORM_STREAM, "gram": FORM_GRAM}
MAX_TREE_DEPTH = 12
ABI_VERSION = 4

EXPORTS = ["b2m_last_error", "b2m_abi_version", "b2m_struct_sizes", "b2m_model_create", "b2m_model_destroy",
           "b2m_model_dim", "b2m_model_class", "b2m_model_glm_path", "b2m_model_glm_form", "b2m_logp_grad", "b2m_hmc_run", "b2m_mh_run", "b2m_nuts_run",
           "b2m_launch_count", "b2m_comm_unique_id", "b2m_comm_init", "b2m_comm_destroy", "b2m_model_set_comm",
           "b2m_comm_allreduce_f32", "b2m_profile", "b2m_profile_read", "b2m_diag_series", "b2m_diag_params", "b2m_sample",
           "b2m_options_size", "b2m_peer_alloc", "b2m_peer_open", "b2m_peer_close", "b2m_peer_free", "b2m_model_peer_bytes",
           "b2m_model_peer_attach", "b2m_mass_from_draws", "b2m_quantiles", "b2m_model_attach_module", "b2m_model_has_module", "b2m_profile_read_ex",
           "b2m_loglik_stats"]

_lib = None


class B2MError(RuntimeError):
    """A nonzero status from libb200mcmc.so (message from b2m_last_error)."""


def lib_path() -> str:
    return _build.LIB


def load(build_if_missing: bool = True):
    """dlopen the in-tree library (building it with nvcc first if it is absent or stale and a
    compiler is available) and declare the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    dbg = os.environ.get("B2M_LIB")       # developer switch: the debug-assert build (python -m mlx_mcmc_b200.build --debug)
    if dbg:
        if not os.path.exists(dbg):
            raise ImportError(f"B2M_LIB={dbg} does not exist")
        path, build_if_missing = dbg, False
    if build_if_missing and not _build.is_current():
        try:
            _build.build()
        except Exception as e:
            # A library that does not match the checked-in sources must never run silently: parity claims refer to the
            # sources.  (A box without nvcc gets the library from the snapshot, built and stamped where the sources were.)
            raise ImportError(f"libb200mcmc.so is missing or older than its sources and could not be rebuilt here: {e}") from e
    if not os.path.exists(path):
        raise ImportError(f"{path} not found; run `python -m mlx_mcmc_b200.build` (needs nvcc)")
    lib = C.CDLL(path)
    lib.b2m_last_error.restype = C.c_char_p
    lib.b2m_abi_version.restype = C.c_int
    lib.b2m_launch_count.restype = C.c_int64
    lib.b2m_struct_sizes.argtypes = [C.POINTER(C.c_int32)]
    lib.b2m_model_create.argtypes = [C.POINTER(Term), C.c_int32, C.POINTER(LinEntry), C.c_int32,
                                     C.POINTER(Array), C.c_int32, C.c_int32, C.POINTER(ModelOptions), C.POINTER(c_p)]
    lib.b2m_model_attach_module.argtypes = [c_p, c_p, C.c_int64, C.c_int32]
    lib.b2m_model_has_module.argtypes = [c_p]
    lib.b2m_peer_alloc.argtypes = [C.c_int64, C.POINTER(c_p), c_p]
    lib.b2m_peer_open.argtypes = [c_p, C.POINTER(c_p)]
    lib.b2m_peer_close.argtypes = [c_p]
    lib.b2m_peer_free.argtypes = [c_p]
    lib.b2m_model_peer_bytes.argtypes = [c_p, C.c_int64, C.c_int32, C.POINTER(C.c_int64)]
    lib.b2m_model_peer_attach.argtypes = [c_p, C.POINTER(c_p), C.c_int32, C.c_int32, C.c_int64, C.c_int64]
    lib.b2m_mass_from_draws.argtypes = [c_p, C.c_int64, C.c_int64, C.c_int64, c_p, c_p]
    lib.b2m_quantiles.argtypes = [c_p, C.c_int64, C.POINTER(C.c_double), C.c_int32, C.POINTER(C.c_double), c_p]
    lib.b2m_model_destroy.argtypes = [c_p]
    lib.b2m_model_destroy.restype = None
    lib.b2m_model_dim.argtypes = [c_p]
    lib.b2m_model_class.argtypes = [c_p]
    lib.b2m_model_glm_path.argtypes = [c_p]
    lib.b2m_model_glm_form.argtypes = [c_p]
    lib.b2m_logp_grad.argtypes = [c_p, c_p, C.c_int64, c_p, c_p, C.c_int32, c_p]
    lib.b2m_loglik_stats.argtypes = [c_p, c_p, C.c_int64, C.POINTER(C.c_int32), C.c_int32, c_p, C.c_int64, c_p]
    lib.b2m_hmc_run.argtypes = [c_p, C.POINTER(HmcArgs), c_p]
    lib.b2m_mh_run.argtypes = [c_p, C.POINTER(MhArgs), c_p]
    lib.b2m_nuts_run.argtypes = [c_p, C.POINTER(NutsArgs), c_p]
    lib.b2m_diag_series.argtypes = [c_p, C.c_int64, C.c_int64, C.c_int64, C.c_int32, c_p, c_p, c_p, c_p, c_p]
    lib.b2m_diag_params.argtypes = [c_p, c_p, c_p, c_p, C.c_int64, C.c_int64, C.c_int64, c_p, c_p]
    lib.b2m_sample.argtypes = [C.c_int32, c_f, c_f, c_p, C.c_int32, C.c_uint64, C.c_int64, c_p, c_p]
    lib.b2m_profile.argtypes = [C.c_int32]
    lib.b2m_profile_read.argtypes = [C.POINTER(C.c_double)]
    lib.b2m_profile_read_ex.argtypes = [C.POINTER(C.c_double)]
    lib.b2m_comm_unique_id.argtypes = [c_p]
    lib.b2m_comm_init.argtypes = [c_p, C.c_int32, C.c_int32, C.POINTER(c_p)]
    lib.b2m_comm_destroy.argtypes = [c_p]
    lib.b2m_comm_destroy.restype = None
    lib.b2m_model_set_comm.argtypes = [c_p, c_p, c_p]
    lib.b2m_comm_allreduce_f32.argtypes = [c_p, c_p, C.c_int64, c_p]
    if lib.b2m_abi_version() != ABI_VERSION:
        raise ImportError(f"libb200mcmc.so ABI {lib.b2m_abi_version()} != binding {ABI_VERSION}")
    sizes = (C.c_int32 * 6)()
    lib.b2m_struct_sizes(sizes)
    mine = [C.sizeof(Term), C.sizeof(Operand), C.sizeof(LinEntry), C.sizeof(HmcArgs), C.sizeof(MhArgs), C.sizeof(NutsArgs)]
    if list(sizes) != mine:
        raise ImportError(f"struct layout mismatch: library {list(sizes)} vs ctypes mirror {mine}")
    if lib.b2m_options_size() != C.sizeof(ModelOptions):
        raise ImportError(f"b2m_model_options layout mismatch: library {lib.b2m_options_size()} vs {C.sizeof(ModelOptions)}")
    _lib = lib
    return lib


def check(status: int):
    if status != 0:
        msg = load().b2m_last_error()
        raise B2MError(f"libb200mcmc status {status}: {msg.decode() if msg else '?'}")
