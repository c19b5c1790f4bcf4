"""ctypes binding of libdemcmc_b200.so (include/demcmc_b200.h).

The Julia package would bind the same entry points with `ccall` (julia/GPULoglike.jl); this module
is the runnable mirror used where no Julia toolchain exists.  There is no CPU fallback: if the
library is missing, or there is no CUDA device, calls fail loudly.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
DEFAULT_LIB = os.path.join(_HERE, "libdemcmc_b200.so")
ABI_VERSION = 8

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)
_bp = C.POINTER(C.c_uint8)


class DemcmcError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libdemcmc_b200 error {code}: {msg}")
        self.code = code


class Prior(C.Structure):
    _fields_ = [("kind", C.c_int32), ("ref", C.c_int32), ("a", C.c_double), ("b", C.c_double)]


class Model(C.Structure):
    _fields_ = [("kind", C.c_int32), ("d", C.c_int32), ("n_obs", C.c_int64), ("n_dim", C.c_int32),
                ("n_per", C.c_int32), ("x", C.c_void_p), ("choice", C.c_void_p), ("sigma", _dp),
                ("lba_floor", C.c_double), ("prior", C.POINTER(Prior)), ("data_on_device", C.c_int32),
                ("n_cols", C.c_int32), ("cov", _dp), ("center", _dp), ("source", C.c_char_p), ("n_sim", C.c_int32),
                ("sim_floor", C.c_double)]


class Config(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("n_groups", C.c_int32), ("Np", C.c_int32), ("d", C.c_int32),
                ("burnin", C.c_int32), ("n_initial", C.c_int32),
                ("alpha", C.c_double), ("beta", C.c_double), ("eps", C.c_double), ("sigma", C.c_double),
                ("kappa", C.c_double), ("theta_snooker", C.c_double),
                ("proposal", C.c_int32), ("n_blocks", C.c_int32), ("blocks", _bp), ("lo", _dp), ("hi", _dp),
                ("seed", C.c_uint64), ("device", C.c_int32), ("group_begin", C.c_int32),
                ("group_count", C.c_int32), ("donors", C.c_int32), ("trace", C.c_int32),
                ("store_every", C.c_int32), ("update", C.c_int32), ("fitness", C.c_int32),
                ("n_devices", C.c_int32), ("devices", _ip)]


class Tape(C.Structure):
    _fields_ = [("mig_u", _dp), ("mig_n", _ip), ("mig_groups", _ip), ("mig_pick_u", _dp), ("kind", _bp),
                ("idx", _ip), ("gamma1", _dp), ("gamma2", _dp), ("u_acc", _dp), ("noise", _dp), ("keep", _bp),
                ("idx_row", _ip)]


class Counters(C.Structure):
    _fields_ = [("iterations", C.c_int64), ("sweeps", C.c_int64), ("particle_updates", C.c_int64),
                ("loglike_evals", C.c_int64), ("kernel_launches", C.c_int64), ("levels", C.c_int64),
                ("device_ms", C.c_double), ("loglike_ms", C.c_double), ("persistent_chunks", C.c_int64),
                ("mailbox_events", C.c_int64), ("cross_migrations", C.c_int64)]


class Evidence(C.Structure):
    _fields_ = [("n_rungs", C.c_int32), ("log_z_ti", C.c_double), ("log_z_ti2", C.c_double), ("log_z_ss", C.c_double),
                ("se_ti", C.c_double), ("se_ss", C.c_double)]


# every symbol include/demcmc_b200.h declares (tests check the library exports all of them)
SYMBOLS = [
    "demcmc_last_error", "demcmc_abi_version", "demcmc_device_count", "demcmc_backend_name", "demcmc_create",
    "demcmc_destroy", "demcmc_set_model", "demcmc_compile_loglike", "demcmc_compile_simulator", "demcmc_set_history", "demcmc_set_state", "demcmc_run", "demcmc_replay", "demcmc_get_samples",
    "demcmc_get_accept", "demcmc_get_lp", "demcmc_get_chains", "demcmc_get_moments", "demcmc_set_iteration", "demcmc_set_weights", "demcmc_set_blocking_schedule", "demcmc_get_history_by_slot", "demcmc_get_state", "demcmc_get_trace",
    "demcmc_get_trace_xdot", "demcmc_eval_xdot", "demcmc_eval_simulated", "demcmc_set_sufficient_stat", "demcmc_get_diagnostics",
    "demcmc_get_migration", "demcmc_get_counters", "demcmc_set_timing", "demcmc_set_max_chunk", "demcmc_set_lanes", "demcmc_eval", "demcmc_eval_pointwise", "demcmc_loo",
    "demcmc_set_temperatures", "demcmc_get_loglike", "demcmc_power_posterior", "demcmc_op_project", "demcmc_op_reset",
    "demcmc_op_de_proposal", "demcmc_op_snooker", "demcmc_op_accept", "demcmc_op_select", "demcmc_comm_unique_id",
    "demcmc_comm_init", "demcmc_fp64_peak", "demcmc_fp64_peaks", "demcmc_copy_peak",
]

_lib = None
_lib_path = None


def _declare(L):
    L.demcmc_last_error.restype = C.c_char_p
    L.demcmc_backend_name.restype = C.c_char_p
    for name in SYMBOLS:
        fn = getattr(L, name)
        if name not in ("demcmc_last_error", "demcmc_backend_name"):
            fn.restype = C.c_int
    L.demcmc_create.argtypes = [C.POINTER(Config), C.POINTER(C.c_void_p)]
    L.demcmc_destroy.argtypes = [C.c_void_p]
    L.demcmc_set_model.argtypes = [C.c_void_p, C.POINTER(Model)]
    L.demcmc_compile_loglike.argtypes = [C.c_char_p, C.c_char_p, C.c_int64]
    L.demcmc_compile_simulator.argtypes = [C.c_char_p, C.c_char_p, C.c_int64]
    L.demcmc_set_history.argtypes = [C.c_void_p, _dp]
    L.demcmc_set_state.argtypes = [C.c_void_p, _dp, _ip]
    L.demcmc_run.argtypes = [C.c_void_p, C.c_int64]
    L.demcmc_replay.argtypes = [C.c_void_p, C.POINTER(Tape), C.c_int64]
    L.demcmc_get_samples.argtypes = [C.c_void_p, _dp, C.c_int64]
    L.demcmc_get_accept.argtypes = [C.c_void_p, _bp, C.c_int64]
    L.demcmc_get_lp.argtypes = [C.c_void_p, _dp, C.c_int64]
    L.demcmc_get_chains.argtypes = [C.c_void_p, C.c_int64, C.c_int64, _dp]
    L.demcmc_set_iteration.argtypes = [C.c_void_p, C.c_int64]
    L.demcmc_set_weights.argtypes = [C.c_void_p, _dp]
    L.demcmc_set_blocking_schedule.argtypes = [C.c_void_p, _bp, C.c_int64]
    L.demcmc_get_moments.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.POINTER(C.c_int64), _dp, _dp]
    L.demcmc_get_history_by_slot.argtypes = [C.c_void_p, C.c_int64, C.c_int64, _dp, _dp, _ip, _bp]
    L.demcmc_get_state.argtypes = [C.c_void_p, _dp, _dp, _ip]
    L.demcmc_get_trace.argtypes = [C.c_void_p, _dp, _dp, _dp, _bp]
    L.demcmc_get_diagnostics.argtypes = [C.c_void_p, C.c_int64, C.c_int64, _dp, _dp]
    L.demcmc_get_trace_xdot.argtypes = [C.c_void_p, _dp]
    L.demcmc_eval_xdot.argtypes = [C.c_void_p, _dp, C.c_int64, _dp]
    L.demcmc_eval_simulated.argtypes = [C.c_void_p, _dp, C.c_int64, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), _dp, _dp]
    L.demcmc_set_sufficient_stat.argtypes = [C.c_void_p, C.c_int32]
    L.demcmc_get_migration.argtypes = [C.c_void_p, _ip]
    L.demcmc_get_counters.argtypes = [C.c_void_p, C.POINTER(Counters)]
    L.demcmc_set_timing.argtypes = [C.c_void_p, C.c_int64, C.c_int32]
    L.demcmc_set_max_chunk.argtypes = [C.c_void_p, C.c_int32]
    L.demcmc_set_lanes.argtypes = [C.c_void_p, C.c_int32]
    L.demcmc_eval.argtypes = [C.c_void_p, _dp, C.c_int64, _dp, _dp]
    L.demcmc_eval_pointwise.argtypes = [C.c_void_p, _dp, C.c_int64, C.c_int64, C.c_int64, _dp]
    L.demcmc_loo.argtypes = [C.c_void_p, _dp, C.c_int64, _dp, _dp, _dp, _dp]
    L.demcmc_set_temperatures.argtypes = [C.c_void_p, _dp, C.c_int32]
    L.demcmc_get_loglike.argtypes = [C.c_void_p, _dp, C.c_int64]
    L.demcmc_power_posterior.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.POINTER(Evidence), _dp, _dp, _dp, _dp, _dp, _dp]
    L.demcmc_op_project.argtypes = [C.c_int, _dp, _dp, C.c_int32, _dp]
    L.demcmc_op_reset.argtypes = [C.c_int, _dp, _dp, _bp, C.c_int32, _dp]
    L.demcmc_op_de_proposal.argtypes = [C.c_int, _dp, _dp, _dp, _dp, C.c_double, C.c_double, _dp, C.c_int32, _dp]
    L.demcmc_op_snooker.argtypes = [C.c_int, _dp, _dp, _dp, _dp, C.c_double, _dp, C.c_int32, _dp, _dp]
    L.demcmc_op_accept.argtypes = [C.c_int, _dp, _dp, _dp, _dp, C.c_int32, _bp]
    L.demcmc_op_select.argtypes = [C.c_int, _dp, C.c_int32, C.c_double, _ip, _ip]
    L.demcmc_comm_unique_id.argtypes = [_bp]
    L.demcmc_comm_init.argtypes = [C.c_void_p, _bp, C.c_int32, C.c_int32]
    L.demcmc_fp64_peak.argtypes = [C.c_int, _dp]
    L.demcmc_fp64_peaks.argtypes = [C.c_int, _dp, _dp]
    L.demcmc_copy_peak.argtypes = [C.c_int, _dp]


def use_library(path: str):
    """Bind an explicit shared object (tests inject the host-only test double this way; the
    package itself only ever loads DEFAULT_LIB)."""
    global _lib, _lib_path
    if not os.path.exists(path):
        raise FileNotFoundError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). libdemcmc_b200 has no CPU fallback.")
    L = C.CDLL(path)
    _declare(L)
    if L.demcmc_abi_version() != ABI_VERSION:
        raise DemcmcError(-1, f"ABI version mismatch: library {L.demcmc_abi_version()} != {ABI_VERSION}")
    _lib, _lib_path = L, path
    return L


def lib():
    if _lib is None:
        use_library(DEFAULT_LIB)
    return _lib


def lib_path():
    return _lib_path


def check(rc):
    if rc != 0:
        raise DemcmcError(rc, lib().demcmc_last_error().decode())


def ptr(a, ct):
    return a.ctypes.data_as(ct) if a is not None else ct()


def f8(a):
    return np.ascontiguousarray(a, dtype=np.float64)
