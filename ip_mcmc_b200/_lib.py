"""ctypes binding of libipmcmc.so (include/ipmcmc.h).  There is NO fallback: if the library is
missing or a call fails, an exception is raised."""
import ctypes as C
import os

from . import build as _build

ABI_VERSION = 2
MAX_DIM = 32          # parameter vector on the lanes of one warp
MAX_DIM_WIDE = 256    # Burgers KL prior: parameter vector in shared memory (include/ipmcmc.h)
MAX_OBS = 64
N_COUNTERS = 6
MODEL_BURGERS, MODEL_LORENZ = 1, 2
NUMERICS_EXACT, NUMERICS_FUSED = 0, 1
PROPOSE_RW, PROPOSE_PCN = 0, 1
ACCEPT_RW, ACCEPT_PCN = 0, 1
BURGERS_NO_MONOTONE_SHORTCUT = 1

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)
c_int64_p = C.POINTER(C.c_int64)


class PotentialDesc(C.Structure):
    _fields_ = [("n_obs", C.c_int32), ("whiten_dense", C.c_int32), ("y", c_double_p), ("perm", c_int32_p),
                ("scale", c_double_p), ("LP", c_double_p), ("log_const", C.c_double)]


class BurgersDesc(C.Structure):
    _fields_ = [("n_cells", C.c_int32), ("numerics", C.c_int32), ("max_fv_steps", C.c_int32),
                ("n_params", C.c_int32), ("T", C.c_double), ("dx", C.c_double), ("dx_meas", C.c_double),
                ("x", c_double_p), ("param_mean", c_double_p), ("win_left", c_int32_p),
                ("win_right", c_int32_p), ("n_kl_modes", C.c_int32), ("flags", C.c_int32),
                ("kl_basis", c_double_p), ("potential", PotentialDesc)]


class LorenzDesc(C.Structure):
    _fields_ = [("K", C.c_int32), ("J", C.c_int32), ("max_attempts", C.c_int32), ("numerics", C.c_int32),
                ("T", C.c_double), ("c", C.c_double), ("rtol", C.c_double), ("atol", C.c_double),
                ("param_mean", c_double_p), ("potential", PotentialDesc)]


class SamplerDesc(C.Structure):
    _fields_ = [("dim", C.c_int32), ("proposer", C.c_int32), ("accepter", C.c_int32),
                ("factor_kind", C.c_int32), ("recompute_phi_u", C.c_int32), ("has_constraint", C.c_int32),
                ("reserved0", C.c_int32), ("reserved1", C.c_int32),
                ("coef_u", C.c_double), ("coef_w", C.c_double), ("coef_sched_dev", C.c_void_p),
                ("n_sched", C.c_int64), ("factor", c_double_p), ("prior_chol", c_double_p),
                ("box_lo", c_double_p), ("box_hi", c_double_p), ("box_shift", c_double_p),
                ("seed", C.c_uint64), ("chain_offset", C.c_int64), ("first_step", C.c_int64),
                ("record_start", C.c_int64), ("record_interval", C.c_int64)]


class ChainBuffers(C.Structure):
    _fields_ = [("u_dev", C.c_void_p), ("phi_dev", C.c_void_p), ("model_state_dev", C.c_void_p),
                ("mom_count_dev", C.c_void_p), ("mom_mean_dev", C.c_void_p), ("mom_m2_dev", C.c_void_p),
                ("counters_dev", C.c_void_p), ("trace_dev", C.c_void_p), ("n_record", C.c_int64),
                ("steplog_dev", C.c_void_p), ("vlog_dev", C.c_void_p), ("inject_w_dev", C.c_void_p),
                ("inject_u_dev", C.c_void_p), ("slot_chain_dev", C.c_void_p), ("n_slots", C.c_int32),
                ("warps_per_cta", C.c_int32), ("sched_dev", C.c_void_p), ("sched_len", C.c_int64),
                ("sched_chunk", C.c_int32), ("reserved", C.c_int32)]


class HostIO(C.Structure):
    _fields_ = [("u0_host", c_double_p), ("phi0_host", c_double_p), ("model_state_host", c_double_p),
                ("samples_host", c_double_p), ("n_record", C.c_int64), ("u_host", c_double_p),
                ("phi_host", c_double_p), ("counters_host", c_int64_p), ("pooled_host", c_double_p),
                ("scheduler", C.c_int32), ("sched_chunk", C.c_int32)]


# every symbol include/ipmcmc.h declares
SYMBOLS = {
    "ipmcmc_burgers_create": (C.c_int, [C.POINTER(BurgersDesc), C.POINTER(C.c_void_p)]),
    "ipmcmc_lorenz_create": (C.c_int, [C.POINTER(LorenzDesc), C.POINTER(C.c_void_p)]),
    "ipmcmc_destroy": (None, [C.c_void_p]),
    "ipmcmc_forward": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p]),
    "ipmcmc_run": (C.c_int, [C.c_void_p, C.POINTER(SamplerDesc), C.POINTER(ChainBuffers), C.c_int64,
                             C.c_int64, C.c_void_p]),
    "ipmcmc_run_tempered": (C.c_int, [C.c_void_p, C.POINTER(SamplerDesc), C.POINTER(ChainBuffers), C.c_void_p,
                                      C.c_int64, C.c_int64, C.c_void_p]),
    "ipmcmc_swap_replicas": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_uint64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p]),
    "ipmcmc_pool_scratch_bytes": (C.c_int64, [C.c_int64, C.c_int32]),
    "ipmcmc_pool_moments": (C.c_int, [C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "ipmcmc_sample_host": (C.c_int, [C.c_void_p, C.POINTER(SamplerDesc), C.c_int64, C.c_int64, C.POINTER(HostIO),
                                     C.c_void_p]),
    "ipmcmc_diag_scratch_bytes": (C.c_int64, [C.c_int64, C.c_int32, C.c_int64]),
    "ipmcmc_diag_tau": (C.c_int, [C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "ipmcmc_diag_seqstats": (C.c_int, [C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                       C.c_int64, C.c_void_p]),
    "ipmcmc_diag_variogram": (C.c_int, [C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.c_int64, C.c_int64,
                                        C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]),
    "ipmcmc_diag_truncate": (C.c_int, [C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p]),
    "ipmcmc_histogram_accumulate": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_void_p]),
    "ipmcmc_lorenz_rhs": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p]),
    "ipmcmc_lorenz_rk45_attempt": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_double, C.c_double, C.c_void_p, C.c_void_p]),
    "ipmcmc_div_probe": (C.c_int, [C.c_int64, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ipmcmc_rng_probe": (C.c_int, [C.c_uint64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int32,
                                   C.c_void_p, C.c_void_p]),
    "ipmcmc_fp64_peak": (C.c_int, [C.c_int32, c_double_p]),
    "ipmcmc_last_error": (C.c_char_p, []),
    "ipmcmc_abi_version": (C.c_int, []),
}

_lib = None


class EngineError(RuntimeError):
    pass


def lib_path():
    # IPMCMC_LIB: developer override used by tools/build_variants.py for A/B measurements of kernel
    # variants (same ABI, same sources, different -D switches)
    return os.environ.get("IPMCMC_LIB") or _build.LIB


def load():
    """Load libipmcmc.so (must have been built: `python -m ip_mcmc_b200.build` or
    __graft_entry__.build()).  Raises if it is missing -- there is no CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise EngineError("%s not found: build it with `python -m ip_mcmc_b200.build` "
                          "(the engine has no CPU fallback)" % path)
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)      # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.ipmcmc_abi_version() != ABI_VERSION:
        raise EngineError("ABI version mismatch")
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().ipmcmc_last_error().decode()
        if rc == -1:
            raise ValueError(msg)
        raise EngineError("libipmcmc error %d: %s" % (rc, msg))


def as_double_p(a):
    return a.ctypes.data_as(c_double_p)


def as_int32_p(a):
    return a.ctypes.data_as(c_int32_p)
