"""ctypes binding of the C ABI declared in include/extmcmc.h.

This is the Python stand-in for the Julia `ccall((:extmcmc_xxx, "libextmcmc_cuda"), ...)`
stubs shown in INTEGRATION.md (Julia is not installed in this environment).  There is no
CPU fallback: if libextmcmc_cuda.so is missing or no B200 is visible, every entry point
that needs the device raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libextmcmc_cuda.so")

ABI_VERSION = 2

# status codes
OK, EINVAL, EUNSUPPORTED, ECUDA, ENCCL, EOOM, EDOMAIN, ESTALE = 0, -1, -2, -3, -4, -5, -6, -7
# laws
LAW_GSN_IID_1D, LAW_GSN_MV, LAW_LOGISTIC, LAW_HIER_NORMAL, LAW_USER = 1, 2, 3, 4, 5
USER_GRAD_NONE, USER_GRAD_HAND, USER_GRAD_FORWARD = 0, 1, 2
USER_THETA_TERM = 1                                  # flags of a user law
# kernels
KERNEL_RW_UNIFORM, KERNEL_RW_GAUSS, KERNEL_RW_GAUSS_MIX, KERNEL_MALA = 1, 2, 3, 4
# priors
PRIOR_IMPROPER, PRIOR_IMPROPER_POS, PRIOR_NORMAL, PRIOR_GAMMA, PRIOR_UNIFORM, PRIOR_PRODUCT = 0, 1, 2, 3, 4, 5
PRIOR_EXPONENTIAL, PRIOR_INV_GAMMA, PRIOR_BETA, PRIOR_LOGNORMAL, PRIOR_CAUCHY = 6, 7, 8, 9, 10
PRIOR_MVNORMAL = 11
PRIOR_USER = 12
# adaptation
ADAPT_NONE, ADAPT_UNIF_RW, ADAPT_HAARIO, ADAPT_MALA = 0, 1, 2, 3
# sharding
SHARD_CHAINS, SHARD_OBS = 0, 1
# rng
RNG_PHILOX, RNG_REPLAY = 0, 1

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)
c_int64_p = C.POINTER(C.c_int64)
c_uint8_p = C.POINTER(C.c_uint8)


class Adapt(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("adapt_every_k_steps", C.c_int32),
        ("target_accpt_rate", C.c_double),
        ("scale", C.c_double),
        ("min", C.c_double),
        ("max", C.c_double),
        ("offset", C.c_double),
    ]


class Update(C.Structure):
    _fields_ = [
        ("kernel", C.c_int32),
        ("n_coords", C.c_int32),
        ("coords", c_int32_p),
        ("step", c_double_p),
        ("pos", c_uint8_p),
        ("prior", C.c_int32),
        ("n_prior_params", C.c_int32),
        ("prior_params", c_double_p),
        ("adapt", Adapt),
    ]


class Step(C.Structure):
    _fields_ = [
        ("mcmciter", C.c_int64),
        ("prev_mcmciter", C.c_int64),
        ("pidx", C.c_int32),
        ("prev_pidx", C.c_int32),
    ]


class Config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32),
        ("device", C.c_int32),
        ("n_chains", C.c_int64),
        ("chain_offset", C.c_int64),
        ("n_params", C.c_int32),
        ("n_updates", C.c_int32),
        ("law", C.c_int32),
        ("obs_dim", C.c_int32),
        ("seed", C.c_uint64),
        ("shard_mode", C.c_int32),
        ("rank", C.c_int32),
        ("world_size", C.c_int32),
        ("history_window", C.c_int32),
        ("roll_window", C.c_int32),
        ("use_graphs", C.c_int32),
        ("instrument", C.c_int32),
        ("sweep_variant", C.c_int32),
        ("stats_mode", C.c_int32),
        ("reserved_", C.c_int32 * 3),
    ]


Handle = C.c_void_p
# double f(double lambda, int64 N, int64 mcmc_iter, void *user): HaarioTypeAdaptation's weight schedule
LambdaFn = C.CFUNCTYPE(C.c_double, C.c_double, C.c_int64, C.c_int64, C.c_void_p)

# name -> (restype, argtypes); every symbol declared in include/extmcmc.h
SIGNATURES = {
    "extmcmc_abi_version": (C.c_int32, []),
    "extmcmc_create": (C.c_int32, [C.POINTER(Config), C.POINTER(Handle)]),
    "extmcmc_destroy": (C.c_int32, [Handle]),
    "extmcmc_last_error": (C.c_char_p, [Handle]),
    "extmcmc_upload_obs": (C.c_int32, [Handle, c_double_p, C.c_int64, C.c_int32, c_double_p]),
    "extmcmc_generate_obs_normal": (C.c_int32, [Handle, C.c_int64, C.c_int64, C.c_double, C.c_double, C.c_uint64]),
    "extmcmc_set_user_law": (C.c_int32, [Handle, C.c_char_p, C.c_int32]),
    "extmcmc_user_law_check": (C.c_int32, [C.c_char_p, C.c_int32, C.c_int32, C.c_int32, C.c_char_p, C.c_int64]),
    "extmcmc_set_user_law_chunked": (C.c_int32, [Handle, C.c_char_p, C.c_int32]),
    "extmcmc_user_law_check_chunked": (C.c_int32, [C.c_char_p, C.c_int32, C.c_int32, C.c_int32,
                                                   C.POINTER(C.c_int32), C.c_char_p, C.c_int64]),
    "extmcmc_set_user_law_ex": (C.c_int32, [Handle, C.c_char_p, C.c_int32, C.c_int32, C.c_int32]),
    "extmcmc_user_law_check_ex": (C.c_int32, [C.c_char_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                              C.POINTER(C.c_int32), C.c_char_p, C.c_int64]),
    "extmcmc_set_user_law_theta_only": (C.c_int32, [Handle, C.c_char_p, C.c_int32, C.c_int32, C.c_int32, C.c_uint64]),
    "extmcmc_user_law_check_theta_only": (C.c_int32, [C.c_char_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                                      C.c_int32, C.c_uint64, C.POINTER(C.c_int32), C.c_char_p,
                                                      C.c_int64]),
    "extmcmc_user_prior_check": (C.c_int32, [C.c_char_p, C.c_int32, C.c_int32, C.c_char_p, C.c_int64]),
    "extmcmc_set_user_prior": (C.c_int32, [Handle, C.c_int32, C.c_char_p, C.c_int32]),
    "extmcmc_eval_user_prior": (C.c_int32, [Handle, C.c_int32, c_double_p, c_double_p]),
    "extmcmc_set_update": (C.c_int32, [Handle, C.c_int32, C.POINTER(Update)]),
    "extmcmc_set_state": (C.c_int32, [Handle, c_double_p]),
    "extmcmc_set_seed": (C.c_int32, [Handle, C.c_uint64]),
    "extmcmc_set_lambda_fn": (C.c_int32, [Handle, C.c_int32, LambdaFn, C.c_void_p]),
    "extmcmc_checkpoint_size": (C.c_int32, [Handle, c_int64_p]),
    "extmcmc_checkpoint_save": (C.c_int32, [Handle, C.c_void_p, C.c_int64]),
    "extmcmc_checkpoint_load": (C.c_int32, [Handle, C.c_void_p, C.c_int64]),
    "extmcmc_comm_unique_id": (C.c_int32, [c_uint8_p]),
    "extmcmc_comm_init": (C.c_int32, [Handle, c_uint8_p]),
    "extmcmc_p2p_export": (C.c_int32, [Handle, c_uint8_p]),
    "extmcmc_p2p_import": (C.c_int32, [Handle, c_uint8_p]),
    "extmcmc_run_block": (C.c_int32, [Handle, C.POINTER(Step), C.c_int32]),
    "extmcmc_run_block_replay": (C.c_int32, [Handle, C.POINTER(Step), C.c_int32, C.c_int32, c_double_p, c_double_p]),
    "extmcmc_sync": (C.c_int32, [Handle]),
    "extmcmc_get_state": (C.c_int32, [Handle, c_double_p, c_double_p]),
    "extmcmc_get_history": (C.c_int32, [Handle, C.c_int64, C.c_int64, c_double_p, c_double_p, c_double_p, c_double_p, c_uint8_p]),
    "extmcmc_history_fetch_begin": (C.c_int32, [Handle, C.c_int64, C.c_int64]),
    "extmcmc_history_fetch_end": (C.c_int32, [Handle, c_double_p, c_double_p, c_double_p, c_double_p, c_uint8_p]),
    "extmcmc_get_stats": (C.c_int32, [Handle, c_double_p, c_double_p, c_double_p, c_int64_p, c_int64_p]),
    "extmcmc_get_eps": (C.c_int32, [Handle, C.c_int32, c_double_p]),
    "extmcmc_get_adapt_state": (C.c_int32, [Handle, C.c_int32, c_double_p, c_double_p]),
    "extmcmc_eval_loglik": (C.c_int32, [Handle, c_double_p]),
    "extmcmc_eval_grad": (C.c_int32, [Handle, c_double_p, c_double_p]),
    "extmcmc_timer_start": (C.c_int32, [Handle]),
    "extmcmc_timer_stop": (C.c_int32, [Handle, C.POINTER(C.c_float)]),
    "extmcmc_event_record": (C.c_int32, [Handle, C.c_int32]),
    "extmcmc_event_elapsed": (C.c_int32, [Handle, C.c_int32, C.c_int32, C.POINTER(C.c_float)]),
    "extmcmc_get_sweep_time": (C.c_int32, [Handle, C.POINTER(C.c_float), c_int64_p]),
    "extmcmc_launch_count": (C.c_int64, [Handle]),
    "extmcmc_flush_l2": (C.c_int32, [Handle]),
    "extmcmc_measure_fp64_peak": (C.c_int32, [Handle, c_double_p]),
    "extmcmc_measure_dmma_peak": (C.c_int32, [Handle, c_double_p]),
    "extmcmc_sweep_variant_name": (C.c_char_p, [Handle]),
}

_lib = None


class ExtMCMCError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libextmcmc_cuda error {code}: {msg}")
        self.code = code


def load():
    """dlopen libextmcmc_cuda.so and type every entry point.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback for the GPU path)"
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.extmcmc_abi_version() != ABI_VERSION:
        raise ImportError("libextmcmc_cuda.so ABI version mismatch")
    _lib = lib
    return lib


def check(handle, rc):
    if rc != OK:
        msg = load().extmcmc_last_error(handle)
        raise ExtMCMCError(rc, msg.decode() if msg else "")
    return rc


def dptr(a):
    return a.ctypes.data_as(c_double_p) if a is not None else None
