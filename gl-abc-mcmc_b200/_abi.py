"""ctypes mirror of include/glabc.h (the C-ABI boundary) and the loader of libglabc.so.

The library is the product: there is no CPU fallback.  `load()` raises if the shared object is
missing (run `python -c "import __graft_entry__ as g; g.build()"`), and `Context()` raises if no
CUDA device is usable.
"""
import ctypes as C
import os

MAX_DIM = 8
MAX_MODES = 8
MAX_K = 16
AUX_SLOTS = 8
AUX_LOGW, AUX_LOCAL, AUX_WIDE, AUX_LW_WIDE, AUX_HAVE_GRAD = 0, 1, 2, 3, 4
DEBUG_SLOTS = 4 + MAX_K
STATE64_SLOTS, S64_THETA, S64_Y, S64_GRAD, S64_LOGW = 16, 0, 4, 8, 12
DEBUG64_SLOTS = 36
MAX_NUM_GRAD = 4096

OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_CUDA, ERR_NO_DEVICE = range(5)

MODEL_ABS_NORMAL, MODEL_ID_NORMAL = 1, 2
DIST_NONE, DIST_DIAG_GAUSSIAN, DIST_UNIFORM, DIST_GAMMA, DIST_GAUSSIAN_MIXTURE = range(5)
SLOT_LOCAL, SLOT_GLOBAL, SLOT_IMPORTANCE = range(3)
RNG_NATIVE, RNG_REPLAY = 0, 1
ARITH_FAST, ARITH_STRICT = 0, 1
TRACE_NONE, TRACE_TIME_MAJOR, TRACE_CHAIN_MAJOR, TRACE_EVENTS = 0, 1, 2, 3
FLOW_FAST, FLOW_PRECISE = 0, 1

STAT_STEPS, STAT_GLOBAL_STEPS, STAT_ACC_LOCAL, STAT_ACC_GLOBAL, STAT_SUM = 0, 1, 2, 3, 4


def nstats(d):
    return 4 + 2 * d + (d * (d + 1)) // 2


def tape_global_slots(d, yd):
    return 2 + d + yd


def tape_isir_slots(d, yd, k):
    return 2 + k * (d + yd)


def tape_mala_slots(d, yd, k, num):
    return 2 + k * (d + yd) + d * num * yd


_F8 = C.c_float * MAX_DIM


class ModelPOD(C.Structure):
    """glabc_model_t"""
    _fields_ = [("family", C.c_int32), ("theta_dim", C.c_int32), ("y_dim", C.c_int32), ("reserved", C.c_int32),
                ("y_obs", _F8), ("noise_loc", _F8), ("noise_scale", _F8), ("prior_loc", _F8),
                ("prior_log_scale", _F8), ("prior_scale", _F8),
                ("eps_log_scale", C.c_float), ("eps_scale", C.c_float), ("epsilon", C.c_double)]


class DistPOD(C.Structure):
    """glabc_dist_t"""
    _fields_ = [("kind", C.c_int32), ("dim", C.c_int32), ("n_modes", C.c_int32), ("reserved", C.c_int32),
                ("a", _F8), ("b", _F8), ("c", _F8),
                ("mix_loc", _F8 * MAX_MODES), ("mix_log_scale", _F8 * MAX_MODES), ("mix_scale", _F8 * MAX_MODES),
                ("mix_log_w", C.c_float * MAX_MODES), ("mix_w", C.c_float * MAX_MODES)]


class RunPOD(C.Structure):
    """glabc_run_t"""
    _fields_ = [("n_chains", C.c_int64), ("n_steps", C.c_int64), ("step_base", C.c_int64),
                ("chain_id_base", C.c_int64), ("seed", C.c_uint64), ("global_frequency", C.c_float),
                ("rng_mode", C.c_int32), ("arith_mode", C.c_int32), ("trace_layout", C.c_int32),
                ("write_row0", C.c_int32), ("block_threads", C.c_int32), ("n_candidates", C.c_int32),
                ("num_grad", C.c_int32), ("tau", C.c_float),
                ("trace_rows", C.c_int64), ("trace_chains", C.c_int64), ("trace_chain_off", C.c_int64),
                ("trace_row_base", C.c_int64),
                ("theta", C.c_void_p), ("y", C.c_void_p), ("aux", C.c_void_p), ("trace", C.c_void_p),
                ("stats", C.c_void_p), ("tape32", C.c_void_p), ("tape64", C.c_void_p), ("debug", C.c_void_p),
                ("tape_dump", C.c_void_p), ("tape64_dump", C.c_void_p),
                ("state64", C.c_void_p), ("tape_grad0", C.c_void_p), ("tape_grad0_dump", C.c_void_p),
                ("debug64", C.c_void_p), ("tau64", C.c_double), ("stream", C.c_void_p)]


class AglmcmcPOD(C.Structure):
    """glabc_aglmcmc_t"""
    _fields_ = [("step_size", C.c_int32), ("init", C.c_int32), ("alpha", C.c_float), ("hat_eps_T", C.c_float),
                ("kde_rule", C.c_int32), ("tape_rounds", C.c_int32),
                ("init_p", C.c_void_p), ("init_s", C.c_void_p), ("ad_idx", C.c_void_p), ("ad_noise", C.c_void_p),
                ("ad_sim", C.c_void_p), ("ad_rec", C.c_void_p), ("ad_blk", C.c_void_p), ("init_w", C.c_void_p),
                ("dump_rounds", C.c_int32), ("reserved", C.c_int32)]


class FlowPOD(C.Structure):
    """glabc_flow_t"""
    _fields_ = [("n_blocks", C.c_int32), ("hidden", C.c_int32), ("dim", C.c_int32), ("reserved", C.c_int32),
                ("w1", C.c_void_p), ("b1", C.c_void_p), ("w2", C.c_void_p), ("b2", C.c_void_p), ("w3", C.c_void_p),
                ("b3", C.c_void_p), ("base_loc", C.c_float * 2), ("base_log_scale", C.c_float * 2)]


class BlockIsirPOD(C.Structure):
    """glabc_block_isir_t"""
    _fields_ = [("step_size", C.c_int32), ("block", C.c_int32), ("blk_theta", C.c_void_p), ("blk_x", C.c_void_p),
                ("blk_w", C.c_void_p), ("blk_lq", C.c_void_p), ("kk", C.c_void_p), ("pending", C.c_void_p),
                ("next_step", C.c_void_p), ("lq_cur", C.c_void_p), ("lq_valid", C.c_void_p)]


USER_MAX_PARAMS, USER_MAX_NOISE = 64, 32
USER_SIMULATE, USER_PRIOR, USER_DISCREPANCY, USER_LOG_KERNEL = range(4)


class UserModelPOD(C.Structure):
    """glabc_user_model_t"""
    _fields_ = [("theta_dim", C.c_int32), ("y_dim", C.c_int32), ("n_noise", C.c_int32), ("n_params", C.c_int32),
                ("source", C.c_char_p), ("params", C.c_float * USER_MAX_PARAMS), ("epsilon", C.c_double)]


BW_SILVERMAN, BW_SCOTT = 0, 1
AG_REC_SLOTS = 8
AG_MAX_BLOCK = 4096


def fill(arr, values):
    values = [float(v) for v in values]
    if len(values) > len(arr):
        raise ValueError(f"at most {len(arr)} values fit, got {len(values)}")
    for i, v in enumerate(values):
        arr[i] = v


LIB_NAME = "libglabc.so"
_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GLABC_LIB") or os.path.join(_HERE, "csrc", LIB_NAME)  # GLABC_LIB: kernel-experiment builds

# every symbol include/glabc.h declares (tests/test_abi_symbols.py parses the header and checks)
_SIGNATURES = {
    "glabc_version": (C.c_int, []),
    "glabc_ctx_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "glabc_ctx_destroy": (C.c_int, [C.c_void_p]),
    "glabc_last_error": (C.c_char_p, [C.c_void_p]),
    "glabc_status_string": (C.c_char_p, [C.c_int]),
    "glabc_device_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "glabc_model_set": (C.c_int, [C.c_void_p, C.POINTER(ModelPOD), C.c_size_t]),
    "glabc_dist_set": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(DistPOD), C.c_size_t]),
    "glabc_model_prior_set": (C.c_int, [C.c_void_p, C.POINTER(DistPOD), C.c_size_t]),
    "glabc_dist_log_prob": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "glabc_dist_sample": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "glabc_run_global": (C.c_int, [C.c_void_p, C.POINTER(RunPOD)]),
    "glabc_run_global_user": (C.c_int, [C.c_void_p, C.POINTER(RunPOD), C.POINTER(UserModelPOD)]),
    "glabc_run_isir_user": (C.c_int, [C.c_void_p, C.POINTER(RunPOD), C.POINTER(UserModelPOD)]),
    "glabc_run_mala_user": (C.c_int, [C.c_void_p, C.POINTER(RunPOD), C.POINTER(UserModelPOD)]),
    "glabc_user_model_check": (C.c_int, [C.POINTER(UserModelPOD), C.c_int32, C.c_char_p, C.c_size_t]),
    "glabc_user_model_check_proposals": (C.c_int, [C.POINTER(UserModelPOD), C.c_int32, C.c_int32, C.c_int32, C.c_char_p, C.c_size_t]),
    "glabc_user_simulate": (C.c_int, [C.c_void_p, C.POINTER(UserModelPOD), C.c_void_p, C.c_int64, C.c_uint64, C.c_uint64,
                                      C.c_void_p, C.c_void_p]),
    "glabc_user_evaluate": (C.c_int, [C.c_void_p, C.POINTER(UserModelPOD), C.c_int32, C.c_void_p, C.c_int64, C.c_void_p,
                                      C.c_void_p]),
    "glabc_run_global_host": (C.c_int, [C.c_void_p, C.POINTER(RunPOD), C.c_int64]),
    "glabc_run_isir": (C.c_int, [C.c_void_p, C.POINTER(RunPOD)]),
    "glabc_run_isir_host": (C.c_int, [C.c_void_p, C.POINTER(RunPOD), C.c_int64]),
    "glabc_run_mala": (C.c_int, [C.c_void_p, C.POINTER(RunPOD)]),
    "glabc_run_mala_host": (C.c_int, [C.c_void_p, C.POINTER(RunPOD), C.c_int64]),
    "glabc_run_aglmcmc": (C.c_int, [C.c_void_p, C.POINTER(RunPOD), C.POINTER(AglmcmcPOD)]),
    "glabc_kde_fit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32,
                                C.c_void_p, C.c_void_p, C.c_void_p]),
    "glabc_kde_log_prob": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                     C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p]),
    "glabc_kde_sample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                   C.c_int32, C.c_int64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "glabc_run_block_isir": (C.c_int, [C.c_void_p, C.POINTER(RunPOD), C.POINTER(BlockIsirPOD)]),
    "glabc_block_weights": (C.c_int, [C.c_void_p, C.POINTER(RunPOD), C.POINTER(BlockIsirPOD), C.c_uint32]),
    "glabc_flow_set": (C.c_int, [C.c_void_p, C.POINTER(FlowPOD), C.c_size_t, C.c_void_p]),
    "glabc_flow_sample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "glabc_flow_log_prob": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "glabc_esjd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
    "glabc_expand_events": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_int32]),
    "glabc_run_aglmcmc_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
    "glabc_aglmcmc_state": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int64), C.c_int64, C.c_int32, C.c_int32, C.c_void_p]),
    "glabc_flow_precision": (C.c_int, [C.c_void_p, C.c_int32]),
    "glabc_flow_sample_native": (C.c_int, [C.c_void_p, C.c_uint64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "glabc_flow_param_count": (C.c_int64, [C.c_int32]),
    "glabc_flow_train_init": (C.c_int, [C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float]),
    "glabc_flow_grad": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "glabc_flow_adam_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "glabc_flow_train_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "glabc_flow_get": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "glabc_flow_train_state": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int64), C.c_int32, C.c_void_p]),
    "glabc_resample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    "glabc_summarize": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
    "glabc_philox_kat": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
}

_lib = None


class GlabcError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"glabc status {status}: {message}")
        self.status = status


def load(path=None):
    """dlopen libglabc.so and bind the signatures.  Loading needs no GPU; running does."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise ImportError(
            f"{p} is missing: the CUDA extension has not been built. Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). "
            "There is no CPU fallback.")
    lib = C.CDLL(p)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    if path is None:
        _lib = lib
    return lib


class Context:
    """glabc_ctx: one per (thread, device)."""

    def __init__(self, device=-1):
        self.lib = load()
        h = C.c_void_p()
        st = self.lib.glabc_ctx_create(int(device), C.byref(h))
        if st != OK:
            raise GlabcError(st, self.lib.glabc_status_string(st).decode() +
                             " — glabc needs a CUDA device (sm_100a); there is no CPU fallback")
        self.handle = h
        self.n_calls = 0          # status-checked C-ABI calls so far (bench.py reports kernel-launching calls from it)

    def check(self, st):
        self.n_calls += 1
        if st != OK:
            raise GlabcError(st, self.lib.glabc_last_error(self.handle).decode())

    def device_info(self):
        sm, khz, cc = C.c_int32(), C.c_int32(), C.c_int32()
        self.check(self.lib.glabc_device_info(self.handle, C.byref(sm), C.byref(khz), C.byref(cc)))
        return dict(sm_count=sm.value, clock_khz=khz.value, cc=cc.value)

    def close(self):
        if getattr(self, "handle", None):
            self.lib.glabc_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
