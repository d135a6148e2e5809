"""ctypes binding of libpgmorl_b200.so (C ABI: include/pgmorl_b200.h).

There is no CPU fallback: if the library is missing or a call fails, this raises.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PGM_LIB_PATH", os.path.join(HERE, "libpgmorl_b200.so"))

_lib = None


class PgmError(RuntimeError):
    pass


class PpoHyper(C.Structure):
    """pgm_ppo_hyper; defaults = the reference's injected PPO flags (morl/run.py:56-70)."""
    _fields_ = [("clip_param", C.c_double), ("value_loss_coef", C.c_double),
                ("entropy_coef", C.c_double), ("max_grad_norm", C.c_double),
                ("beta1", C.c_double), ("beta2", C.c_double), ("adam_eps", C.c_double)]

    def __init__(self, clip_param=0.2, value_loss_coef=0.5, entropy_coef=0.0, max_grad_norm=0.5,
                 beta1=0.9, beta2=0.999, adam_eps=1e-5):
        super().__init__(clip_param, value_loss_coef, entropy_coef, max_grad_norm, beta1, beta2, adam_eps)


_P = C.c_void_p
_I = C.c_int
_Z = C.c_size_t
_F = C.c_float

# name -> (restype, argtypes); every symbol include/pgmorl_b200.h declares
SIGNATURES = {
    "pgm_abi_version": (_I, []),
    "pgm_last_error": (C.c_char_p, []),
    "pgm_n_par": (_I, [_I, _I, _I]),
    "pgm_param_offsets": (_I, [_I, _I, _I, _P]),
    "pgm_n_par_h": (_I, [_I, _I, _I, _I]),
    "pgm_param_offsets_h": (_I, [_I, _I, _I, _I, _P]),
    "pgm_policy_forward_f32": (_I, [_P, _P, _P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "pgm_policy_step_f32": (_I, [_P, _P, _P, _P, _I, _P, _Z, _P, _Z, _P, _Z, _P, _Z, _P, _I, _I, _I, _I, _I, _P]),
    "pgm_policy_forward_h_f32": (_I, [_P, _P, _P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "pgm_policy_step_h_f32": (_I, [_P, _P, _P, _P, _I, _P, _Z, _P, _Z, _P, _Z, _P, _Z, _P, _I, _I, _I, _I, _I, _I, _P]),
    "pgm_gae_adv_f32": (_I, [_P, _P, _P, _P, _P, _P, _F, _F, _P, _P, _I, _I, _I, _I, _P]),
    "pgm_returns_adv_f32": (_I, [_P, _P, _P, _P, _P, _P, _P, _F, _F, _I, _P, _P, _I, _I, _I, _I, _P]),
    "pgm_ppo_workspace_bytes": (_Z, [_I, _I, _I, _I, _I, _I]),
    "pgm_ppo_update_f32": (_I, [_P, _P, _P, _P, _P, _P, _Z, _P, _P, _P, _Z, _P, _P, _P, _I, _I, _I,
                                C.POINTER(PpoHyper), _P, _P, _Z, _I, _I, _I, _I, _I, _I, _P]),
    "pgm_fit_hyperbolic_f64": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _P]),
    "pgm_fit_neighbours_workspace_bytes": (_Z, [_I, _I, _I, _I]),
    "pgm_fit_neighbours_f64": (_I, [_P, _I, _I, _P, _I, _P, _P, _I, _I, _P, _P, _P, _P, _Z, _P]),
    "pgm_fit_gather_f64": (_I, [_P, _P, _I, _I, _I, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P]),
    "pgm_ep_filter_f64": (_I, [_P, _I, _I, _P, _P, _P]),
    "pgm_front_metrics_f64": (_I, [_P, _I, _I, _P, _P, _Z, _P]),
    "pgm_select_workspace_bytes": (_Z, [_I, _I, _I, _I]),
    "pgm_select_greedy_f64": (_I, [_P, _I, _P, _I, _I, C.c_double, _I, _P, _P, _P, _P, _P, _P, _Z, _P]),
    "pgm_vecnorm_step_f64": (_I, [_P] * 14 + [_P, _Z, _P, _Z, _P, _Z] + [C.c_double] * 4 + [_I] * 6 + [_P]),
    "pgm_vecnorm_rollout_step_f64": (_I, [_P] * 16 + [_P, _Z, _P, _Z, _P, _Z, _P, _Z] + [C.c_double] * 4 + [_I] * 5 + [_P]),
    "pgm_ppo_grad_f32": (_I, [_P, _P, _Z, _P, _P, _P, _Z, _P, _P, _P, _I, C.POINTER(PpoHyper), _P, _P, _P,
                              _Z, _I, _I, _I, _I, _I, _I, _P]),
    "pgm_ppo_workspace_bytes_h": (_Z, [_I, _I, _I, _I, _I, _I, _I]),
    "pgm_ppo_update_h_f32": (_I, [_P, _P, _P, _P, _P, _P, _Z, _P, _P, _P, _Z, _P, _P, _P, _I, _I, _I,
                                  C.POINTER(PpoHyper), _P, _P, _Z, _I, _I, _I, _I, _I, _I, _I, _P]),
    "pgm_ppo_grad_h_f32": (_I, [_P, _P, _Z, _P, _P, _P, _Z, _P, _P, _P, _I, C.POINTER(PpoHyper), _P, _P, _P,
                                _Z, _I, _I, _I, _I, _I, _I, _I, _P]),
    "pgm_n_par_x": (_I, [_I, _I, _I, _I, _I]),
    "pgm_param_offsets_x": (_I, [_I, _I, _I, _I, _I, _P]),
    "pgm_policy_forward_x_f32": (_I, [_P, _P, _P, _I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "pgm_policy_step_x_f32": (_I, [_P, _P, _P, _P, _I, _P, _Z, _P, _Z, _P, _Z, _P, _Z, _P, _I, _I, _I, _I, _I, _I, _I,
                                   _P]),
    "pgm_ppo_workspace_bytes_x": (_Z, [_I, _I, _I, _I, _I, _I, _I, _I]),
    "pgm_ppo_update_x_f32": (_I, [_P, _P, _P, _P, _P, _P, _Z, _P, _P, _P, _Z, _P, _P, _P, _I, _I, _I,
                                  C.POINTER(PpoHyper), _P, _P, _Z, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "pgm_ppo_grad_x_f32": (_I, [_P, _P, _Z, _P, _P, _P, _Z, _P, _P, _P, _I, C.POINTER(PpoHyper), _P, _P, _P,
                                _Z, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "pgm_front_metrics_x_f64": (_I, [_P, _I, _I, _I, _P, _P, _Z, _P]),
    "pgm_select_workspace_bytes_x": (_Z, [_I, _I, _I, _I, _I]),
    "pgm_select_greedy_x_f64": (_I, [_P, _I, _P, _I, _I, C.c_double, _I, _I, _P, _P, _P, _P, _P, _P, _Z, _P]),
}


# diagnostics library (include/pgmorl_b200_diag.h): tcgen05 self-test / layout probe / MMA pacing; tests and profiles only
DIAG_LIB_PATH = os.environ.get("PGM_DIAG_LIB_PATH", os.path.join(HERE, "libpgmorl_b200_diag.so"))
DIAG_SIGNATURES = {
    "pgm_tc_selftest": (_I, [_P, _I, _P]),
    "pgm_tc_mma_bench": (_I, [_P] + [_I] * 8 + [_P]),
    "pgm_tc_layout_probe": (_I, [_P] + [_I] * 19 + [_P]),
    "pgm_ffma2_burn": (_I, [_P, _I, _I, _P]),
}
_diag = None


def diag_lib():
    """Load (once) the diagnostics library. Not used by the product path."""
    global _diag
    if _diag is None:
        if not os.path.exists(DIAG_LIB_PATH):
            raise PgmError(f"{DIAG_LIB_PATH} is missing: build it with `python -m pgmorl_b200.build`")
        l = C.CDLL(DIAG_LIB_PATH)
        for name, (res, args) in DIAG_SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype, fn.argtypes = res, args
        l.pgm_last_error.restype = C.c_char_p
        _diag = l
    return _diag


def check_diag(rc):
    if rc != 0:
        raise PgmError(f"pgmorl_b200 (diag) error {rc}: {diag_lib().pgm_last_error().decode()}")


def lib():
    """Load (once) and return the shared library with typed entry points."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PgmError(
            f"{LIB_PATH} is missing: build it with `python -m pgmorl_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback for the MOPG / selection path.")
    l = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(l, name)       # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    if l.pgm_abi_version() != 1:
        raise PgmError("libpgmorl_b200.so ABI version mismatch")
    _lib = l
    return l


def check(rc):
    if rc != 0:
        raise PgmError(f"pgmorl_b200 error {rc}: {lib().pgm_last_error().decode()}")


def ptr(t):
    """Device/host pointer of a torch tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())
