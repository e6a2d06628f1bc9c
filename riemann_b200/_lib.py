"""
ctypes binding of the C ABI in include/riemann_b200.h.

There is no CPU fallback: if the CUDA library is missing or cannot be loaded this
module raises ImportError on first use, and every host class fails loudly.
PyTorch tensors are used only as device-buffer handles (``tensor.data_ptr()``).
"""
import ctypes as C
import os

from .sampling_errors import ParameterError

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RIEMANN_B200_LIB") or os.path.join(_HERE, "libriemann_b200.so")   # env: kernel experiments

RMN_OK, RMN_ERR_PARAM, RMN_ERR_CUDA, RMN_ERR_UNSUPPORTED = 0, -1, -2, -3
CP_LANES = 16
CP_SLOT = dict(sel1=0, sel2=1, sel3=2, bd=3, s=4, du=5, n=6, acc=7, xi=8)
CP_NSLOT = 8 + CP_LANES
CP_NDIAG = 8
DIAG_HDR = 6
SMALL_D_MAX = 8
PRECISIONS = {"f64": 0, "tf32x3": 1, "tf32-metric": 2}


class Inject(C.Structure):
    _fields_ = [("d_xi", C.c_void_p), ("d_u", C.c_void_p), ("d_tape", C.c_void_p), ("d_usel", C.c_void_p)]


class Trace(C.Structure):
    _fields_ = [("first", C.c_int64), ("thin", C.c_int64), ("d_theta", C.c_void_p),
                ("d_logpost", C.c_void_p), ("d_k", C.c_void_p), ("d_cpx", C.c_void_p),
                ("d_cpv", C.c_void_p), ("d_sig", C.c_void_p), ("d_prop_logpost", C.c_void_p),
                ("d_accepted", C.c_void_p), ("d_logqratio", C.c_void_p), ("d_prop_theta", C.c_void_p),
                ("d_prop_k", C.c_void_p), ("d_prop_cpx", C.c_void_p), ("d_prop_cpv", C.c_void_p),
                ("d_prop_sig", C.c_void_p)]


_P = C.c_void_p
_PP = C.POINTER(C.c_void_p)
_D = C.c_double
_I = C.c_int
_L = C.c_int64

# name -> (restype, argtypes); every symbol include/riemann_b200.h declares
SIGNATURES = {
    "rmn_version": (_I, []),
    "rmn_last_error": (C.c_char_p, []),
    "rmn_model_gaussian_create": (_I, [_PP, _I, _P, _P, _P, _D]),
    "rmn_model_changepoint_create": (_I, [_PP, _I, _P, _P, _D, _D, _D, _I, _D, _D]),
    "rmn_model_logistic_create": (_I, [_PP, _L, _I, _P, _P, _D]),
    "rmn_model_destroy": (_I, [_P]),
    "rmn_model_dim": (_I, [_P]),
    "rmn_model_logpost": (_I, [_P, _I, _L, _P, _P, _P]),
    "rmn_model_grad": (_I, [_P, _L, _P, _P, _P]),
    "rmn_model_metric": (_I, [_P, _L, _P, _P, _P]),
    "rmn_model_cp_logpost": (_I, [_P, _I, _L, _P, _P, _P, _P, _P, _P]),
    "rmn_proposal_rw_create": (_I, [_PP, _I, _P, _I, _D]),
    "rmn_proposal_hmc_create": (_I, [_PP, _I, _D, _I, _P, _P, _P, _I, _D]),
    "rmn_proposal_pcn_create": (_I, [_PP, _I, _P, _P, _D]),
    "rmn_proposal_mmala_create": (_I, [_PP, _I, _D]),
    "rmn_proposal_changepoint_create": (_I, [_PP, _D, _P]),
    "rmn_proposal_destroy": (_I, [_P]),
    "rmn_sampler_workspace_bytes": (C.c_size_t, [_P, _P, _L]),
    "rmn_sampler_create": (_I, [_PP, _P, _P, _L, _L, C.c_uint64, _P, C.c_size_t]),
    "rmn_sampler_workspace_bytes_ex": (C.c_size_t, [_P, _P, _L, _I]),
    "rmn_sampler_create_ex": (_I, [_PP, _P, _P, _L, _L, C.c_uint64, _P, C.c_size_t, _I]),
    "rmn_sampler_destroy": (_I, [_P]),
    "rmn_sampler_set_state": (_I, [_P, _P, _P]),
    "rmn_sampler_get_state": (_I, [_P, _P, _P, _P]),
    "rmn_sampler_cp_set_state": (_I, [_P, _P, _P, _P, _P, _P]),
    "rmn_sampler_cp_get_state": (_I, [_P, _P, _P, _P, _P, _P, _P]),
    "rmn_sampler_run": (_I, [_P, _L, C.POINTER(Inject), C.POINTER(Trace), _P]),
    "rmn_sampler_get_adapt": (_I, [_P, _P, _P, _P, _P]),
    "rmn_sampler_set_adapt": (_I, [_P, _P, _P, _P, _P]),
    "rmn_sampler_get_step": (_L, [_P]),
    "rmn_sampler_set_step": (_I, [_P, _L]),
    "rmn_sampler_diag_dim": (_I, [_P]),
    "rmn_sampler_reset_diagnostics": (_I, [_P, _P]),
    "rmn_sampler_reduce_diagnostics": (_I, [_P, _P, _P]),
    "rmn_sampler_launch_count": (_L, [_P]),
    "rmn_sampler_chain_moments": (_I, [_P, _P, _P, _P]),
    "rmn_sampler_set_move_schedule": (_I, [_P, _I]),
    "rmn_sampler_cp_set_summary": (_I, [_P, _I, _P, _D, _D, _I, _L]),
    "rmn_sampler_cp_get_summary": (_I, [_P, _P, _P, _P, _P, _P]),
    "rmn_sampler_cp_set_rung_summary": (_I, [_P, _I, _I, _P, _D, _D, _I, _L]),
    "rmn_sampler_cp_get_swap_stats": (_I, [_P, _P, _P, _P, _P, _P, _P]),
    "rmn_sampler_set_tempering": (_I, [_P, _I, _P, _D]),
    "rmn_autocorr_tau": (_I, [_P, _L, _L, _L, _D, _P, _P, _P]),
    "rmn_nccl_unique_id": (_I, [_P, C.c_size_t]),
    "rmn_sampler_set_row_comm": (_I, [_P, _P, C.c_size_t, _I, _I]),
    "rmn_sampler_get_adaptcov": (_I, [_P, _P, _P]),
    "rmn_proposal_adaptcov_create": (_I, [_PP, _I, _P, _P, _D, _I, _I]),
    "rmn_proposal_set_scale_adapt": (_I, [_P, _I, _D]),
    "rmn_proposal_hmc_set_cov_adapt": (_I, [_P, _P, _P, _D, _I, _I]),
    "rmn_sampler_enable_kernel_timing": (_I, [_P, _I]),
    "rmn_sampler_kernel_timing": (_I, [_P, _P, _P, _P, _P]),
    "rmn_philox_raw": (_I, [_L, _P, _P, _P, _P]),
    "rmn_rng_draws": (_I, [C.c_uint64, _L, _L, _L, _I, _P, _P, _P]),
    "rmn_tf32x3_gemm": (_I, [_L, _I, _I, _P, _P, _P, _P, _P, _P]),
    "rmn_tf32_gemm": (_I, [_L, _I, _I, _P, _P, _P, _P]),
    "rmn_bf16_gemm": (_I, [_L, _I, _I, _P, _P, _P, _P]),
    "rmn_proposal_rw_set_pooled_cov_adapt": (_I, [_P, _L, _D, _D, _L]),
    "rmn_sampler_get_pooled_cov": (_I, [_P, _P, _P, _P, _P]),
    "rmn_tf32x3_gemm_splitk": (_I, [_L, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P]),
    "rmn_logistic_math": (_I, [_L, _P, _P, _P, _P, _P]),
}

_lib = None


def load():
    """Load the C-ABI library (no compute).  Raises ImportError if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "riemann_b200: CUDA library %s not found. Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). "
            "There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)       # AttributeError if a declared symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    """Map C status codes to exceptions (SURVEY.md section 8b error convention)."""
    if rc == RMN_OK:
        return
    msg = load().rmn_last_error().decode("utf-8", "replace")
    if rc in (RMN_ERR_PARAM, RMN_ERR_UNSUPPORTED):
        raise ParameterError(msg)
    raise RuntimeError("riemann_b200: " + msg)


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("riemann_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device (or host numpy) pointer as c_void_p; None -> NULL."""
    if t is None:
        return C.c_void_p(0)
    if hasattr(t, "data_ptr"):
        return C.c_void_p(t.data_ptr())
    return C.c_void_p(t.ctypes.data)
