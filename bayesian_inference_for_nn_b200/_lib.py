"""ctypes binding of libpyesian_b200.so (the C ABI in include/pyesian_b200.h).

There is no CPU fallback: if the shared library is missing or the device is not a B200-class GPU
the product path raises.  Nothing here imports torch, TensorFlow or the oracle.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libpyesian_b200.so")

# enums (values mirror include/pyesian_b200.h)
ACT_LINEAR, ACT_RELU, ACT_SOFTMAX, ACT_TANH, ACT_SIGMOID = 0, 1, 2, 3, 4
LOSS_SPARSE_CE, LOSS_MSE = 0, 1
MEM_HOST, MEM_DEVICE = 0, 1
PRIOR_SCALAR, PRIOR_PER_VARIABLE, PRIOR_PER_ELEMENT = 0, 1, 2
HMC_REFERENCE, HMC_CANONICAL = 0, 1
SVGD_REFERENCE_LIVE, SVGD_CANONICAL_MEDIAN = 0, 1
SG_SGLD, SG_SWAG = 0, 1
UQ_CANONICAL, UQ_REFERENCE = 0, 1
PATH_AUTO, PATH_GENERIC, PATH_FUSED_SMALL, PATH_TENSOR = 0, 1, 2, 3


class PyesianB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libpyesian_b200 error %d: %s" % (code, msg))
        self.code = code


class ModelDesc(C.Structure):
    _fields_ = [("n_layers", C.c_int32), ("in_dim", C.c_int32), ("units", C.POINTER(C.c_int32)),
                ("activation", C.POINTER(C.c_int32)), ("use_bias", C.POINTER(C.c_int32))]


class HmcDiag(C.Structure):
    _fields_ = [("mean_loss", C.c_double), ("accept_rate", C.c_double), ("n_accepted", C.c_int64),
                ("n_total", C.c_int64), ("n_nan", C.c_int64), ("grad_evals", C.c_int64),
                ("device_ms", C.c_double), ("kernel_launches", C.c_int64)]


_P = C.c_void_p
_f32p, _f64p, _i32p = C.c_void_p, C.c_void_p, C.c_void_p   # raw addresses (numpy .ctypes.data or device ptr)

# name -> (argtypes); every function returns int except pyb_last_error
SIGNATURES = {
    "pyb_version": [],
    "pyb_device_count": [C.POINTER(C.c_int32)],
    "pyb_create": [C.POINTER(ModelDesc), C.c_int32, C.c_uint64, C.POINTER(_P)],
    "pyb_destroy": [_P],
    "pyb_param_count": [_P, C.POINTER(C.c_int64)],
    "pyb_set_option": [_P, C.c_char_p, C.c_double],
    "pyb_get_info": [_P, C.c_char_p, C.POINTER(C.c_double)],
    "pyb_set_dataset": [_P, _f32p, C.c_int64, C.c_void_p, C.c_int32, C.c_int32, C.c_int64],
    "pyb_set_prior_gaussian": [_P, _f32p, _f32p, C.c_int32],
    "pyb_hmc_init": [_P, C.c_int64, C.c_int64, C.c_double, C.c_double, C.c_int32, C.c_int32, _f32p],
    "pyb_hmc_inject": [_P, _f32p, _f32p],
    "pyb_hmc_run": [_P, C.c_int32, C.c_int32, C.c_int32, C.POINTER(HmcDiag)],
    "pyb_hmc_eval": [_P, _f32p, C.c_int64, _f32p, _f32p, _f32p],
    "pyb_hmc_get_state": [_P, _f32p, _f32p],
    "pyb_hmc_last": [_P, _f32p, _f32p, _f32p, _f32p, _f32p, _i32p, _f32p],
    "pyb_hmc_reset_samples": [_P],
    "pyb_hmc_sample_count": [_P, C.POINTER(C.c_int64)],
    "pyb_hmc_samples": [_P, _f32p, _i32p, _i32p],
    "pyb_hmc_adapt_begin": [_P, C.c_double],
    "pyb_hmc_adapt_end": [_P],
    "pyb_hmc_step_sizes": [_P, _f64p],
    "pyb_hmc_set_step_sizes": [_P, _f64p],
    "pyb_hmc_set_temperatures": [_P, _f64p, C.c_int32],
    "pyb_hmc_tempering_stats": [_P, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p],
    "pyb_hmc_last_swaps": [_P, _f32p, _i32p],
    "pyb_hmc_track_predictive": [_P, _f32p, C.c_int64, _i32p],
    "pyb_hmc_predictive_sums": [_P, _f64p, _f64p, C.POINTER(C.c_int64)],
    "pyb_hmc_predictive_finish": [_P, _f64p, _f64p, C.c_int64, C.c_int64, C.c_int32, C.c_double, _f32p, _f32p, _f32p,
                                  _f32p, _f32p, _f32p],
    "pyb_hmc_track_params": [_P, C.c_int64, C.c_int32],
    "pyb_hmc_param_sums": [_P, _f64p, C.POINTER(C.c_int64)],
    "pyb_hmc_param_finish": [_P, _f64p, C.c_int64, C.c_int64, C.c_int64, C.c_int32, _f64p, _f64p, _f64p, _f64p, _f64p],
    "pyb_svgd_init": [_P, C.c_int64, C.c_int64, C.c_double, C.c_int32, _f64p],
    "pyb_svgd_step": [_P, _i32p, C.c_int64, C.POINTER(C.c_double)],
    "pyb_svgd_phi": [_P, _f64p, _f32p, C.c_int64, C.c_int32, _f32p, C.POINTER(C.c_double)],
    "pyb_svgd_get_particles": [_P, _f64p],
    "pyb_svgd_set_validation": [_P, _f32p, C.c_void_p, C.c_int64],
    "pyb_svgd_validation_loss": [_P, C.POINTER(C.c_double), _f32p],
    "pyb_svgd_set_comm": [_P, C.c_int32, C.c_int32, C.c_void_p],
    "pyb_set_comm": [_P, C.c_int32, C.c_int32, C.c_void_p],
    "pyb_nccl_unique_id": [C.c_void_p],
    "pyb_sg_init": [_P, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _f32p, C.c_int32],
    "pyb_sg_step": [_P, _i32p, C.c_int64, C.c_double, _f32p, _f32p, C.POINTER(C.c_double)],
    "pyb_sg_get": [_P, _f32p, _f32p, _f32p, _f32p, C.POINTER(C.c_int32), C.POINTER(C.c_int64)],
    "pyb_predict": [_P, _f32p, C.c_int64, _f32p, _f32p, C.c_int64, _f32p, _f32p, _f32p],
    "pyb_predict_uncertainty": [_P, _f32p, C.c_int64, _f32p, _f32p, C.c_int64, _i32p, C.c_int32, C.c_double, _f32p, _f32p,
                                _f32p, _f32p],
    "pyb_buffer_create": [_P, C.c_void_p, C.c_int64, C.POINTER(C.c_void_p)],
    "pyb_buffer_destroy": [_P, C.c_void_p],
    "pyb_gather_rows": [_P, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p],
    "pyb_debug_tc_gemm": [_P, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p],
    "pyb_debug_relu_mask": [_P, C.c_int64, C.c_void_p],
}

_lib = None


def load():
    """Load the shared library (once).  Raises if it has not been built — no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libpyesian_b200.so is not built (%s). Run `python -m bayesian_inference_for_nn_b200.build`. "
            "There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = C.c_int
    lib.pyb_last_error.argtypes = []
    lib.pyb_last_error.restype = C.c_char_p
    _lib = lib
    return lib


def check(status):
    if status != 0:
        msg = load().pyb_last_error()
        raise PyesianB200Error(status, msg.decode("utf-8", "replace") if msg else "")


def preload_nccl():
    """Map libnccl.so.2 into the process (RTLD_GLOBAL) so the library's dlopen-by-soname finds it.
    torch already does this when it is imported; otherwise use the copy bundled with the CUDA wheels."""
    import glob
    import sys
    if "torch" in sys.modules:
        return True
    for base in sys.path:
        for cand in glob.glob(os.path.join(base, "nvidia", "nccl", "lib", "libnccl.so.2")):
            try:
                C.CDLL(cand, mode=C.RTLD_GLOBAL)
                os.environ.setdefault("PYB_NCCL_LIB", cand)
                return True
            except OSError:
                pass
    return False


def nccl_unique_id() -> bytes:
    preload_nccl()
    buf = C.create_string_buffer(128)
    check(load().pyb_nccl_unique_id(buf))
    return buf.raw


def device_count():
    n = C.c_int32(0)
    check(load().pyb_device_count(C.byref(n)))
    return n.value
