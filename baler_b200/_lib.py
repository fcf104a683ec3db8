"""ctypes binding of libbaler_b200.so (the C ABI declared in include/baler_b200.h).

There is no CPU fallback: if the library is missing or no CUDA device is present every compute
entry point raises.  Build with `python -m baler_b200.build` (or `__graft_entry__.build()`).
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libbaler_b200.so")

BB_F32, BB_F16, BB_F64 = 0, 1, 2
BB_ACT_NONE, BB_ACT_LEAKY, BB_ACT_RELU = 0, 1, 2
BB_PREC_AUTO, BB_PREC_FP32, BB_PREC_SPLIT16, BB_PREC_FAST16, BB_PREC_FP64 = 0, 1, 2, 3, 4
PRECISIONS = {"auto": BB_PREC_AUTO, "exact": BB_PREC_AUTO, "fp32": BB_PREC_FP32,
              "split16": BB_PREC_SPLIT16, "fast": BB_PREC_FAST16, "fast16": BB_PREC_FAST16, "fp64": BB_PREC_FP64}


class BalerB200Error(RuntimeError):
    def __init__(self, code, what):
        super().__init__("%s failed: %s (code %d)" % (what, _lib().bb_strerror(code).decode(), code))
        self.code = code


class TrainHyper(C.Structure):
    _fields_ = [("lr", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double),
                ("reg_param", C.c_double), ("l1", C.c_int), ("world_size", C.c_int)]


_P = C.c_void_p
_PP = C.POINTER(C.c_void_p)
_SIGNATURES = {
    "bb_version": (C.c_int, []),
    "bb_strerror": (C.c_char_p, [C.c_int]),
    "bb_ctx_create": (C.c_int, [C.c_int, _PP]),
    "bb_ctx_destroy": (C.c_int, [_P]),
    "bb_ctx_sm_count": (C.c_int, [_P]),
    "bb_model_create_dense": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, C.c_int, _P, _P, _P, _P, _PP]),
    "bb_model_destroy": (C.c_int, [_P]),
    "bb_model_trim": (C.c_int, [_P]),
    "bb_host_convert": (C.c_int, [_P, C.c_int, _P, C.c_int, C.c_int64]),
    "bb_host_colminmax_f32": (C.c_int, [_P, C.c_int64, C.c_int, _P, _P]),
    "bb_model_n_features": (C.c_int, [_P]),
    "bb_model_z_dim": (C.c_int, [_P]),
    "bb_model_auto_precision": (C.c_int, [_P]),
    "bb_model_chain_precision": (C.c_int, [_P, C.c_int]),
    "bb_model_range_flag": (C.c_int, [_P, C.c_int, C.POINTER(C.c_int)]),
    "bb_colminmax_f32": (C.c_int, [_P, _P, C.c_int64, C.c_int, _P, _P, _P]),
    "bb_colminmax_f64": (C.c_int, [_P, _P, C.c_int64, C.c_int, _P, _P, _P]),
    "bb_normalize_f32": (C.c_int, [_P, _P, C.c_int64, C.c_int, _P, _P, _P, _P]),
    "bb_normalize_f64": (C.c_int, [_P, _P, C.c_int64, C.c_int, _P, _P, _P, _P]),
    "bb_renormalize_f32": (C.c_int, [_P, _P, C.c_int64, C.c_int, _P, _P, _P, _P]),
    "bb_encode_f32": (C.c_int, [_P, _P, C.c_int64, _P, _P, _P, C.c_int, C.c_int, _P]),
    "bb_decode_f32": (C.c_int, [_P, _P, C.c_int, C.c_int64, _P, _P, _P, C.c_int, _P]),
    "bb_encode_f64": (C.c_int, [_P, _P, C.c_int64, _P, _P, _P, _P]),
    "bb_decode_f64": (C.c_int, [_P, _P, C.c_int64, _P, _P, _P, _P]),
    "bb_compress_host": (C.c_int, [_P, _P, C.c_int64, _P, C.c_int, _P, C.c_int, C.c_int]),
    "bb_decompress_host": (C.c_int, [_P, _P, C.c_int, C.c_int64, _P, _P, C.c_int, C.c_int]),
    "bb_compress_host_f64": (C.c_int, [_P, _P, C.c_int64, _P, C.c_int, _P]),
    "bb_decompress_host_f64": (C.c_int, [_P, _P, C.c_int64, _P, _P]),
    "bb_latent_quantize_q8": (C.c_int, [_P, _P, C.c_int64, C.c_int, _P, _P, _P, _P]),
    "bb_latent_dequantize_q8": (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int, _P, _P]),
    "bb_compress_host_q8": (C.c_int, [_P, _P, C.c_int64, _P, C.c_int, _P, _P, _P, C.c_int]),
    "bb_decompress_host_q8": (C.c_int, [_P, _P, _P, _P, C.c_int64, _P, _P, C.c_int, C.c_int]),
    "bb_latent_quantize_packed": (C.c_int, [_P, _P, C.c_int64, C.c_int, C.c_int, _P, _P, _P, _P]),
    "bb_latent_dequantize_packed": (C.c_int, [_P, C.c_int, _P, _P, _P, C.c_int64, C.c_int, _P, _P]),
    "bb_compress_host_packed": (C.c_int, [_P, _P, C.c_int64, _P, C.c_int, C.c_int, _P, _P, _P, C.c_int]),
    "bb_decompress_host_packed": (C.c_int, [_P, C.c_int, _P, _P, _P, C.c_int64, _P, _P, C.c_int, C.c_int]),
    "bb_trainer_create": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, C.c_int, _PP]),
    "bb_trainer_create_dbn": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, _P, C.c_int, _PP]),
    "bb_trainer_set_dropout": (C.c_int, [_P, C.c_uint64, _P]),
    "bb_trainer_get_bn": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "bb_trainer_bn_running_dev": (C.c_int, [_P, _PP, _PP, C.POINTER(C.c_int)]),
    "bb_trainer_bn_running_dev_f64": (C.c_int, [_P, _PP, _PP, C.POINTER(C.c_int)]),
    "bb_trainer_set_dropout_mt19937": (C.c_int, [_P, _P, C.c_int]),
    "bb_trainer_get_dropout_mt19937": (C.c_int, [_P, _P, C.POINTER(C.c_int)]),
    "bb_trainer_destroy": (C.c_int, [_P]),
    "bb_trainer_set_precision": (C.c_int, [_P, C.c_int]),
    "bb_trainer_precision": (C.c_int, [_P]),
    "bb_trainer_range_flag": (C.c_int, [_P, C.c_int, C.POINTER(C.c_int)]),
    "bb_trainer_debug_layer": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, C.c_int]),
    "bb_trainer_profile": (C.c_int, [_P, C.c_int, _P]),
    "bb_trainer_dp_export": (C.c_int, [_P, C.c_int, _P]),
    "bb_trainer_dp_connect": (C.c_int, [_P, C.c_int, C.c_int, _P]),
    "bb_trainer_param_count": (C.c_int, [_P]),
    "bb_trainer_params_dev": (_P, [_P]),
    "bb_trainer_grads_dev": (_P, [_P]),
    "bb_trainer_params_dev_f64": (_P, [_P]),
    "bb_trainer_grads_dev_f64": (_P, [_P]),
    "bb_trainer_get_params": (C.c_int, [_P, _P, _P]),
    "bb_trainer_step": (C.c_int, [_P, _P, C.c_int, C.POINTER(TrainHyper), C.c_int, _P, _P]),
    "bb_trainer_epoch": (C.c_int, [_P, _P, C.c_int64, C.c_int, C.POINTER(TrainHyper), C.POINTER(C.c_double), _P]),
    "bb_trainer_validate": (C.c_int, [_P, _P, C.c_int64, C.c_int, C.POINTER(C.c_double), _P]),
    "bb_trainer_step_f64": (C.c_int, [_P, _P, C.c_int, C.POINTER(TrainHyper), C.c_int, _P, _P]),
    "bb_trainer_epoch_f64": (C.c_int, [_P, _P, C.c_int64, C.c_int, C.POINTER(TrainHyper), C.POINTER(C.c_double), _P]),
    "bb_trainer_validate_f64": (C.c_int, [_P, _P, C.c_int64, C.c_int, C.POINTER(C.c_double), _P]),
    "bb_trainer_epoch_host": (C.c_int, [_P, _P, C.c_int, C.c_int64, C.c_int, C.POINTER(TrainHyper), C.c_int64,
                                        C.POINTER(C.c_double), _P]),
    "bb_trainer_validate_host": (C.c_int, [_P, _P, C.c_int, C.c_int64, C.c_int, C.c_int64, C.POINTER(C.c_double), _P]),
    "bb_ltrainer_epoch_host": (C.c_int, [_P, _P, C.c_int, C.c_int64, C.c_int, C.POINTER(TrainHyper), C.c_int64,
                                         C.POINTER(C.c_double), _P]),
    "bb_ltrainer_validate_host": (C.c_int, [_P, _P, C.c_int, C.c_int64, C.c_int, C.c_int64, C.POINTER(C.c_double), _P]),
    "bb_trainer_activation_means": (C.c_int, [_P, _P]),
    "bb_mse_sum_f32": (C.c_int, [_P, _P, _P, C.c_int64, _P, _P]),
    "bb_error_bounded_deltas_f32": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int, _P, _P, C.c_double, C.c_int64, C.c_int64, _P, _P, _P, _P, _P]),
    "bb_ltrainer_create": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, C.c_int, _PP]),
    "bb_ltrainer_create_ex": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int, C.c_int, _PP]),
    "bb_ltrainer_get_bn": (C.c_int, [_P, _P]),
    "bb_ltrainer_bn_running_dev": (_P, [_P, C.POINTER(C.c_int)]),
    "bb_ltrainer_destroy": (C.c_int, [_P]),
    "bb_ltrainer_param_count": (C.c_int, [_P]),
    "bb_ltrainer_params_dev": (_P, [_P]),
    "bb_ltrainer_grads_dev": (_P, [_P]),
    "bb_ltrainer_get_params": (C.c_int, [_P, _P, _P]),
    "bb_ltrainer_step": (C.c_int, [_P, _P, C.c_int, C.POINTER(TrainHyper), C.c_int, _P, _P]),
    "bb_ltrainer_step_swae": (C.c_int, [_P, _P, C.c_int, C.POINTER(TrainHyper), C.c_int, _P, _P, C.c_int, C.c_int, C.c_float, _P, _P]),
    "bb_ltrainer_epoch": (C.c_int, [_P, _P, C.c_int64, C.c_int, C.POINTER(TrainHyper), C.POINTER(C.c_double), _P]),
    "bb_ltrainer_validate": (C.c_int, [_P, _P, C.c_int64, C.c_int, C.POINTER(C.c_double), _P]),
    "bb_ltrainer_create_dbn": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, _P, C.c_int, _PP]),
    "bb_ltrainer_set_dropout": (C.c_int, [_P, C.c_uint64, _P]),
    "bb_ltrainer_bn_batches_tracked": (C.c_int, [_P, _P]),
    "bb_ltrainer_activation_means": (C.c_int, [_P, _P]),
}

_handle = None


def _lib():
    global _handle
    if _handle is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "baler_b200: %s is missing - build it with `python -m baler_b200.build`; "
                "there is no CPU fallback" % LIB_PATH)
        h = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(h, name)
            fn.restype, fn.argtypes = res, args
        _handle = h
    return _handle


def lib():
    return _lib()


def check(code, what):
    if code != 0:
        raise BalerB200Error(code, what)


def exported_symbols():
    """names bound here; tests check them against include/baler_b200.h and the built .so"""
    return sorted(_SIGNATURES)
