"""ctypes binding of include/honk2_b200.h.  There is no fallback: if the shared library is
missing or a call fails, a NativeError is raised."""
import ctypes as C
import os

from .build import LIB_PATH

KWS_FP32, KWS_BF16, KWS_BF16X3 = 0, 1, 2
PRECISIONS = {"fp32": KWS_FP32, "bf16": KWS_BF16, "bf16x3": KWS_BF16X3}
ABI_VERSION = 2


class NativeError(RuntimeError):
    pass


class ResNetConfig(C.Structure):
    _fields_ = [("n_layers", C.c_int), ("n_maps", C.c_int), ("use_dilation", C.c_int),
                ("pool_h", C.c_int), ("pool_w", C.c_int), ("n_labels", C.c_int)]


class ResNetWeights(C.Structure):
    _fields_ = [("conv0_w", C.c_void_p), ("conv_w", C.POINTER(C.c_void_p)),
                ("bn_mean", C.POINTER(C.c_void_p)), ("bn_var", C.POINTER(C.c_void_p)),
                ("out_w", C.c_void_p), ("out_b", C.c_void_p)]


class CnnConfig(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        "time", "freq", "conv0_out", "conv0_kh", "conv0_kw", "conv0_sh", "conv0_sw", "pool0_kh", "pool0_kw",
        "conv1_out", "conv1_kh", "conv1_kw", "conv1_sh", "conv1_sw", "pool1_kh", "pool1_kw",
        "lin0_out", "dnn0_out", "dnn1_out", "n_labels")]


class CnnWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "conv0_w", "conv0_b", "conv1_w", "conv1_b", "lin0_w", "lin0_b", "dnn0_w", "dnn0_b",
        "dnn1_w", "dnn1_b", "lin1_w", "lin1_b")]


# name -> (restype, argtypes); every symbol include/honk2_b200.h declares
SIGNATURES = {
    "kws_abi_version": (C.c_int, []),
    "kws_last_error": (C.c_char_p, []),
    "kws_device_info": (C.c_int, [C.POINTER(C.c_int)] * 3),
    "kws_frontend_create": (C.c_int, [C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_int,
                                      C.POINTER(C.c_void_p)]),
    "kws_frontend_destroy": (None, [C.c_void_p]),
    "kws_frontend_n_frames": (C.c_int, [C.c_void_p, C.c_int]),
    "kws_frontend_n_mels": (C.c_int, [C.c_void_p]),
    "kws_mfcc_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]),
    "kws_mfcc_forward_pcm16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]),
    "kws_mfcc_stream_scratch_bytes": (C.c_size_t, [C.c_void_p, C.c_int64, C.c_int, C.c_int]),
    "kws_mfcc_stream_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                          C.c_size_t, C.c_void_p]),
    "kws_mfcc_stream_forward_pcm16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p,
                                                C.c_void_p, C.c_size_t, C.c_void_p]),
    "kws_live_state_bytes": (C.c_size_t, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]),
    "kws_live_create": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "kws_live_destroy": (None, [C.c_void_p]),
    "kws_live_reset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "kws_live_push": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "kws_live_push_pcm16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "kws_live_cnn_state_bytes": (C.c_size_t, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]),
    "kws_live_cnn_create": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                      C.POINTER(C.c_void_p)]),
    "kws_live_cnn_destroy": (None, [C.c_void_p]),
    "kws_live_cnn_reset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "kws_live_cnn_push": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "kws_live_cnn_push_pcm16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "kws_live_cnn_ragged_workspace_bytes": (C.c_size_t, [C.c_void_p]),
    "kws_live_cnn_push_ragged": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_int64, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "kws_live_cnn_push_ragged_pcm16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                 C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_size_t,
                                                 C.c_void_p]),
    "kws_live_ragged_workspace_bytes": (C.c_size_t, [C.c_void_p]),
    "kws_live_push_ragged": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_int64, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "kws_live_push_ragged_pcm16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_int64, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "kws_resnet_create": (C.c_int, [C.POINTER(ResNetConfig), C.POINTER(C.c_void_p)]),
    "kws_resnet_set_weights": (C.c_int, [C.c_void_p, C.POINTER(ResNetWeights), C.c_void_p]),
    "kws_cnn_create": (C.c_int, [C.POINTER(CnnConfig), C.POINTER(C.c_void_p)]),
    "kws_cnn_set_weights": (C.c_int, [C.c_void_p, C.POINTER(CnnWeights), C.c_void_p]),
    "kws_model_destroy": (None, [C.c_void_p]),
    "kws_model_n_labels": (C.c_int, [C.c_void_p]),
    "kws_model_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int]),
    "kws_model_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                    C.c_void_p, C.c_size_t, C.c_void_p]),
    "kws_model_wave_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int]),
    "kws_model_forward_wave": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p,
                                         C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "kws_model_forward_wave_pcm16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p,
                                               C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "kws_model_last_launches": (C.c_int64, [C.c_void_p]),
    "kws_model_kernel_path": (C.c_char_p, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "kws_eval_accumulate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p]),
    "kws_model_set_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "kws_model_profile_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64),
                                         C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "kws_model_set_chunk": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "kws_acc_accumulate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p,
                                     C.c_void_p]),
}

_lib = None


def lib_path():
    return os.environ.get("HONK2_B200_LIB", LIB_PATH)


def load():
    """dlopen the native library and bind every declared symbol (raises if one is missing)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise NativeError(
            f"native library {path} is missing: run `python -m honk2_b200.build` (needs nvcc); "
            "honk2_b200 has no CPU or PyTorch fallback")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.kws_abi_version() != ABI_VERSION:
        raise NativeError(f"{path}: ABI version {lib.kws_abi_version()} != {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


def loaded():
    """The library if it has already been loaded, else None (never triggers a load)."""
    return _lib


def check(status, what):
    if status != 0:
        msg = load().kws_last_error()
        raise NativeError(f"{what} failed (status {status}): {msg.decode() if msg else '?'}")
