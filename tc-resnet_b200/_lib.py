"""ctypes binding of libtcr_b200.so (include/tcr_b200.h).

The product path: there is NO CPU fallback.  If the CUDA library has not been built
(``python -c "import __graft_entry__ as g; g.build()"`` or ``make -C tc-resnet_b200/csrc``) importing
this module raises, and every wrapper raises ``TcrError`` on a non-zero status.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtcr_b200.so")

TCR_MODEL_TCRESNET8 = 8
TCR_MODEL_TCRESNET14 = 14
ABI_VERSION = 6          # TCR_ABI_VERSION of include/tcr_b200.h this binding was written against
TCR_INPUT_WAV_F32, TCR_INPUT_FEATURES, TCR_INPUT_WAV_PCM16 = 0, 1, 2
TCR_OPT_MOMENTUM, TCR_OPT_ADAM, TCR_OPT_RMSPROP = 0, 1, 2
TCR_FEATURE_MFCC = 0
TCR_FEATURE_LOG_MEL = 1
KIND_NAMES = {0: "weight", 1: "beta", 2: "gamma", 3: "moving_mean", 4: "moving_variance"}


class TcrError(RuntimeError):
    pass


class TcrConfig(C.Structure):
    _fields_ = [
        ("model", C.c_int32), ("width_multiplier", C.c_float), ("num_classes", C.c_int32),
        ("sample_rate", C.c_int32), ("clip_samples", C.c_int32), ("window_size_samples", C.c_int32),
        ("window_stride_samples", C.c_int32), ("num_mel_bins", C.c_int32), ("num_mfccs", C.c_int32),
        ("lower_edge_hertz", C.c_float), ("upper_edge_hertz", C.c_float), ("feature_kind", C.c_int32),
        ("max_batch", C.c_int32), ("bn_decay", C.c_float), ("bn_epsilon", C.c_float),
        ("dropout_keep_prob", C.c_float), ("label_smoothing", C.c_float), ("device", C.c_int32),
    ]


class TcrInfo(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("frames", C.c_int32), ("features", C.c_int32), ("fft_length", C.c_int32),
        ("num_conv_layers", C.c_int32), ("num_blocks", C.c_int32), ("last_channels", C.c_int32),
        ("last_frames", C.c_int32), ("num_trainable", C.c_int64), ("num_moving", C.c_int64),
        ("forward_flops_per_utt", C.c_int64), ("workspace_bytes", C.c_int64),
    ]


class TcrParamDesc(C.Structure):
    _fields_ = [
        ("name", C.c_char * 96), ("kind", C.c_int32), ("rank", C.c_int32), ("shape", C.c_int32 * 4),
        ("offset", C.c_int64), ("numel", C.c_int64),
    ]


class TcrKernelStat(C.Structure):
    _fields_ = [("name", C.c_char * 64), ("total_ms", C.c_double), ("launches", C.c_int64)]


class TcrDscnnConfig(C.Structure):
    _fields_ = [("size", C.c_int32), ("height", C.c_int32), ("width", C.c_int32), ("num_classes", C.c_int32),
                ("max_batch", C.c_int32), ("device", C.c_int32)]


class TcrStepArgs(C.Structure):
    _fields_ = [
        ("input", C.c_void_p), ("input_is_features", C.c_int32), ("onehot", C.c_void_p), ("n", C.c_int32),
        ("params", C.c_void_p), ("slots", C.c_void_p), ("moving", C.c_void_p),
        ("learning_rate", C.c_float), ("momentum", C.c_float), ("weight_decay", C.c_float),
        ("dropout_seed", C.c_uint64), ("dropout_mask", C.c_void_p), ("losses", C.c_void_p),
        ("logits", C.c_void_p), ("probs", C.c_void_p), ("grads", C.c_void_p), ("apply_update", C.c_int32),
        ("clips", C.c_void_p), ("background", C.c_void_p), ("pcm_stride", C.c_int64), ("input_resident", C.c_int32),
        # ABI v6: update rule (zero = momentum, as before)
        ("optimizer", C.c_int32), ("slots2", C.c_void_p), ("opt_scalars", C.c_void_p), ("beta1", C.c_float),
        ("beta2", C.c_float), ("epsilon", C.c_float), ("rms_decay", C.c_float), ("ema", C.c_void_p), ("ema_decay", C.c_float),
    ]


# Every symbol include/tcr_b200.h declares: (restype, argtypes)
SYMBOLS = {
    "tcr_abi_version": (C.c_int, []),
    "tcr_last_error": (C.c_char_p, []),
    "tcr_config_default": (C.c_int, [C.POINTER(TcrConfig)]),
    "tcr_create": (C.c_int, [C.POINTER(TcrConfig), C.POINTER(C.c_void_p)]),
    "tcr_destroy": (C.c_int, [C.c_void_p]),
    "tcr_get_info": (C.c_int, [C.c_void_p, C.POINTER(TcrInfo)]),
    "tcr_param_table": (C.c_int, [C.c_void_p, C.POINTER(C.POINTER(TcrParamDesc)), C.POINTER(C.c_int32)]),
    "tcr_init_variables": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "tcr_mfcc_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "tcr_mfcc_forward_pcm16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "tcr_set_background_samples": (C.c_int, [C.c_void_p, C.c_int64]),
    "tcr_augment_pcm16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "tcr_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                              C.c_uint64, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                              C.c_void_p]),
    "tcr_eval_accumulate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "tcr_comm_set_sync_bn": (C.c_int, [C.c_void_p, C.c_int32]),
    "tcr_train_step": (C.c_int, [C.c_void_p, C.POINTER(TcrStepArgs), C.c_void_p]),
    "tcr_train_step_host": (C.c_int, [C.c_void_p, C.POINTER(TcrStepArgs), C.c_int32, C.c_void_p, C.POINTER(C.c_float),
                                      C.POINTER(C.c_int64)]),
    "tcr_host_flush": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int64)]),
    "tcr_workspace_tensor": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "tcr_comm_unique_id": (C.c_int, [C.c_void_p]),
    "tcr_comm_init": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]),
    "tcr_comm_p2p_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tcr_comm_p2p_attach": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]),
    "tcr_comm_p2p_detach": (C.c_int, [C.c_void_p]),
    "tcr_comm_destroy": (C.c_int, [C.c_void_p]),
    "tcr_measure_fp32_peak": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.c_void_p]),
    "tcr_dscnn_create": (C.c_int, [C.POINTER(TcrDscnnConfig), C.POINTER(C.c_void_p)]),
    "tcr_dscnn_destroy": (C.c_int, [C.c_void_p]),
    "tcr_dscnn_param_table": (C.c_int, [C.c_void_p, C.POINTER(C.POINTER(TcrParamDesc)), C.POINTER(C.c_int32),
                                        C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "tcr_dscnn_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tcr_profile_enable": (C.c_int, [C.c_int]),
    "tcr_profile_read": (C.c_int, [C.POINTER(C.POINTER(TcrKernelStat)), C.POINTER(C.c_int32)]),
    "tcr_launch_count": (C.c_int, [C.POINTER(C.c_uint64)]),
}


def load(path: str | None = None) -> C.CDLL:
    """dlopen the C-ABI library and set prototypes.  Raises if the file or any symbol is missing."""
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise TcrError(
            f"{path} not found: the CUDA library has not been built. Run `make -C tc-resnet_b200/csrc` "
            "(or __graft_entry__.build()). There is no CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)      # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    if lib.tcr_abi_version() != ABI_VERSION:
        raise TcrError(f"ABI version mismatch: library {lib.tcr_abi_version()}, binding {ABI_VERSION}")
    return lib


def check(lib: C.CDLL, status: int, what: str) -> None:
    if status != 0:
        msg = lib.tcr_last_error()
        raise TcrError(f"{what} failed (status {status}): {msg.decode() if msg else ''}")
