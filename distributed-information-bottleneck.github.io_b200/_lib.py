"""ctypes binding of libdib_b200.so (include/dib_b200.h).  There is deliberately NO fallback: if the CUDA
library is missing or no B200 is visible, every compute entry point raises."""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int32, c_int64, c_size_t, c_uint32, c_uint64, c_void_p

from . import build as _build

ABI_VERSION = 2

ACTIVATIONS = {None: 0, "linear": 0, "relu": 1, "tanh": 2, "leaky_relu": 3, "sigmoid": 4, "elu": 5}
LOSSES = {"bce_logits": 0, "sparse_ce_logits": 1, "mse": 2, "external": 3, "bce_probs": 4, "infonce": 5}
# similarity_type of utils.get_scaled_similarity (utils.py:127-175) -> the `kind` of the InfoNCE entry points
SIMILARITIES = {"l2sq": 0, "l2": 1, "l1": 2, "linf": 3, "cosine": 4}
ENCODER_KINDS = {"mlp": 0, "simple": 1}
# 'fp16' / 'bf16': fused 16-bit-operand tcgen05 kernels (fp32 accumulate); 'tf32': kind::tf32 GEMMs on fp32 storage;
# 'fp32': exact CUDA-core FMA parity path.  See enum dib_precision in include/dib_b200.h.
PRECISIONS = {"fp32": 0, "tf32": 1, "bf16": 2, "fp16": 3}


class DibConfig(ctypes.Structure):
    _fields_ = [
        ("abi_version", c_int32),
        ("number_features", c_int32),
        ("feature_dimensionalities", POINTER(c_int32)),
        ("number_encoder_layers", c_int32),
        ("feature_encoder_architecture", POINTER(c_int32)),
        ("number_integration_layers", c_int32),
        ("integration_network_architecture", POINTER(c_int32)),
        ("output_dimensionality", c_int32),
        ("use_positional_encoding", c_int32),
        ("number_positional_encoding_frequencies", c_int32),
        ("activation_fn", c_int32),
        ("leaky_relu_alpha", c_float),
        ("feature_embedding_dimension", c_int32),
        ("output_activation_fn", c_int32),
        ("loss", c_int32),
        ("precision", c_int32),
        ("max_batch", c_int64),
        ("logvar_offset", c_float),
        ("kl_loss_exponent", c_float),
        ("kl_loss_scale", c_float),
        ("encoder_kind", c_int32),
        ("dropout_rate", c_float),
    ]


class DibOutputEncoderConfig(ctypes.Structure):
    _fields_ = [
        ("input_dimensionality", c_int32),
        ("number_layers", c_int32),
        ("architecture", POINTER(c_int32)),
    ]


# name -> (restype, argtypes); mirrors include/dib_b200.h one to one
SIGNATURES = {
    "dib_create": (c_int32, [POINTER(DibConfig), POINTER(c_void_p)]),
    "dib_destroy": (None, [c_void_p]),
    "dib_param_count": (c_int64, [c_void_p]),
    "dib_param_layout": (c_int32, [c_void_p, POINTER(c_int64), POINTER(c_int32), POINTER(c_int32), c_int32]),
    "dib_workspace_bytes": (c_size_t, [c_void_p]),
    "dib_stats_count": (c_int32, [c_void_p]),
    "dib_forward": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_uint64,
                              c_uint32, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dib_encode_feature": (c_int32, [c_void_p, c_void_p, c_int32, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "dib_train_step": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_float, c_void_p,
                                 c_uint64, c_uint32, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dib_train_step_phased": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_float, c_void_p,
                                        c_uint64, c_uint32, c_uint64, c_void_p, c_void_p, c_void_p, c_int32, c_void_p]),
    "dib_set_noise_step_device": (c_int32, [c_void_p, c_void_p]),
    "dib_adam_step": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_float,
                                c_float, c_float, c_void_p]),
    "dib_optimizer_step": (c_int32, [c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_float,
                                     c_float, c_float, c_void_p]),
    "dib_integration_forward": (c_int32, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "dib_positional_encoding": (c_int32, [c_void_p, c_int64, c_int32, c_int32, c_void_p, c_void_p]),
    "dib_metrics_update": (c_int32, [c_void_p, c_void_p, c_void_p, c_int32, c_void_p]),
    "dib_metrics_update_ex": (c_int32, [c_void_p, c_void_p, c_void_p, c_int32, c_float, c_float, c_void_p]),
    "dib_encoders_forward": (c_int32, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_uint64, c_uint32, c_uint64, c_void_p,
                                       c_void_p, c_void_p, c_void_p]),
    "dib_encoders_backward": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_float, c_void_p, c_uint64,
                                        c_uint32, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dib_bhattacharyya": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p]),
    "dib_pairwise_gaussian": (c_int32, [c_int32, c_void_p, c_int64, c_void_p, c_int64, c_int32, c_void_p, c_void_p,
                                        c_void_p]),
    "dib_scaled_similarity": (c_int32, [c_int32, c_void_p, c_int64, c_void_p, c_int64, c_int32, c_float, c_void_p, c_void_p]),
    "dib_infonce_head": (c_int32, [c_int32, c_void_p, c_void_p, c_int64, c_int32, c_float, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p]),
    "dib_infonce_head_tc_scratch_bytes": (c_int64, [c_int64, c_int32]),
    "dib_infonce_head_tc": (c_int32, [c_int32, c_void_p, c_void_p, c_int64, c_int32, c_float, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_void_p]),
    "dib_attach_output_encoder": (c_int32, [c_void_p, POINTER(DibOutputEncoderConfig)]),
    "dib_output_encoder_param_count": (c_int64, [c_void_p]),
    "dib_output_encoder_param_layout": (c_int32, [c_void_p, POINTER(c_int64), POINTER(c_int32), POINTER(c_int32), c_int32]),
    "dib_output_encoder_forward": (c_int32, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "dib_infonce_train_step": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int32, c_float, c_void_p,
                                         c_uint64, c_uint32, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dib_infonce_forward": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int32, c_float, c_void_p,
                                      c_uint64, c_uint32, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dib_infonce_scratch_bytes": (c_int64, [c_int32, c_int64, c_int32]),
    "dib_ctw_estimate_entropy": (c_int32, [c_void_p, c_int64, c_int32, c_void_p]),
    "dib_ctw_estimate_entropy_batch": (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p]),
    "dib_ctw_last_error": (c_char_p, []),
    "dib_compression_matrices": (c_int32, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p,
                                           c_void_p, c_void_p, c_void_p]),
    "dib_mi_sandwich_bounds": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_uint64, c_uint32, c_void_p, c_void_p, c_void_p]),
    "dib_mi_sandwich_bounds_batched": (c_int32, [c_void_p, c_int32, c_int64, c_int32, c_void_p, c_uint64, c_int32, c_void_p,
                                                 c_void_p, c_void_p]),
    "dib_launch_count": (c_uint64, []),
    "dib_profile_enable": (c_int32, [c_void_p, c_int32]),
    "dib_profile_read": (c_int32, [c_void_p, c_char_p, c_size_t, POINTER(c_float), c_int32]),
    "dib_debug_gemm_tc": (c_int32, [c_int32, c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_int32,
                                    c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int64, c_int32,
                                    c_void_p]),
    "dib_debug_force_unfused": (c_int32, [c_void_p, c_int32]),
    "dib_debug_set_variant": (c_int32, [c_int32, c_int32]),
    "dib_last_error": (c_char_p, []),
    "dib_build_info": (c_char_p, []),
    "dib_model_info": (c_int32, [c_void_p, c_char_p, c_size_t]),
}

_lib = None


class DibError(RuntimeError):
    pass


def library_path():
    return _build.LIB_PATH


def load():
    """Load (building first if the sources are newer and nvcc is present).  Raises if unavailable."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.build_library()
    if not os.path.exists(path):
        raise DibError(f"{path} is missing: run `python __graft_entry__.py build`")
    lib = ctypes.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status):
    if status != 0:
        raise DibError(load().dib_last_error().decode())


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else c_void_p(t.data_ptr())
