"""ctypes binding of libafs_b200.so -- the only door from Python into the CUDA kernels.

The signatures below restate include/afs_b200.h one to one.  There is no fallback:
if the library cannot be loaded (not built, wrong arch) `lib()` raises, and every
op in `audio_fewshot_b200.ops` raises with it.
"""
import ctypes as C
import os
import threading

from . import build as _build

_c_float_p = C.POINTER(C.c_float)
_c_int32_p = C.POINTER(C.c_int32)


class LogMelCfg(C.Structure):
    _fields_ = [
        ("n_fft", C.c_int32),
        ("hop", C.c_int32),
        ("n_mels", C.c_int32),
        ("center", C.c_int32),
        ("log_mult", C.c_float),
        ("log_eps", C.c_float),
    ]


class AugCfg(C.Structure):
    _fields_ = [
        ("gain_db_lo", C.c_float),
        ("gain_db_hi", C.c_float),
        ("max_shift", C.c_int32),
        ("noise_std_lo", C.c_float),
        ("noise_std_hi", C.c_float),
    ]


class SpecAugCfg(C.Structure):
    _fields_ = [
        ("type", C.c_int32),
        ("n_rect", C.c_int32),
        ("rect", (C.c_int32 * 4) * 8),
        ("fill", C.c_float),
        ("p0", C.c_float),
        ("p1", C.c_float),
        ("i0", C.c_int32),
    ]


# name -> (restype, argtypes); must list every symbol include/afs_b200.h declares
SIGNATURES = {
    "afs_abi_version": (C.c_int, []),
    "afs_status_string": (C.c_char_p, [C.c_int]),
    "afs_last_cuda_error": (C.c_int, []),
    "afs_launch_count": (C.c_uint64, []),
    "afs_logmel_plan_create": (C.c_int, [C.POINTER(LogMelCfg), C.c_void_p, C.c_void_p, C.c_int,
                                         C.POINTER(C.c_void_p)]),
    "afs_logmel_plan_destroy": (C.c_int, [C.c_void_p]),
    "afs_logmel_num_frames": (C.c_int, [C.c_void_p, C.c_int64]),
    "afs_logmel_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p,
                                 C.POINTER(AugCfg), C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p]),
    "afs_logmel_fwd_pcm16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_float, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p,
                                       C.POINTER(AugCfg), C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p]),
    "afs_conv1_bn_act_pool3_fwd": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                             C.c_int32, C.c_float, C.c_void_p, C.c_void_p]),
    "afs_conv1_bn_act_pool3_fwd_tf32": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                                  C.c_int32, C.c_float, C.c_void_p, C.c_void_p]),
    "afs_conv1_train_num_partials": (C.c_int32, [C.c_int32]),
    "afs_conv1_autocorr": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "afs_conv1_train_stats": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "afs_conv1_train_grads": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "afs_conv1_train_fwd": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_float, C.c_void_p, C.c_void_p]),
    "afs_conv1_train_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p]),
    "afs_conv3x3_c64_packed_floats": (C.c_size_t, []),
    "afs_conv3x3_c64_pack_weights": (C.c_int, [C.c_void_p, C.c_void_p]),
    "afs_conv3x3_c64_bn_act_fwd_tf32": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                                  C.c_float, C.c_int32, C.c_void_p, C.c_void_p]),
    "afs_conv3x3_c64_packed_bf16_elems": (C.c_size_t, []),
    "afs_conv3x3_c64_pack_weights_bf16": (C.c_int, [C.c_void_p, C.c_void_p]),
    "afs_conv3x3_c64_bn_act_fwd_bf16": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                                  C.c_float, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]),
    "afs_conv1_bn_act_pool3_fwd_tf32_bf16out": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                                          C.c_void_p, C.c_int32, C.c_float, C.c_void_p, C.c_void_p]),
    "afs_pool3_linear_fwd": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                       C.c_int32, C.c_void_p, C.c_void_p]),
    "afs_maxpool3_nhwc_fwd": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                        C.c_void_p]),
    "afs_add_bias_act_pool_nhwc_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                                 C.c_int32, C.c_float, C.c_int32, C.c_void_p, C.c_void_p]),
    "afs_add_bias_act_pool_nhwc_bf16_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                                      C.c_int32, C.c_float, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]),
    "afs_proto_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "afs_proto_tc_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32]),
    "afs_proto_fwd_tc": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "afs_proto_fwd": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_size_t, C.c_void_p]),
    "afs_proto_bwd": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64,
                                C.c_void_p]),
    "afs_proto_bwd_cos_workspace_bytes": (C.c_size_t, [C.c_int32] * 4),
    "afs_proto_bwd_cos": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                    C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_size_t,
                                    C.c_void_p]),
    "afs_dn4_workspace_bytes": (C.c_size_t, [C.c_int32] * 6),
    "afs_dn4_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                              C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                              C.c_void_p, C.c_size_t, C.c_void_p]),
    "afs_dn4_tc_workspace_bytes": (C.c_size_t, [C.c_int32] * 5),
    "afs_dn4_fwd_tc": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                 C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_size_t, C.c_void_p]),
    "afs_dn4_tc2_workspace_bytes": (C.c_size_t, [C.c_int32] * 6),
    "afs_dn4_fwd_tc2": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                  C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_size_t, C.c_void_p]),
    "afs_dn4_bwd_workspace_bytes": (C.c_size_t, [C.c_int32] * 3),
    "afs_dn4_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                              C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                              C.c_void_p]),
    "afs_bdc_bwd": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
                              C.c_void_p, C.c_void_p, C.c_void_p]),
    "afs_bdc_set_tensor_core": (C.c_int, [C.c_int32]),
    "afs_bdc_fwd": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                              C.c_void_p, C.c_void_p]),
    "afs_bdc_wide_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32]),
    "afs_bdc_wide_fwd": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                   C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "afs_bdc_wide_bwd": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "afs_spec_augment": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_float,
                                   C.POINTER(SpecAugCfg), C.c_void_p, C.c_void_p, C.c_void_p]),
    "afs_vote_acc": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "afs_energy_score": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
                                   C.c_void_p]),
}

_lock = threading.Lock()
_lib = None


class AfsError(RuntimeError):
    pass


def lib_path():
    return _build.LIB_PATH


def lib():
    """Load (once) and return the ctypes handle.  Raises if the library is missing."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = lib_path()
        if not os.path.exists(path):
            raise AfsError(
                "libafs_b200.so is not built (%s). Run `python -m audio_fewshot_b200.build`; "
                "there is no CPU or PyTorch fallback for these ops." % path
            )
        handle = C.CDLL(path)
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the symbol is not exported
            fn.restype = restype
            fn.argtypes = argtypes
        if handle.afs_abi_version() != 1:
            raise AfsError("libafs_b200.so ABI version mismatch")
        _lib = handle
        return _lib


def check(status, what):
    if status != 0:
        h = lib()
        msg = h.afs_status_string(status).decode()
        extra = ""
        if status == -3:
            extra = " (cudaError %d)" % h.afs_last_cuda_error()
        raise AfsError("%s failed: %s%s" % (what, msg, extra))
