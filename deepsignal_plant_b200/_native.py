"""ctypes binding of libdsp_b200.so (include/dsp_b200.h).

The product path has no CPU fallback: if the library is missing or cannot be loaded,
``lib()`` raises and every operator that needs it fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DSP_B200_LIB") or os.path.join(_HERE, "libdsp_b200.so")

# every symbol include/dsp_b200.h declares (tests check the export list against this)
SYMBOLS = (
    "dsp_abi_version", "dsp_last_error", "dsp_create", "dsp_destroy", "dsp_set_param",
    "dsp_pack_weights", "dsp_forward", "dsp_forward_host", "dsp_forward_host_submit",
    "dsp_forward_host_wait", "dsp_launch_count",
    "dsp_set_timing", "dsp_get_timing", "dsp_freq_aggregate", "dsp_selftest",
    "dsp_parse_features", "dsp_format_calls", "dsp_freq_release_cache", "dsp_extract_features", "dsp_format_sampleinfo", "dsp_find_sites", "dsp_extract_features_f64",
    "dsp_format_features", "dsp_parse_calls", "dsp_format_freq",
    "dsp_comm_create", "dsp_comm_export", "dsp_comm_connect", "dsp_comm_destroy", "dsp_freq_aggregate_distributed",
    "dsp_comm_route_rows", "dsp_comm_last_timing", "dsp_comm_allreduce_f32", "dsp_freq_aggregate_host", "dsp_device_warmup",
    "dsp_train_shape", "dsp_train_arena_bytes", "dsp_train_workspace_bytes", "dsp_train_forward", "dsp_train_backward",
    "dsp_ranger_step", "dsp_train_forward_batch", "dsp_train_backward_batch",
)

TRAIN_MAX_MODELS = 8    # DSP_TRAIN_MAX_MODELS

MODULES = {"both_bilstm": 0, "seq_bilstm": 1, "signal_bilstm": 2}
PRECISIONS = {"fp32": 0, "fp16": 1}


class DspConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "seq_len", "signal_len", "num_layers1", "num_layers2", "num_classes", "hidden_size",
        "vocab_size", "embedding_size", "is_base", "is_signallen", "module", "device",
        "precision", "reserved")] + [("max_batch", C.c_int64)]


class DspError(RuntimeError):
    pass


_lib = None


def lib():
    """Load the shared library once; raise if it is not there (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH) and "DSP_B200_LIB" not in os.environ:
        # a source checkout that was never built: compile it (nvcc, sm_100a) rather than give up; this is the
        # only automatic step -- there is still no CPU or PyTorch fallback if it fails
        try:
            from . import build as _build
            _build.build()
        except Exception as e:                                  # noqa: BLE001 -- reported below
            raise DspError("libdsp_b200.so is not built and building it failed: %s" % e)
    if not os.path.exists(LIB_PATH):
        raise DspError(
            "libdsp_b200.so is not built (%s). Run `python -m deepsignal_plant_b200.build` "
            "(needs nvcc); there is no CPU or PyTorch fallback for this path." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, fp, i64, u64 = C.c_void_p, C.c_void_p, C.c_int64, C.c_uint64
    L.dsp_abi_version.restype = C.c_int
    L.dsp_last_error.restype = C.c_char_p
    L.dsp_create.argtypes = [C.POINTER(vp), C.POINTER(DspConfig)]
    L.dsp_destroy.argtypes = [vp]
    L.dsp_set_param.argtypes = [vp, C.c_char_p, fp, i64]
    L.dsp_pack_weights.argtypes = [vp]
    L.dsp_forward.argtypes = [vp, fp, fp, fp, fp, fp, C.POINTER(vp), u64, i64, fp, fp, vp, vp]
    L.dsp_forward_host.argtypes = [vp, fp, fp, fp, fp, fp, u64, i64, fp, fp, vp]
    L.dsp_forward_host_submit.argtypes = [vp, fp, fp, fp, fp, fp, u64, i64, fp, fp, vp, C.POINTER(i64)]
    L.dsp_forward_host_wait.argtypes = [vp, i64]
    L.dsp_launch_count.argtypes = [vp]
    L.dsp_launch_count.restype = i64
    L.dsp_set_timing.argtypes = [vp, C.c_int]
    L.dsp_get_timing.argtypes = [vp, C.c_int, C.POINTER(C.c_float), C.POINTER(i64)]
    L.dsp_freq_aggregate.argtypes = [C.c_int, vp, vp, vp, vp, i64, C.c_double, C.c_int,
                                     vp, vp, vp, vp, vp, vp, vp, C.POINTER(i64), vp]
    L.dsp_freq_aggregate_host.argtypes = [C.c_int, vp, vp, C.c_int32, vp, vp, vp, vp, i64, C.c_double, C.c_int,
                                          vp, vp, vp, vp, vp, vp, vp, i64, C.POINTER(i64)]
    L.dsp_device_warmup.argtypes = [C.c_int]
    L.dsp_selftest.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_double)]
    i32 = C.c_int32
    L.dsp_parse_features.argtypes = [vp, i64, i32, i32, i32, i64, fp, fp, fp, fp, fp, vp, vp, i64, vp,
                                     C.POINTER(i64), C.POINTER(i64), i32]
    L.dsp_format_calls.argtypes = [vp, vp, fp, i32, fp, vp, i64, vp, i64, C.POINTER(i64), i32]
    L.dsp_extract_features.argtypes = [C.c_int, vp, vp, vp, vp, i64, vp, vp, vp, vp, vp, i64, i32, i32, i32, i32,
                                       vp, u64, vp, vp, fp, fp, fp, fp, fp, vp]
    L.dsp_format_sampleinfo.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, vp, i64, vp, i32]
    L.dsp_extract_features_f64.argtypes = L.dsp_extract_features.argtypes
    L.dsp_format_features.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i64, i32, i32, vp, i64, C.POINTER(i64), i32]
    L.dsp_parse_calls.argtypes = [vp, i64, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, C.POINTER(i64), C.POINTER(i32),
                                  C.POINTER(i64), i32]
    L.dsp_format_freq.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, vp, vp, vp, vp, vp, vp, vp, i64, i32, vp, i64,
                                  C.POINTER(i64), i32]
    L.dsp_find_sites.argtypes = [C.c_int, vp, vp, i64, i64, C.c_char_p, i32, i32, i32, i32, vp, vp, vp, vp, vp, i64,
                                 vp, vp, vp, vp, C.POINTER(i64), vp]
    L.dsp_comm_create.argtypes = [C.POINTER(vp), C.c_int, C.c_int, C.c_int, i64]
    L.dsp_comm_export.argtypes = [vp, vp, i64, C.POINTER(i64)]
    L.dsp_comm_connect.argtypes = [vp, vp, i64]
    L.dsp_comm_destroy.argtypes = [vp]
    L.dsp_freq_aggregate_distributed.argtypes = [vp, vp, vp, vp, vp, i64, u64, C.c_double, vp, i32, vp, i64,
                                                 C.POINTER(i64), C.POINTER(i64), vp, vp]
    L.dsp_comm_route_rows.argtypes = [vp, vp, i64, i32, i32, vp, vp, i64, C.POINTER(i64), vp]
    L.dsp_comm_last_timing.argtypes = [vp, vp]
    L.dsp_comm_allreduce_f32.argtypes = [vp, C.POINTER(vp), C.POINTER(i64), C.c_int32, vp]
    L.dsp_train_shape.argtypes = [vp, C.POINTER(i32), C.POINTER(i32)]
    L.dsp_train_arena_bytes.argtypes = [vp, i64]
    L.dsp_train_arena_bytes.restype = i64
    L.dsp_train_workspace_bytes.argtypes = [vp, i64]
    L.dsp_train_workspace_bytes.restype = i64
    L.dsp_train_forward.argtypes = [vp, C.POINTER(vp), i32, fp, fp, fp, fp, fp, C.POINTER(vp), u64, C.POINTER(vp), i64, vp,
                                    fp, vp]
    L.dsp_train_backward.argtypes = [vp, C.POINTER(vp), i32, C.POINTER(vp), vp, fp, i64, vp, C.POINTER(vp), vp]
    L.dsp_train_forward_batch.argtypes = [vp, i32, C.POINTER(vp), i32, C.POINTER(vp), C.POINTER(vp), C.POINTER(u64),
                                          C.POINTER(vp), i64, C.POINTER(vp), C.POINTER(vp), vp]
    L.dsp_train_backward_batch.argtypes = [vp, i32, C.POINTER(vp), i32, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), i64,
                                           C.POINTER(vp), C.POINTER(vp), vp]
    d = C.c_double
    L.dsp_ranger_step.argtypes = [i32] + [C.POINTER(vp)] * 5 + [C.POINTER(i64), C.POINTER(i64), C.POINTER(C.c_float),
                                                                 C.POINTER(i32), d, d, d, d, d, i32, vp]
    for name in SYMBOLS:
        getattr(L, name)  # AttributeError here means header and library disagree
    _lib = L
    return L


def check(status, what="libdsp_b200"):
    if status != 0:
        msg = lib().dsp_last_error()
        raise DspError("%s failed (status %d): %s" % (what, status, msg.decode() if msg else "?"))
