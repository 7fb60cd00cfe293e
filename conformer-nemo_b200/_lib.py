"""ctypes binding of libcfb.so (include/cfb.h).  This is the whole Python<->CUDA boundary: plain pointers and ints.

The library is built in-tree by ``build.py`` (nvcc, sm_100a).  There is no CPU fallback: if the library is missing
the import of the encoder fails loudly with the build instruction.
"""
from __future__ import annotations

import ctypes
import os
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libcfb.so")

CFB_OK = 0
CFB_F32, CFB_BF16, CFB_F16, CFB_I64, CFB_I32 = 0, 1, 2, 3, 4
CFB_PREC_BF16, CFB_PREC_FP32_VALIDATE = 0, 1
EPI_LINEAR, EPI_SWISH, EPI_RELU, EPI_RESID, EPI_QKV, EPI_GLU = range(6)
STATUS_NAMES = {1: "invalid argument", 2: "unsupported configuration", 3: "missing weight", 4: "CUDA error",
                5: "workspace", 6: "call order"}

# every symbol include/cfb.h declares (tests check that the built library exports each of them)
SYMBOLS = [
    "cfb_create", "cfb_destroy", "cfb_last_error", "cfb_set_weight", "cfb_finalize_weights", "cfb_output_frames",
    "cfb_workspace_bytes", "cfb_forward", "cfb_packed_workspace_bytes", "cfb_forward_packed", "cfb_debug_buffer", "cfb_set_profiling", "cfb_profile_report",
    "cfb_last_launch_count", "cfb_op_gemm", "cfb_op_ctc_head", "cfb_ctc_head_scratch_bytes", "cfb_op_ctc_collapse",
    "cfb_op_layernorm", "cfb_op_layernorm_dual", "cfb_op_depthwise", "cfb_op_dw_pw2", "cfb_op_logmel", "cfb_op_logmel_raw",
    "cfb_op_feature_buffers", "cfb_op_rel_attention", "cfb_op_lengths",
    "cfb_rnnt_greedy_scratch_bytes", "cfb_op_rnnt_greedy", "cfb_rnnt_beam_scratch_bytes", "cfb_op_rnnt_beam",
]


class CfbConfig(ctypes.Structure):
    _fields_ = [
        ("feat_in", ctypes.c_int32), ("n_layers", ctypes.c_int32), ("d_model", ctypes.c_int32),
        ("feat_out", ctypes.c_int32), ("subsampling_factor", ctypes.c_int32),
        ("subsampling_conv_channels", ctypes.c_int32), ("ff_expansion_factor", ctypes.c_int32),
        ("n_heads", ctypes.c_int32), ("conv_kernel_size", ctypes.c_int32), ("xscaling", ctypes.c_int32),
        ("precision", ctypes.c_int32), ("reserved", ctypes.c_int32 * 5),
    ]


class CfbRnntWeights(ctypes.Structure):
    _fp = ctypes.POINTER(ctypes.c_float)
    _fields_ = [
        ("enc_hidden", ctypes.c_int32), ("pred_hidden", ctypes.c_int32), ("joint_hidden", ctypes.c_int32),
        ("num_classes_with_blank", ctypes.c_int32), ("activation", ctypes.c_int32), ("reserved", ctypes.c_int32 * 3),
        ("embed", _fp), ("w_ih", _fp), ("w_hh", _fp), ("b_ih", _fp), ("b_hh", _fp), ("w_pred", _fp), ("b_pred", _fp),
        ("w_enc", _fp), ("b_enc", _fp), ("w_out", _fp), ("b_out", _fp),
    ]


class CfbRnntBeamCaps(ctypes.Structure):
    _fields_ = [("max_expansions", ctypes.c_int32), ("max_hyps", ctypes.c_int32), ("max_nodes", ctypes.c_int32),
                ("max_states", ctypes.c_int32), ("max_len", ctypes.c_int32), ("reserved", ctypes.c_int32 * 3)]


_lock = threading.Lock()
_lib = None


def load_library() -> ctypes.CDLL:
    """Loads libcfb.so once per process and declares argument types."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build the CUDA library first (python conformer-nemo_b200/build.py). "
                "There is no CPU or PyTorch fallback for the encoder forward.")
        lib = ctypes.CDLL(LIB_PATH)
        vp, i32, i64, sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_size_t
        lib.cfb_create.argtypes = [ctypes.POINTER(CfbConfig), i32, ctypes.POINTER(vp)]
        lib.cfb_destroy.argtypes = [vp]
        lib.cfb_destroy.restype = None
        lib.cfb_last_error.argtypes = [vp]
        lib.cfb_last_error.restype = ctypes.c_char_p
        lib.cfb_set_weight.argtypes = [vp, ctypes.c_char_p, vp, i32, ctypes.POINTER(i64), i32]
        lib.cfb_finalize_weights.argtypes = [vp]
        lib.cfb_output_frames.argtypes = [vp, i32, ctypes.POINTER(i32)]
        lib.cfb_workspace_bytes.argtypes = [vp, i32, i32, ctypes.POINTER(sz)]
        lib.cfb_forward.argtypes = [vp, vp, i32, vp, i32, i32, vp, i32, vp, vp, sz, vp]
        lib.cfb_packed_workspace_bytes.argtypes = [vp, vp, i32, i32, ctypes.POINTER(sz)]
        lib.cfb_forward_packed.argtypes = [vp, vp, i32, vp, vp, i32, i32, vp, i32, vp, vp, sz, vp]
        lib.cfb_debug_buffer.argtypes = [vp, i32, i32, ctypes.c_char_p, ctypes.POINTER(sz), ctypes.POINTER(sz)]
        lib.cfb_last_launch_count.argtypes = [vp]
        lib.cfb_set_profiling.argtypes = [vp, i32]
        lib.cfb_profile_report.argtypes = [vp, ctypes.c_char_p, sz]
        lib.cfb_op_gemm.argtypes = [i32, i32, vp, i64, vp, i64, vp, vp, i32, i32, i32, vp, i64, i32, ctypes.c_float,
                                    vp, i32, i32, vp, vp]
        lib.cfb_ctc_head_scratch_bytes.argtypes = [i32, i32, i32]
        lib.cfb_op_ctc_head.argtypes = [vp, i32, vp, vp, i32, i32, i32, vp, vp, vp, sz, vp]
        lib.cfb_op_ctc_collapse.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp]
        lib.cfb_op_layernorm.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp, i32, vp]
        lib.cfb_op_layernorm_dual.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i32, vp]
        lib.cfb_op_depthwise.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]
        lib.cfb_op_logmel.argtypes = [vp, vp, i32, i32, vp, i32, i32, i32, vp, vp, i32, ctypes.c_float, ctypes.c_float,
                                      ctypes.c_float, vp, i32, vp, vp, vp]
        lib.cfb_op_logmel_raw.argtypes = [vp, vp, i32, i32, vp, i32, i32, i32, vp, vp, i32, ctypes.c_float, ctypes.c_float,
                                          vp, i32, vp, vp]
        lib.cfb_op_feature_buffers.argtypes = [vp, i32, i32, i32, vp, vp, i32, i32, i32, vp, vp]
        lib.cfb_op_dw_pw2.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, vp]
        lib.cfb_op_rel_attention.argtypes = [i32, vp, vp, i64, vp, vp, i32, i32, i32, i32, i32, vp]
        lib.cfb_op_lengths.argtypes = [vp, vp, i32, i32, i32, vp]
        lib.cfb_rnnt_greedy_scratch_bytes.argtypes = [i32, i32, i32, i32, i32]
        lib.cfb_op_rnnt_greedy.argtypes = [ctypes.POINTER(CfbRnntWeights), vp, i32, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp,
                                           vp, vp, vp, sz, vp]
        caps = ctypes.POINTER(CfbRnntBeamCaps)
        lib.cfb_rnnt_beam_scratch_bytes.argtypes = [i32, i32, i32, i32, i32, i32, caps]
        lib.cfb_op_rnnt_beam.argtypes = [ctypes.POINTER(CfbRnntWeights), vp, i32, vp, i32, i32, i32, i32, ctypes.c_float, caps,
                                         vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]
        for name in SYMBOLS:
            fn = getattr(lib, name)
            if name in ("cfb_ctc_head_scratch_bytes", "cfb_rnnt_greedy_scratch_bytes", "cfb_rnnt_beam_scratch_bytes"):
                fn.restype = ctypes.c_size_t
            elif name not in ("cfb_destroy", "cfb_last_error"):
                fn.restype = ctypes.c_int
        _lib = lib
        return lib


def last_error(handle) -> str:
    msg = load_library().cfb_last_error(handle)
    return msg.decode("utf-8", "replace") if msg else ""


def check(status: int, handle=None, what: str = "cfb call") -> None:
    """Maps a non-zero cfb_status to the exception class the reference would raise for the same mistake."""
    if status == CFB_OK:
        return
    msg = f"{what}: {STATUS_NAMES.get(status, status)}: {last_error(handle)}"
    if status == 2:
        raise NotImplementedError(msg)
    if status == 1:
        raise ValueError(msg)
    raise RuntimeError(msg)
