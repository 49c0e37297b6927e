"""ctypes binding of libdfb200.so (the C ABI declared in include/dfb200.h).

There is no CPU fallback: importing this module without the built shared object raises, and
every entry point fails with a ``RuntimeError`` when no sm_100 device is usable.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libdfb200.so")

DFB_ERR_INVALID, DFB_ERR_CUDA, DFB_ERR_UNSUPPORTED, DFB_ERR_OOM = -1, -2, -3, -4


class DfbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(msg)
        self.code = code


class ModelConfigC(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "model_kind", "nb_erb", "nb_df", "df_order", "df_lookahead", "conv_lookahead", "conv_ch",
        "conv_kt", "inp_kt", "emb_hidden", "df_hidden", "enc_gru_layers", "erb_gru_layers",
        "df_gru_layers", "df_pathway_kt", "enc_concat", "g_df_fc_emb", "g_enc_in", "g_enc_out",
        "g_erb_in", "g_erb_out", "g_df_in", "g_df_skip", "g_df_out")] + [
        ("lsnr_scale", C.c_float), ("lsnr_offset", C.c_float), ("norm_alpha", C.c_float)]


class TensorC(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.POINTER(C.c_float)), ("numel", C.c_int64)]


def build(force: bool = False) -> str:
    """Compile libdfb200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
    src_dir = os.path.join(_HERE, "csrc")
    if force and os.path.exists(SO_PATH):
        os.remove(SO_PATH)
    subprocess.check_call(["make", "-C", src_dir, "-j4"], stdout=subprocess.DEVNULL)
    return SO_PATH


_lib = None

_VP, _FP, _I64, _I, _F = C.c_void_p, C.POINTER(C.c_float), C.c_int64, C.c_int, C.c_float
_I64P = C.POINTER(C.c_int64)

SIGNATURES = {
    # name: (restype, argtypes)
    "dfb_last_error": (C.c_char_p, []),
    "dfb_version": (C.c_char_p, []),
    "dfb_kernel_launches": (_I64, []),
    "dfb_profile_enable": (_I, [_I, C.c_char_p]),
    "dfb_profile_report": (_I64, [C.c_char_p, _I64]),
    "dfb_state_create": (_I, [C.POINTER(_VP), _I, _I, _I, _I, _I, _I]),
    "dfb_state_free": (None, [_VP]),
    "dfb_state_erb_widths": (_I, [_VP, _I64P]),
    "dfb_state_fft_window": (_I, [_VP, _FP]),
    "dfb_state_params": (_I, [_VP, C.POINTER(_I), C.POINTER(_I), C.POINTER(_I), C.POINTER(_I)]),
    "dfb_erb_widths": (_I, [_I, _I, _I, _I, _I64P]),
    "dfb_analysis": (_I, [_VP, _VP, _I64, _I64, _VP, _VP]),
    "dfb_analysis_host": (_I, [_VP, _VP, _I64, _I64, _VP]),
    "dfb_analysis_host_ex": (_I, [_VP, _VP, _I64, _I64, _I, _VP]),
    "dfb_synthesis_host_ex": (_I, [_VP, _VP, _I64, _I64, _I, _VP]),
    "dfb_state_reset": (_I, [_VP]),
    "dfb_synthesis": (_I, [_VP, _VP, _I64, _I64, _VP, _VP]),
    "dfb_synthesis_host": (_I, [_VP, _VP, _I64, _I64, _VP]),
    "dfb_erb_host": (_I, [_I, _VP, _I64, _I64, _I64P, _I, _I, _VP]),
    "dfb_erb_inv_host": (_I, [_I, _VP, _I64, _I64P, _I, _VP]),
    "dfb_erb_norm_host": (_I, [_I, _VP, _I64, _I64, _I64, _F, _VP, _VP]),
    "dfb_unit_norm_host": (_I, [_I, _VP, _I64, _I64, _I64, _F, _VP, _VP]),
    "dfb_unit_norm_init": (_I, [_I64, _VP]),
    "dfb_features": (_I, [_VP, _VP, _I64, _I64, _I, _F, _VP, _VP, _VP, _VP]),
    "dfb_features_host": (_I, [_VP, _VP, _I64, _I64, _I, _F, _VP, _VP, _VP]),
    "dfb_resample_host": (_I, [_I, _VP, _I64, _I64, _VP, _I, _I, _I, _VP, _I64]),
    "dfb_metrics": (_I, [_I, _VP, _VP, _VP, _I64, _I64, _I, C.c_uint, _VP, _VP]),
    "dfb_metrics_host": (_I, [_I, _VP, _VP, _VP, _I64, _I64, _I, C.c_uint, _VP]),
    "dfb_model_create": (_I, [C.POINTER(_VP), _I, C.POINTER(ModelConfigC), C.POINTER(TensorC), _I, _I64P]),
    "dfb_model_free": (None, [_VP]),
    "dfb_model_forward": (_I, [_VP, _VP, _VP, _I64, _I64, _VP, _VP, _VP, _VP, _VP]),
    "dfb_apply": (_I, [_VP, _VP, _VP, _VP, _VP, _I64, _I64, _VP, _VP]),
    "dfb_model_forward_full": (_I, [_VP, _VP, _VP, _VP, _VP, _I64, _I64, _VP, _VP, _VP, _VP, _VP, _VP]),
    "dfb_enhance": (_I, [_VP, _VP, _VP, _I64, _I64, _I, _F, _VP, _VP]),
    "dfb_enhance_host": (_I, [_VP, _VP, _VP, _I64, _I64, _I, _F, _VP]),
    "dfb_enhance_out_len": (_I64, [_VP, _I64, _I]),
    "dfb_model_workspace_bytes": (_I64, [_VP]),
    "dfb_stream_create": (_I, [C.POINTER(_VP), _VP, _VP, _I64, _F]),
    "dfb_stream_free": (None, [_VP]),
    "dfb_stream_reset": (_I, [_VP]),
    "dfb_stream_frame_length": (_I64, [_VP]),
    "dfb_stream_latency_frames": (_I64, [_VP]),
    "dfb_stream_set_lsnr_thresholds": (_I, [_VP, _I, _F, _F, _F]),
    "dfb_stream_process": (_I, [_VP, _VP, _I64, _VP, _VP]),
    "dfb_stream_flush": (_I, [_VP, _VP, _VP]),
    "dfb_stream_process_host": (_I, [_VP, _VP, _I64, _VP]),
    "dfb_model_set_precision": (_I, [_VP, _I]),
    "dfb_model_set_max_workspace": (_I, [_VP, _I64]),
    "dfb_model_set_options": (_I, [_VP, _I, _F, _I]),
    "dfb_model_set_chunking": (_I, [_VP, _I, _I, _I]),
    "dfb_debug_gru_timing": (_I, [_VP, _I, _VP]),
    "dfb_model_debug_fetch": (_I64, [_VP, C.c_char_p, _VP, _I64]),
}


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise ImportError(
                f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  deepfilternet_b200 has no CPU fallback.")
        L = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # raises AttributeError when a declared symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().dfb_last_error()
        raise DfbError(rc, (msg or b"unknown error").decode())
