"""ctypes binding of ``libcara_b200.so`` (the C ABI declared in include/cara_b200.h).

The library is the product: there is no CPU / eager fallback.  ``lib()`` raises if the shared object is
missing or does not export what the header declares.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcara_b200.so")

EPI_NONE, EPI_GELU, EPI_DGELU, EPI_DELTA = 0, 1, 2, 3
SIDE_NONE, SIDE_FWD, SIDE_BWD = 0, 1, 2
SYNC_WORDS = 16386
ABI_VERSION = 3


class GemmDesc(C.Structure):
    _fields_ = [
        ("M", C.c_int), ("N", C.c_int), ("K0", C.c_int),
        ("A0", C.c_void_p), ("lda0", C.c_long),
        ("B0", C.c_void_p), ("ldb0", C.c_long),
        ("K1", C.c_int), ("ext_slices", C.c_int),
        ("A1", C.c_void_p), ("lda1", C.c_long),
        ("B1", C.c_void_p), ("ldb1", C.c_long),
        ("bias", C.c_void_p),
        ("out", C.c_void_p), ("ldo", C.c_int),
        ("out2", C.c_void_p), ("ldo2", C.c_int),
        ("aux", C.c_void_p), ("ldaux", C.c_int),
        ("epi", C.c_int), ("num_sms", C.c_int),
        ("side", C.c_int), ("side_rp", C.c_int), ("side_slices", C.c_int),
        ("P", C.c_void_p), ("ldp", C.c_long),
        ("side_scales", C.c_void_p), ("side_T", C.c_void_p),
        ("side_U", C.c_void_p), ("side_ldu", C.c_long),
        ("side_dc", C.c_void_p), ("sync_ws", C.c_void_p),
        ("aux2", C.c_void_p), ("ldaux2", C.c_int),
        ("delta", C.c_void_p), ("seq_n", C.c_int),
    ]


_P = C.c_void_p


class StageDesc(C.Structure):
    """struct cara_stage_desc (include/cara_b200.h)."""
    _PTRS_IN = ["A1", "A3", "A4", "P1", "P2", "R1", "R2", "bias1", "bias2", "bias3", "ai", "pi", "mi", "s_a", "s_m",
                "fb_proj", "fb_fc1", "fb_fc2"]
    _PTRS_OUT = ["kr", "cs_qkv", "cs_proj", "cs_fc1", "a_fc2", "cs_fc2", "b_proj", "b_fc1", "b_fc2",
                 "cs_qkv_pad", "cs_proj_pad", "cs_fc1_pad", "cs_fc2_pad"]
    _PTRS_G = ["g_kr", "g_cs_qkv", "g_cs_proj", "g_cs_fc1", "g_a_fc2", "g_cs_fc2", "g_b_proj", "g_b_fc1", "g_b_fc2"]
    _LDS = ["ld_kr", "ld_cs_qkv", "ld_cs_proj", "ld_cs_fc1", "ld_a_fc2", "ld_cs_fc2"]
    _PTRS_D = ["dA1", "dA3", "dA4", "dP1", "dP2", "dR1", "dR2", "dbias1", "dbias2", "dbias3"]
    _fields_ = ([(n, C.c_int) for n in ("R", "Rp", "C", "D", "L")] + [(n, C.c_void_p) for n in _PTRS_IN + _PTRS_OUT + _PTRS_G] +
                [(n, C.c_long) for n in _LDS] + [(n, C.c_void_p) for n in _PTRS_D])

_SIGS = {
    "cara_abi_version": (C.c_int, []),
    "cara_last_error": (C.c_char_p, []),
    "cara_set_device": (C.c_int, [C.c_int]),
    "cara_gemm_cp": (C.c_int, [C.POINTER(GemmDesc), C.c_void_p]),
    "cara_ln_fwd": (C.c_int, [_P, _P, _P, C.c_int, _P, _P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_float, C.c_int, _P]),
    "cara_ln_bwd": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "cara_ln_rows_supported": (C.c_int, [C.c_int, C.c_int]),
    "cara_ln_fwd_rows": (C.c_int, [_P, _P, _P, C.c_int, _P, _P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_float,
                                   _P, _P, C.c_int, C.c_int, _P, _P, _P]),
    "cara_ln_bwd_rows": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int,
                                   _P, _P, C.c_int, _P, _P, _P, _P]),
    "cara_adapter_rows_fwd": (C.c_int, [_P, C.c_long, C.c_int, C.c_int, _P, _P, C.c_int, C.c_int, _P, _P, _P]),
    "cara_adapter_rows_bwd": (C.c_int, [_P, C.c_long, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int, _P, _P, _P, _P]),
    "cara_adapter_cols": (C.c_int, [_P, C.c_long, C.c_int, C.c_int, _P, C.c_long, C.c_int, C.c_int, _P, _P, _P]),
    "cara_attn_fwd": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, _P]),
    "cara_attn_bwd": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, _P]),
    "cara_attn_tiled_fwd": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, _P]),
    "cara_attn_tiled_bwd": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, _P]),
    "cara_debug_read": (C.c_int, [_P, C.c_int]),
    "cara_gelu_f32": (C.c_int, [_P, _P, _P, C.c_long, _P]),
    "cara_attn_f32": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, _P]),
    "cara_resize_normalize": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int, _P, _P, C.c_int, _P, _P, _P,
                                        C.c_int, C.c_int, _P, _P, _P]),
    "cara_patchify": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "cara_assemble_tokens": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, _P]),
    "cara_factor_operands": (C.c_int, [_P, _P, _P, C.c_long, C.c_int, C.c_int, C.c_int, _P]),
    "cara_stage_terms": (C.c_int, [C.POINTER(StageDesc), C.c_int, _P]),
    "cara_merge_weights": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "cara_adamw_step": (C.c_int, [_P, _P, _P, _P, C.c_long, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                                  C.c_int, C.c_float, _P]),
    "cara_adamw_step_dev": (C.c_int, [_P, _P, _P, _P, C.c_long, _P, C.c_float, C.c_float, C.c_float, C.c_float,
                                      C.c_float, _P]),
    "cara_sgemm": (C.c_int, [_P, C.c_long, C.c_long, _P, C.c_long, C.c_long, _P, C.c_long, _P, C.c_int, C.c_int,
                             C.c_int, C.c_float, C.c_float, _P, C.c_long, _P]),
}

_lib = None


class CaraLibraryError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CaraLibraryError(
                "libcara_b200.so is not built (%s); run `python -m cara_b200.build` -- there is no fallback path"
                % LIB_PATH)
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(handle, name)  # AttributeError if the symbol is missing
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc, what):
    if rc != 0:
        raise CaraLibraryError("%s failed: %s" % (what, lib().cara_last_error().decode()))


def exported_symbols():
    return sorted(_SIGS)
