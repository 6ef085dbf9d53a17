"""ctypes binding of liblac_b200.so (include/lac_b200.h).  No torch types cross this boundary:
callers pass raw device / host addresses (tensor.data_ptr()) and sizes.

There is deliberately no fallback: if the CUDA library is missing, importing the compute
API raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "liblac_b200.so")

LAC_OK, LAC_E_ARG, LAC_E_CUDA, LAC_E_CAP, LAC_E_SYMBOL, LAC_E_STREAM = 0, -1, -2, -3, -4, -5
LAC_ST_CAP, LAC_ST_SYMBOL, LAC_ST_TABLE, LAC_ST_TRUNC = 1, 2, 4, 8
LAC_F_WRAP64 = 1
LAC_ADAPTIVE_MAX_VOCAB = 4096
LAC_MODEL_OUT_BF16, LAC_MODEL_OUT_BF16_ADD, LAC_MODEL_OUT_F32 = 0, 1, 2
ABI_VERSION = 4


class LacError(RuntimeError):
    def __init__(self, code: int, text: str):
        super().__init__(f"lac_b200 error {code}: {text}")
        self.code = code


class EncState(C.Structure):
    _fields_ = [("low", C.c_int64), ("high", C.c_int64), ("nbits", C.c_uint64),
                ("status", C.c_uint32), ("_pad", C.c_uint32)]


class DecState(C.Structure):
    _fields_ = [("low", C.c_int64), ("high", C.c_int64), ("value", C.c_int64), ("pos", C.c_uint64),
                ("status", C.c_uint32), ("_pad", C.c_uint32)]


ENC_STATE_BYTES = C.sizeof(EncState)   # 32
DEC_STATE_BYTES = C.sizeof(DecState)   # 40

_p, _i64, _i32, _int, _f32 = C.c_void_p, C.c_int64, C.c_int32, C.c_int, C.c_float

# name -> argtypes; every symbol include/lac_b200.h declares (tests/test_abi.py checks the set)
SIGNATURES = {
    "lac_abi_version": [],
    "lac_last_error": [],
    "lac_device_info": [_p, _p, _p, _p],
    "lac_workspace_bytes": [_i64, _i32],
    "lac_cdf_build_f32": [_p, _i64, _i32, _i64, _p, _p, _i64, _p],
    "lac_cdf_lookup_f32": [_p, _i64, _i32, _i64, _p, _p, _p, _p, _i64, _p],
    "lac_enc_init": [_p, _i64, _int, _p],
    "lac_dec_init": [_p, _i64, _int, _p, _p, _p],
    "lac_ac_encode_pairs": [_p, _i64, _i64, _i64, _i64, _p, _p, _p, _i64, _int, _int, _p],
    "lac_ac_encode_uniform": [_p, _i64, _i64, _i64, _p, _i32, _p, _p, _i64, _int, _int, _p],
    "lac_ac_decode_uniform": [_i64, _i64, _p, _i32, _p, _p, _p, _p, _i64, _int, _p],
    "lac_ac_encode_logits_f32": [_p, _i64, _i64, _i64, _i64, _i32, _p, _i64, _p, _p, _p, _i64, _int, _int, _p, _i64, _p],
    "lac_ac_decode_logits_f32": [_p, _i64, _i64, _i64, _i64, _i32, _p, _p, _p, _p, _p, _i64, _int, _p, _i64, _p],
    "lac_enc_status": [_p, _i64, _p, _p],
    "lac_dec_status": [_p, _i64, _p, _p],
    "lac_ac_encode_tables": [_p, _i32, _i64, _i64, _p, _i64, _i64, _p, _i64, _i64, _i64, _p, _p, _p, _i64, _int, _int, _int, _p],
    "lac_ac_decode_tables": [_p, _i32, _i64, _i64, _p, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _p, _i64, _int, _int, _p],
    "lac_acs_encode_tables": [_p, _i32, _i64, _i64, _p, _i64, _i64, _i64, _p, _p, _p, _i64, _int, _int, _p],
    "lac_acs_decode_tables": [_p, _i32, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _p, _i64, _int, _p],
    "lac_ac_encode_adaptive": [_p, _i32, _i64, _p, _i64, _i64, _i64, _p, _p, _p, _i64, _int, _int, _p],
    "lac_ac_decode_adaptive": [_p, _i32, _i64, _i64, _i64, _p, _p, _p, _p, _p, _i64, _int, _p],
    "lac_acs_encode_adaptive": [_p, _i32, _i64, _p, _i64, _i64, _i64, _p, _p, _p, _i64, _int, _int, _p],
    "lac_acs_decode_adaptive": [_p, _i32, _i64, _i64, _i64, _p, _p, _p, _p, _p, _i64, _int, _p],
    "lac_model_gemm": [_p, _p, _i64, _i32, _i32, _int, _p, _p, _p],
    "lac_model_rmsnorm": [_p, _i64, _i32, _f32, _p, _p],
    "lac_model_rope_kv": [_p, _i64, _i32, _i32, _i32, _i32, _p, _p, _p, _i64, _p, _p, _i32, _p],
    "lac_model_swiglu": [_p, _i64, _i32, _p, _p],
    "lac_model_attention": [_p, _i32, _i32, _i32, _i32, _i32, _p, _i64, _p, _p, _i32, _p, _p],
    "lac_encode_logits_host": [_p, _p, _i64, _i64, _i32, _p, _i64, _p, _int],
    "lac_decode_logits_host": [_p, _i64, _i64, _i32, _p, _p, _p, _int],
}

_lib = None


def lib():
    """The loaded library; raises if it has not been built (python -c 'import __graft_entry__ as g; g.build()')."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LacError(LAC_E_CUDA, f"{LIB_PATH} is missing: build it with __graft_entry__.build() "
                                       "(make -C lac_b200/csrc). lac_b200 has no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, argtypes in SIGNATURES.items():
            fn = getattr(L, name)
            fn.argtypes = argtypes
            fn.restype = (C.c_char_p if name == "lac_last_error" else
                          C.c_int64 if name == "lac_workspace_bytes" else C.c_int)
        if L.lac_abi_version() != ABI_VERSION:
            raise LacError(LAC_E_ARG, f"ABI version mismatch: library {L.lac_abi_version()}, binding {ABI_VERSION}")
        _lib = L
    return _lib


def check(rc: int):
    if rc != 0:
        raise LacError(rc, (lib().lac_last_error() or b"").decode("utf-8", "replace"))


def device_info():
    sm, maj, mnr, mem = C.c_int(0), C.c_int(0), C.c_int(0), C.c_int64(0)
    check(lib().lac_device_info(C.byref(sm), C.byref(maj), C.byref(mnr), C.byref(mem)))
    return {"sm_count": sm.value, "cc": (maj.value, mnr.value), "hbm_bytes": mem.value}
