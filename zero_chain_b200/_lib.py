"""ctypes loader of libzkb200.so (the C ABI declared in include/zkb200.h).

Fails loudly when the CUDA library is missing: there is no CPU fallback in the product."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libzkb200.so")

vp, sz, i32, u32, dbl = C.c_void_p, C.c_size_t, C.c_int, C.c_uint, C.c_double
PP = C.POINTER(C.c_void_p)

# name -> (restype, argtypes); kept in one place so tests can check it against include/zkb200.h
SIGNATURES = {
    "zk_last_error": (C.c_char_p, []),
    "zk_device_count": (i32, []),
    "zk_version": (C.c_char_p, []),
    "zk_ctx_create": (i32, [i32, vp, PP]),
    "zk_ctx_destroy": (None, [vp]),
    "zk_ctx_sync": (i32, [vp]),
    "zk_ctx_set_opt": (i32, [vp, i32, C.c_long]),
    "zk_ctx_stream": (vp, [vp]),
    "zk_bases_upload": (i32, [vp, i32, vp, sz, i32, i32, PP]),
    "zk_bases_free": (None, [vp]),
    "zk_bases_len": (sz, [vp]),
    "zk_bases_window_bits": (i32, [vp]),
    "zk_msm": (i32, [vp, vp, vp, sz, vp]),
    "zk_msm_device": (i32, [vp, vp, vp, sz, vp]),
    "zk_msm_begin": (i32, [vp, vp, vp, sz]),
    "zk_msm_device_begin": (i32, [vp, vp, vp, sz]),
    "zk_msm_end": (i32, [vp, vp]),
    "zk_ctx_tail_stream": (vp, [vp]),
    "zk_msm_partial_device_begin": (i32, [vp, vp, vp, sz, vp]),
    "zk_points_fold_begin": (i32, [vp, i32, vp, sz]),
    "zk_msm_batch_device": (i32, [vp, vp, vp, sz, sz, vp]),
    "zk_partial_size": (sz, [i32]),
    "zk_msm_partial_device": (i32, [vp, vp, vp, sz, vp]),
    "zk_points_fold": (i32, [vp, i32, vp, sz, vp]),
    "zk_ntt_fr": (i32, [vp, vp, u32, i32]),
    "zk_ntt_fr_device": (i32, [vp, vp, u32, i32]),
    "zk_params_load": (i32, [vp, vp, sz, i32, PP]),
    "zk_params_free": (None, [vp]),
    "zk_params_counts": (i32, [vp, vp]),
    "zk_params_size": (sz, [vp]),
    "zk_params_vk_size": (sz, [vp]),
    "zk_params_write": (i32, [vp, vp, vp]),
    "zk_params_write_vk": (i32, [vp, vp, vp]),
    "zk_params_load_cached": (i32, [vp, vp, sz, C.c_char_p, C.POINTER(i32), PP]),
    "zk_groth16_prove": (i32, [vp, vp, vp, vp, vp, sz, vp, sz, vp, sz, vp, vp, vp, vp, vp, vp]),
    "zk_groth16_prove_batch": (i32, [vp, vp, sz, vp, vp, vp, sz, vp, sz, vp, sz, vp, vp, vp, vp, vp, vp]),
    "zk_r1cs_load": (i32, [vp, sz, sz, sz, vp, vp, vp, vp, vp, vp, vp, vp, vp, PP]),
    "zk_r1cs_free": (None, [vp]),
    "zk_groth16_prove_witness_batch": (i32, [vp, vp, vp, sz, vp, vp, vp, vp, vp]),
    "zk_groth16_generate": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, vp, PP]),
    "zk_scalar_mul_many": (i32, [vp, i32, vp, vp, sz, vp]),
    "zk_field_op": (i32, [vp, i32, i32, vp, vp, sz, vp]),
    "zk_bench_modmul": (i32, [vp, i32, i32, i32, i32, C.POINTER(dbl), C.POINTER(dbl)]),
    "zk_ctx_profile": (i32, [vp, i32]),
    "zk_ctx_profile_read": (i32, [vp, C.POINTER(dbl), C.POINTER(C.c_uint64)]),
    "zk_ctx_profile_counts": (i32, [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "zk_pvk_load": (i32, [vp, vp, sz, PP]),
    "zk_pvk_prepare": (i32, [vp, vp, sz, PP]),
    "zk_pvk_size": (sz, [vp]),
    "zk_pvk_write": (i32, [vp, vp]),
    "zk_pvk_num_inputs": (sz, [vp]),
    "zk_pvk_free": (None, [vp]),
    "zk_groth16_verify_batch": (i32, [vp, vp, sz, vp, vp, sz, vp]),
    "zk_groth16_verify_batch_device": (i32, [vp, vp, sz, vp, vp, sz, vp]),
    "zk_pairing_batch": (i32, [vp, sz, vp, vp, vp]),
}

_lib = None


class ZkError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("zkb200 error %d: %s" % (code, msg))
        self.code = code


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise ImportError("libzkb200.so not built (%s): run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "or `make -C zero_chain_b200/csrc`; there is no CPU fallback" % SO_PATH)
        L = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)      # AttributeError here = header/library mismatch: fail loudly
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(code):
    if code != 0:
        raise ZkError(code, lib().zk_last_error().decode())
