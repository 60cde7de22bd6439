"""ctypes binding of ``libhsv.so`` (the C-ABI declared in ``include/hsv.h``).

The library is built in-tree by ``megatts2_hierspeechpp_b200.build`` (nvcc,
``-gencode arch=compute_100a,code=sm_100a``).  There is NO fallback: if the
shared object is missing or a kernel is asked to run on a non-CUDA tensor the
call raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhsv.so")

# name -> (restype, argtypes); must list every symbol include/hsv.h declares
SIGNATURES = {
    "hsv_version": (c_int, []),
    "hsv_last_error": (c_char_p, []),
    "hsv_device_supported": (c_int, []),
    "hsv_blk16_rows": (c_int64, [c_int64]),
    "hsv_last_launch_config": (c_int, [c_int, c_void_p, c_int]),
    "hsv_act1d_snakebeta": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_int, c_float,
                                    c_void_p]),
    "hsv_act1d_snakebeta_ragged": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64,
                                           c_int, c_float, c_void_p]),
    "hsv_weight_norm_fold": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "hsv_pack_conv_weight": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "hsv_conv1d_umma": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_float,
                                c_int, c_int, c_int, c_int64, c_int, c_int, c_int, c_void_p]),
    "hsv_conv1d_umma_astride": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                        c_int, c_int, c_int64, c_int, c_int, c_int, c_void_p]),
    "hsv_conv1d_umma_blk16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int64, c_void_p, c_int, c_int,
                                      c_int, c_int64, c_int, c_int, c_int, c_void_p]),
    "hsv_conv1d_umma_wn_tail": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                        c_int, c_int64, c_int, c_void_p]),
    "hsv_act_conv1d_umma": (c_int, [c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_int, c_int, c_int, c_int, c_int64, c_int, c_int, c_void_p]),
    "hsv_pack_convT_weight": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "hsv_conv_transpose1d_umma": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                          c_int64, c_int, c_int, c_int, c_void_p]),
    "hsv_conv1d_direct": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_int64,
                                  c_int, c_int, c_int, c_int, c_void_p]),
    "hsv_conv1d_direct_ragged": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int64,
                                         c_int64, c_int, c_int, c_int, c_int, c_void_p]),
    "hsv_conv_transpose1d_direct": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                            c_int64, c_int, c_int, c_void_p]),
    "hsv_sr_pre_interp": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_int64, c_void_p]),
    "hsv_sr_pre_interp_ragged": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                         c_int64, c_int64, c_void_p]),
    "hsv_sr_pre_interp_stream": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                         c_int, c_int64, c_int64, c_int, c_int, c_void_p]),
    "hsv_sr_stream_window": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "hsv_sr_stream_emit": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_int, c_int, c_int, c_int64, c_int, c_void_p]),
    "hsv_interp_linear_table": (c_int, [c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hsv_nearest_gather": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int64, c_void_p]),
    "hsv_add3_bcast": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, c_void_p]),
    "hsv_pack_blk16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int64, c_int, c_float, c_void_p]),
    "hsv_pack_blk16_sum3": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_int, c_float,
                                    c_void_p]),
    "hsv_pack_blk16_sum3_ragged": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_int,
                                           c_float, c_void_p]),
    "hsv_unpack_blk16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int64, c_void_p]),
    "hsv_blk16_stats": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int64, c_void_p]),
    "hsv_pack_blk16_act": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_int, c_int, c_void_p]),
    "hsv_wn_res_pack": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_void_p]),
    "hsv_ln_mod_blk16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_float, c_int,
                                 c_int, c_int64, c_void_p]),
    "hsv_gate_ln_mod_blk16": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                      c_int, c_int64, c_float, c_int, c_int64, c_void_p]),
    "hsv_frame_op": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64,
                             c_float, c_int64, c_void_p]),
    "hsv_mha_blk16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int64,
                              c_int64, c_int64, c_float, c_int, c_void_p]),
    "hsv_mha_ragged": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int,
                               c_int, c_int, c_int64, c_int64, c_int64, c_float, c_int, c_void_p]),
    "hsv_set_mha_variant": (c_int, [c_int]),
    "hsv_mha": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int64,
                        c_int64, c_int64, c_float, c_int, c_void_p]),
    "hsv_conv1d_c1_strided": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_int64,
                                      c_int, c_int, c_int, c_void_p]),
    "hsv_conv1d_c1_strided_ragged": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                             c_int64, c_int64, c_int, c_int, c_int, c_void_p]),
    "hsv_masked_mean": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_void_p]),
    "hsv_masked_mean_ragged": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_void_p]),
    "hsv_seeded_normal": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int64, c_void_p, c_void_p]),
    "hsv_sample_ragged": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_int, c_int,
                                  c_int64, c_void_p]),
    "hsv_sinegen_workspace": (c_int64, [c_int, c_int64, c_int]),
    "hsv_sinegen": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int, c_float, c_int, c_float,
                            c_void_p]),
    "hsv_peak_norm_pcm16": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int64, c_float, c_float, c_int, c_void_p]),
    "hsv_peak_norm_pcm16_rows": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int64, c_float, c_void_p, c_void_p]),
    "hsv_resample_ragged": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int, c_int,
                                    c_void_p, c_void_p, c_int, c_int64, c_int64, c_void_p]),
}

# bring-up aids exported by the library but not part of the drop-in contract
_EXTRA = {
    "hsv_set_umma_debug": (c_int, [c_int]),
    "hsv_set_act_variant": (c_int, [c_int]),
    "hsv_set_pdl": (c_int, [c_int]),
    "hsv_set_umma_trace": (c_int, [c_void_p]),
}

_lib = None
LAUNCHES = [0]   # number of hsv kernel launches issued through check() (bench.py reports it)


class HsvError(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    """Load libhsv.so (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise HsvError(
            f"{LIB_PATH} not found: build the sm_100a kernels first "
            "(python -m megatts2_hierspeechpp_b200.build, or __graft_entry__.build()); there is no CPU fallback")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in {**SIGNATURES, **_EXTRA}.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    if lib.hsv_version() != 100:
        raise HsvError(f"libhsv.so version {lib.hsv_version()} does not match the Python binding (100)")
    if os.environ.get("HSV_UMMA_DEBUG"):
        lib.hsv_set_umma_debug(int(os.environ["HSV_UMMA_DEBUG"]))
    if os.environ.get("HSV_PDL"):
        lib.hsv_set_pdl(int(os.environ["HSV_PDL"]))
    if os.environ.get("HSV_ACT_VARIANT"):
        lib.hsv_set_act_variant(int(os.environ["HSV_ACT_VARIANT"]))
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    LAUNCHES[0] += 1
    if rc != 0:
        msg = load().hsv_last_error()
        raise HsvError(f"{what} failed (rc={rc}): {msg.decode() if msg else '?'}")
