"""ctypes binding of libadapose_b200.so (include/adapose_b200.h).  There is no fallback: if the CUDA library is
missing or a call fails the product path raises."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libadapose_b200.so")

ADP_ABI_VERSION = 6
DT_U8, DT_F32, DT_F64 = 0, 1, 2
ACT_NONE, ACT_RELU, ACT_PRELU, ACT_TANH = 0, 1, 2, 3
LAYOUT_F16, LAYOUT_S2D = 1, 2          # adp_decode x11_format / adp_conv0_plan_create flags
TC_PLAN_INFO_LEN = 16                  # int32 fields of adp_conv_tc_plan_info

vp = C.c_void_p
i32 = C.c_int32


class AdpError(RuntimeError):
    pass


class Act(C.Structure):
    _fields_ = [("hi", vp), ("lo", vp), ("B", i32), ("D", i32), ("H", i32), ("W", i32), ("C", i32), ("f16", i32), ("q8", vp)]


class TcGeom(C.Structure):
    _fields_ = [("ntaps", i32), ("dz", C.c_int8 * 32), ("dy", C.c_int8 * 32), ("dx", C.c_int8 * 32), ("wt", C.c_int8 * 32),
                ("in_mul", i32), ("out_mul", i32), ("out_oz", i32), ("out_oy", i32), ("out_ox", i32),
                ("gD", i32), ("gH", i32), ("gW", i32), ("oD", i32), ("oH", i32), ("oW", i32), ("w_taps", i32)]


class Epilogue(C.Structure):
    _fields_ = [("scale", vp), ("bias", vp), ("prelu", C.c_float), ("act", i32), ("res_after_act", i32),
                ("res_hi", vp), ("res_lo", vp), ("res_cstride", i32), ("out_hi", vp), ("out_lo", vp), ("out_f32", vp), ("out_h16", vp),
                ("out_cstride", i32), ("out_coff", i32), ("bias_per_batch", i32), ("out_q8", vp), ("check_finite", i32)]


DECODE_FIELDS = ["ic_w", "ic_b", "nh0_w", "nh0_b", "nh1_w", "nh1_b", "nh2_w", "nh2_b", "np0_w", "np0_b", "np1_w", "np1_b",
                 "pm0_w", "pm0_b", "pm1_w", "pm1_b", "q0_w", "q0_b", "q1_w", "q1_b", "r0_w", "r0_b", "r1_w", "r1_b",
                 "r2_w", "r2_b", "prob_w"]


class DecodeWeights(C.Structure):
    _fields_ = [(n, vp) for n in DECODE_FIELDS]


# name -> (restype, argtypes); the list doubles as the export check in tests/test_abi.py
SIGNATURES = {
    "adp_abi_version": (C.c_int, []),
    "adp_last_error": (C.c_char_p, []),
    "adp_launch_count": (C.c_uint64, []),
    "adp_launch_count_add": (None, [C.c_uint64]),
    "adp_device_info": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "adp_preprocess": (C.c_int, [vp, C.c_int, vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                 C.c_uint32, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp]),
    "adp_mask_windows": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp]),
    "adp_conv_tc_plan": (C.c_int, [C.POINTER(vp), C.POINTER(Act), vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.POINTER(Epilogue), C.POINTER(TcGeom), C.c_int]),
    "adp_conv_tc_run": (C.c_int, [vp, C.c_int, vp, vp]),
    "adp_conv_tc_plan_info": (C.c_int, [vp, vp]),
    "adp_conv_tc_free": (None, [vp]),
    "adp_maxpool3x3s2": (C.c_int, [C.POINTER(Act), C.POINTER(Act), C.c_int, vp]),
    "adp_psp_priors": (C.c_int, [C.POINTER(Act), C.c_int, vp, vp, vp, C.c_int, vp]),
    "adp_psp_fill_priors": (C.c_int, [vp, C.POINTER(Act), C.c_int, C.c_int, vp]),
    "adp_upsample2x": (C.c_int, [C.POINTER(Act), C.POINTER(Act), C.c_int, vp]),
    "adp_upconv_blend": (C.c_int, [vp, vp, vp, C.c_float, C.c_int, vp]),
    "adp_pack_s2d": (C.c_int, [vp, C.POINTER(Act), C.c_int, C.c_int, vp]),
    "adp_conv0_plan_create": (C.c_int, [C.POINTER(vp), C.POINTER(Act), vp, vp, vp, vp, C.c_int, C.c_int]),
    "adp_conv0_run": (C.c_int, [vp, C.c_int, vp, vp]),
    "adp_conv0_free": (None, [vp]),
    "adp_tconv_plan_create": (C.c_int, [C.POINTER(vp), C.POINTER(Act), vp, C.c_int, vp, vp, vp, C.c_int, vp, C.c_int, C.c_int]),
    "adp_tconv_run": (C.c_int, [vp, C.c_int, vp, vp]),
    "adp_tconv_free": (None, [vp]),
    "adp_warp_matrices": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, C.c_int, vp]),
    "adp_build_volume": (C.c_int, [vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp]),
    "adp_decode_gather": (C.c_int, [vp] * 15 + [C.c_int] * 5 + [vp]),
    "adp_colsum": (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp]),
    "adp_pose_gbias": (C.c_int, [vp, vp, vp, vp, vp, C.c_int, C.c_int, vp]),
    "adp_rot_head": (C.c_int, [vp, vp, C.POINTER(DecodeWeights), vp, vp, C.c_int, C.c_int, vp]),
    "adp_actor_forward": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, C.c_int, vp, vp, vp]),
    "adp_fit": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp]),
    "adp_nocs_match": (C.c_int, [vp] * 10 + [C.c_int] + [vp] * 5 + [C.c_int, C.c_int, vp]),
    "adp_view_fusion": (C.c_int, [vp] * 14 + [C.c_int] * 4 + [vp]),
    "adp_fit_umeyama": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, C.c_uint32, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp]),
}

_lib = None


def load():
    """Load the shared library (building is a separate, explicit step: ``python -m rgbmanip_b200.build``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AdpError(f"{LIB_PATH} is missing: build it with `python -m rgbmanip_b200.build` "
                       "(nvcc, sm_100a).  There is no CPU or PyTorch fallback for this path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError -> the library does not match include/adapose_b200.h
        fn.restype = res
        fn.argtypes = args
    if lib.adp_abi_version() != ADP_ABI_VERSION:
        raise AdpError(f"ABI mismatch: library {lib.adp_abi_version()} vs binding {ADP_ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().adp_last_error()
        raise AdpError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")


def ptr(t):
    """Raw device/host pointer of a torch tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())
