"""ctypes binding of libodevit.so (the C ABI in include/odevit.h).

There is deliberately NO fallback: if the shared library is missing or a tensor is not on a
CUDA device, the call fails loudly.  Build the library with `python -c "import __graft_entry__ as
g; g.build()"` (or `make -C odevit_b200/csrc`).
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
# ODEVIT_LIB: a diagnostic build of the same library (e.g. the -DATTN_TRACE clock-trace build), never a fallback
LIB_PATH = os.environ.get("ODEVIT_LIB") or os.path.join(_HERE, "csrc", "libodevit.so")

ABI_VERSION = 8

# enums of include/odevit.h
FIELD_PARALLEL, FIELD_PARALLEL_L2, FIELD_MACARON = 0, 1, 2
FP32, BF16 = 0, 1
EULER, MIDPOINT, RK4_38 = 0, 1, 2
WS_FIELD, WS_SOLVE_FWD, WS_SOLVE_BWD, WS_ENCODER_FWD, WS_SOLVE_ADAPTIVE, WS_SOLVE_ADAPTIVE_BWD = 0, 1, 2, 3, 4, 5
ERR_WORKSPACE = -2
ERR_NOT_CONVERGED = -6

METHODS = {"euler": EULER, "midpoint": MIDPOINT, "rk4": RK4_38}
STAGES = {"euler": 1, "midpoint": 2, "rk4": 4}
PRECISIONS = {"fp32": FP32, "bf16": BF16}

_vp = ctypes.c_void_p

WEIGHT_FIELDS = ("norm_a_w", "norm_a_b", "norm_b_w", "norm_b_b", "norm_c_w", "norm_c_b",
                 "in_proj_w", "in_proj_b", "out_proj_w", "out_proj_b", "fc1_w", "fc1_b",
                 "fc2_w", "fc2_b", "res_scale")
MOD_FIELDS = ("mod_attn_scale", "mod_attn_shift", "mod_mlp_scale", "mod_mlp_shift")


class Desc(ctypes.Structure):
    _fields_ = [("abi_version", ctypes.c_int32), ("batch", ctypes.c_int32), ("tokens", ctypes.c_int32),
                ("dim", ctypes.c_int32), ("heads", ctypes.c_int32), ("hidden", ctypes.c_int32),
                ("variant", ctypes.c_int32), ("precision", ctypes.c_int32), ("scaler", ctypes.c_float),
                ("attn_drop", ctypes.c_float), ("proj_drop", ctypes.c_float), ("mlp_drop", ctypes.c_float),
                ("drop_seed_lo", ctypes.c_uint32), ("drop_seed_hi", ctypes.c_uint32),
                ("drop_seed_dev", ctypes.c_void_p)]


class Weights(ctypes.Structure):
    _fields_ = [(n, _vp) for n in WEIGHT_FIELDS + MOD_FIELDS] + [("reserved", _vp * 5)]


class WeightGrads(ctypes.Structure):
    _fields_ = [(n, _vp) for n in WEIGHT_FIELDS] + [("reserved", _vp * 9)]


class OdevitError(RuntimeError):
    pass


_lib: Optional[ctypes.CDLL] = None


def lib() -> ctypes.CDLL:
    """Load libodevit.so once; raise if it is not built (no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise OdevitError(
            f"{LIB_PATH} is missing: the CUDA extension is not built. Run "
            "`python -c \"import __graft_entry__ as g; g.build()\"` or `make -C odevit_b200/csrc`. "
            "odevit_b200 has no CPU or PyTorch fallback for the hot path.")
    L = ctypes.CDLL(LIB_PATH)
    L.odevit_abi_version.restype = ctypes.c_int
    L.odevit_build_info.restype = ctypes.c_char_p
    L.odevit_last_error_string.restype = ctypes.c_char_p
    L.odevit_launch_count.restype = ctypes.c_int64
    L.odevit_reset_launch_count.restype = None
    L.odevit_workspace_bytes.restype = ctypes.c_size_t
    L.odevit_workspace_bytes.argtypes = [ctypes.POINTER(Desc), ctypes.c_int32, ctypes.c_int32]
    L.odevit_field_fwd.restype = ctypes.c_int
    L.odevit_field_fwd.argtypes = [ctypes.POINTER(Desc), ctypes.POINTER(Weights), _vp, _vp, _vp,
                                   _vp, ctypes.c_size_t, _vp]
    L.odevit_field_bwd.restype = ctypes.c_int
    L.odevit_field_bwd.argtypes = [ctypes.POINTER(Desc), ctypes.POINTER(Weights), _vp, _vp, _vp, _vp,
                                   ctypes.POINTER(WeightGrads), _vp, ctypes.c_size_t, _vp]
    L.odevit_solve_fwd.restype = ctypes.c_int
    L.odevit_solve_fwd.argtypes = [ctypes.POINTER(Desc), ctypes.POINTER(Weights), ctypes.c_int32, _vp,
                                   ctypes.POINTER(ctypes.c_float), ctypes.c_int32, _vp, _vp, _vp, _vp,
                                   ctypes.c_int32, _vp, ctypes.c_int32, ctypes.c_int32, _vp, ctypes.c_size_t,
                                   _vp, ctypes.c_size_t, _vp]
    L.odevit_tape_bytes.restype = ctypes.c_size_t
    L.odevit_tape_bytes.argtypes = [ctypes.POINTER(Desc), ctypes.c_int32, ctypes.c_int32]
    L.odevit_encoder_cache_bytes.restype = ctypes.c_size_t
    L.odevit_encoder_cache_bytes.argtypes = [ctypes.POINTER(Desc), ctypes.c_int32]
    L.odevit_encoder_fwd.restype = ctypes.c_int
    L.odevit_encoder_fwd.argtypes = [ctypes.POINTER(Desc), ctypes.POINTER(Weights), ctypes.c_int32, ctypes.c_float, _vp, _vp, _vp,
                                     ctypes.c_int32, _vp, ctypes.c_size_t, ctypes.c_int32, _vp, ctypes.c_size_t, _vp]
    L.odevit_jasmin_rowmax.restype = ctypes.c_int
    L.odevit_jasmin_rowmax.argtypes = [_vp, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, _vp, _vp]
    L.odevit_fd_curvature.restype = ctypes.c_int
    L.odevit_fd_curvature.argtypes = [_vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                      ctypes.c_double, _vp, _vp]
    L.odevit_solve_bwd.restype = ctypes.c_int
    L.odevit_solve_bwd.argtypes = [ctypes.POINTER(Desc), ctypes.POINTER(Weights), ctypes.c_int32,
                                   ctypes.POINTER(ctypes.c_float), ctypes.c_int32, _vp, _vp, _vp,
                                   ctypes.POINTER(ctypes.c_int32), ctypes.c_int32, _vp, _vp,
                                   ctypes.POINTER(WeightGrads), _vp, ctypes.c_size_t, _vp, ctypes.c_size_t, _vp]
    L.odevit_solve_fwd_lean.restype = ctypes.c_int
    L.odevit_solve_fwd_lean.argtypes = [ctypes.POINTER(Desc), ctypes.POINTER(Weights), ctypes.c_int32, _vp,
                                        ctypes.POINTER(ctypes.c_float), ctypes.c_int32, _vp, _vp,
                                        ctypes.POINTER(ctypes.c_int32), ctypes.c_int32, _vp, _vp, _vp, ctypes.c_int32,
                                        ctypes.c_int32, _vp, ctypes.c_size_t, _vp]
    L.odevit_solve_adaptive.restype = ctypes.c_int
    L.odevit_solve_adaptive.argtypes = [ctypes.POINTER(Desc), ctypes.POINTER(Weights), _vp, ctypes.POINTER(ctypes.c_float),
                                        ctypes.c_int32, ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_int32,
                                        _vp, _vp, _vp, _vp, _vp, ctypes.c_size_t, _vp]
    L.odevit_solve_adaptive_record.restype = ctypes.c_int
    L.odevit_solve_adaptive_record.argtypes = [ctypes.POINTER(Desc), ctypes.POINTER(Weights), _vp,
                                               ctypes.POINTER(ctypes.c_float), ctypes.c_int32, ctypes.c_double,
                                               ctypes.c_double, ctypes.c_double, ctypes.c_int32, _vp, _vp, _vp, _vp,
                                               ctypes.c_int32, _vp, _vp, _vp, _vp, ctypes.c_size_t, _vp]
    L.odevit_adaptive_tape_bytes.restype = ctypes.c_size_t
    L.odevit_adaptive_tape_bytes.argtypes = [ctypes.POINTER(Desc), ctypes.c_int32]
    L.odevit_solve_adaptive_bwd.restype = ctypes.c_int
    L.odevit_solve_adaptive_bwd.argtypes = [ctypes.POINTER(Desc), ctypes.POINTER(Weights), _vp,
                                            ctypes.POINTER(ctypes.c_float), ctypes.c_int32, _vp, _vp, _vp,
                                            ctypes.c_int32, ctypes.POINTER(ctypes.c_int32), _vp, _vp,
                                            ctypes.POINTER(WeightGrads), _vp, _vp, ctypes.c_size_t, _vp,
                                            ctypes.c_size_t, _vp]
    L.odevit_solve_uses_resident.restype = ctypes.c_int
    L.odevit_solve_uses_resident.argtypes = [ctypes.POINTER(Desc), ctypes.c_int32, ctypes.c_int32]
    L.odevit_tokens_fwd.restype = ctypes.c_int
    L.odevit_tokens_fwd.argtypes = [_vp, _vp] + [ctypes.c_int32] * 6 + [_vp, _vp, _vp, ctypes.c_int32, _vp, _vp]
    L.odevit_head_ce_fwd.restype = ctypes.c_int
    L.odevit_head_ce_fwd.argtypes = [_vp, ctypes.c_int64, _vp, _vp, _vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                     ctypes.c_float, _vp, _vp, _vp, _vp]
    L.odevit_head_ce_bwd.restype = ctypes.c_int
    L.odevit_head_ce_bwd.argtypes = [_vp, ctypes.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, ctypes.c_int32, ctypes.c_int32,
                                     ctypes.c_int32, ctypes.c_float, _vp, _vp, ctypes.c_int64, _vp, _vp, _vp]
    L.odevit_extract_mass_fwd.restype = ctypes.c_int
    L.odevit_extract_mass_fwd.argtypes = [_vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_float, ctypes.c_int32,
                                          ctypes.c_float, _vp, _vp, _vp, _vp]
    L.odevit_extract_mass_bwd.restype = ctypes.c_int
    L.odevit_extract_mass_bwd.argtypes = [_vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_float, ctypes.c_int32,
                                          ctypes.c_float, _vp, _vp, _vp, _vp]
    L.odevit_pil_bilinear_ksize.restype = ctypes.c_int
    L.odevit_pil_bilinear_ksize.argtypes = [ctypes.c_int32, ctypes.c_int32]
    L.odevit_pil_bilinear_tables.restype = ctypes.c_int
    L.odevit_pil_bilinear_tables.argtypes = [ctypes.c_int32, ctypes.c_int32, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32)]
    L.odevit_preprocess_u8.restype = ctypes.c_int
    L.odevit_preprocess_u8.argtypes = [_vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, _vp, _vp,
                                       _vp, _vp, ctypes.c_float, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float),
                                       _vp, _vp, _vp, _vp]
    L.odevit_drop_state_advance.restype = ctypes.c_int
    L.odevit_drop_state_advance.argtypes = [_vp, _vp]
    L.odevit_gemm_bf16.restype = ctypes.c_int
    L.odevit_gemm_bf16.argtypes = [ctypes.c_int32] * 4 + [_vp, _vp, _vp, ctypes.c_int32, ctypes.c_int32, _vp]
    L.odevit_profile_enable.restype = ctypes.c_int
    L.odevit_profile_enable.argtypes = [ctypes.c_int32]
    L.odevit_profile_reserve.restype = ctypes.c_int
    L.odevit_profile_reserve.argtypes = [ctypes.c_int32]
    L.odevit_profile_num_classes.restype = ctypes.c_int
    L.odevit_profile_class_name.restype = ctypes.c_char_p
    L.odevit_profile_class_name.argtypes = [ctypes.c_int32]
    L.odevit_profile_read.restype = ctypes.c_int
    L.odevit_profile_read.argtypes = [ctypes.c_int32, ctypes.POINTER(ctypes.c_double),
                                      ctypes.POINTER(ctypes.c_int64)]
    if L.odevit_abi_version() != ABI_VERSION:
        raise OdevitError(f"libodevit.so ABI {L.odevit_abi_version()} != binding ABI {ABI_VERSION}; rebuild")
    _lib = L
    return L


def check(status: int, what: str) -> None:
    if status != 0:
        msg = lib().odevit_last_error_string().decode("utf-8", "replace")
        raise OdevitError(f"{what} failed with status {status}: {msg}")


def launch_count() -> int:
    return int(lib().odevit_launch_count())


def reset_launch_count() -> None:
    lib().odevit_reset_launch_count()


def profile_enable(on: bool) -> None:
    check(lib().odevit_profile_enable(1 if on else 0), "odevit_profile_enable")


def profile_reserve(pairs: int) -> None:
    check(lib().odevit_profile_reserve(int(pairs)), "odevit_profile_reserve")


def profile_read() -> dict:
    """{class name: (total_ms, launches)} of the launches recorded since profile_enable(True)."""
    L = lib()
    out = {}
    for k in range(L.odevit_profile_num_classes()):
        ms, n = ctypes.c_double(0), ctypes.c_int64(0)
        check(L.odevit_profile_read(k, ctypes.byref(ms), ctypes.byref(n)), "odevit_profile_read")
        if n.value:
            out[L.odevit_profile_class_name(k).decode()] = (ms.value, n.value)
    return out


DECLARED_SYMBOLS = ("odevit_abi_version", "odevit_build_info", "odevit_last_error_string",
                    "odevit_workspace_bytes", "odevit_field_fwd", "odevit_solve_fwd", "odevit_solve_bwd",
                    "odevit_field_bwd", "odevit_tape_bytes", "odevit_fd_curvature", "odevit_jasmin_rowmax", "odevit_encoder_cache_bytes", "odevit_encoder_fwd", "odevit_launch_count", "odevit_reset_launch_count", "odevit_drop_state_advance", "odevit_solve_fwd_lean", "odevit_solve_adaptive", "odevit_solve_adaptive_record", "odevit_adaptive_tape_bytes", "odevit_solve_adaptive_bwd", "odevit_solve_uses_resident", "odevit_tokens_fwd", "odevit_head_ce_fwd", "odevit_head_ce_bwd", "odevit_extract_mass_fwd", "odevit_extract_mass_bwd", "odevit_pil_bilinear_ksize", "odevit_pil_bilinear_tables", "odevit_preprocess_u8",
                    "odevit_gemm_bf16", "odevit_profile_enable", "odevit_profile_reserve", "odevit_profile_num_classes", "odevit_profile_class_name",
                    "odevit_profile_read")
