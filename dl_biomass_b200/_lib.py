"""ctypes binding of libb2pn.so (the C ABI declared in include/b2pn.h).

There is deliberately no fallback: if the library is missing or a call fails, the product path
raises.  Build it with ``python -c "import __graft_entry__ as g; g.build()"`` or
``make -C dl_biomass_b200/csrc``.
"""
from __future__ import annotations

import ctypes
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb2pn.so")
CSRC = os.path.join(_HERE, "csrc")

_lib = None
ABI_VERSION = 7

_vp, _i32, _i64, _f32, _f64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_float, ctypes.c_double

class Mlp3(ctypes.Structure):
    _fields_ = [("c", ctypes.c_int32 * 4), ("act", ctypes.c_int32), ("eps", ctypes.c_float),
                ("momentum", ctypes.c_float), ("w", _vp * 3), ("b", _vp * 3), ("gamma", _vp * 2),
                ("beta", _vp * 2), ("running_mean", _vp * 2), ("running_var", _vp * 2),
                ("num_batches_tracked", _vp * 2)]


class SaArgs(ctypes.Structure):
    _fields_ = [("precision", ctypes.c_int32), ("training", ctypes.c_int32), ("seg_mode", ctypes.c_int32),
                ("K", ctypes.c_int32), ("n_src", ctypes.c_int64), ("n_dst", ctypes.c_int64),
                ("c_in", ctypes.c_int32), ("x_dtype", ctypes.c_int32), ("x", _vp), ("pos_src", _vp),
                ("pos_dst", _vp), ("nbr", _vp), ("cnt", _vp), ("batch", _vp), ("mlp", Mlp3), ("out", _vp),
                ("arg", _vp), ("h1", _vp), ("h2", _vp), ("bn", _vp), ("workspace", _vp),
                ("workspace_bytes", ctypes.c_int64), ("rgrp", _vp), ("row_src", _vp), ("num_rows", _vp),
                ("row_capacity", ctypes.c_int64), ("row_valid", _vp), ("a1", _vp), ("a2", _vp), ("g1", _vp),
                ("g1_ready", ctypes.c_int32), ("sm_limit", ctypes.c_int32), ("deterministic", ctypes.c_int32),
                ("out_bf16", _vp)]


class FpsOptions(ctypes.Structure):
    _fields_ = [("cluster", ctypes.c_int32), ("threads", ctypes.c_int32), ("seed", ctypes.c_uint64), ("rng_state", _vp)]


class SaGrads(ctypes.Structure):
    _fields_ = [("grad_out", _vp), ("grad_w", _vp * 3), ("grad_b", _vp * 3), ("grad_gamma", _vp * 2),
                ("grad_beta", _vp * 2), ("grad_x", _vp)]

class AugmentCloud(ctypes.Structure):
    _fields_ = [("src_off", ctypes.c_int64), ("out_off", ctypes.c_int64), ("uid", ctypes.c_uint64),
                ("n_src", ctypes.c_int32), ("n_keep", ctypes.c_int32), ("n_dup", ctypes.c_int32),
                ("noise_sd", ctypes.c_float), ("cos_a", ctypes.c_float), ("sin_a", ctypes.c_float)]


class HeadArgs(ctypes.Structure):
    _fields_ = [("B", ctypes.c_int32), ("c", ctypes.c_int32 * 4), ("training", ctypes.c_int32), ("p", ctypes.c_float),
                ("eps", ctypes.c_float), ("momentum", ctypes.c_float), ("x", _vp), ("w", _vp * 3), ("b", _vp * 3),
                ("gamma", _vp * 2), ("beta", _vp * 2), ("running_mean", _vp * 2), ("running_var", _vp * 2),
                ("num_batches_tracked", _vp * 2), ("seed", ctypes.c_uint64), ("rng_counter", _vp), ("out", _vp),
                ("xhat", _vp * 2), ("mask", _vp * 2), ("rstd", _vp * 2)]


class HeadGrads(ctypes.Structure):
    _fields_ = [("grad_out", _vp), ("grad_x", _vp), ("grad_w", _vp * 3), ("grad_b", _vp * 3), ("grad_gamma", _vp * 2),
                ("grad_beta", _vp * 2)]


# name -> (restype, argtypes); must list every symbol include/b2pn.h declares (tests check this)
SIGNATURES = {
    "b2pn_abi_version": (ctypes.c_int, []),
    "b2pn_error_string": (ctypes.c_char_p, [ctypes.c_int]),
    "b2pn_launch_count": (_i64, []),
    "b2pn_fps_num_samples": (_i64, [_i64, _f32]),
    "b2pn_fps_f32": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i32, _i64, _vp, _vp, _vp, ctypes.POINTER(FpsOptions), _vp]),
    "b2pn_fps_random_start": (_i64, [ctypes.c_uint64, _i64, _i32, _i64]),
    "b2pn_adam_step": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _f32, _f32, _f32, _f32, _f32, _f32, _vp, _vp]),
    "b2pn_fps_f64": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    "b2pn_ball_query_f32": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i32, _i64, _i64, _f64, _i32, _vp, _vp, _vp]),
    "b2pn_ball_query_workspace_bytes": (_i64, [_i32, _i64]),
    "b2pn_ball_query_grid_f32": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i32, _i64, _i64, _f64, _i32, _vp, _vp, _vp, _i64, _vp]),
    "b2pn_pack_rows_capacity": (_i64, [_i64, _i32]),
    "b2pn_pack_rows_workspace_bytes": (_i64, [_i64]),
    "b2pn_pack_rows": (ctypes.c_int, [_vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "b2pn_sa_workspace_bytes": (_i64, [ctypes.POINTER(SaArgs), _i32]),
    "b2pn_sa_forward": (ctypes.c_int, [ctypes.POINTER(SaArgs), _vp]),
    "b2pn_sa_eval_fused": (ctypes.c_int, [ctypes.POINTER(SaArgs)]),
    "b2pn_augment_batch": (ctypes.c_int, [_vp, _vp, ctypes.c_int32, ctypes.POINTER(AugmentCloud), ctypes.c_int32,
                                          ctypes.c_uint64, _vp, _vp, _vp, _vp, _vp]),
    "b2pn_augment_draw": (ctypes.c_uint64, [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint64]),
    "b2pn_augment_max_points": (ctypes.c_int32, []),
    "b2pn_weighted_mse": (ctypes.c_int, [_vp, _vp, _vp, ctypes.c_int32, ctypes.c_int32, _vp, _vp, _vp]),
    "b2pn_sa_gather_rows": (ctypes.c_int, [ctypes.POINTER(SaArgs), _vp]),
    "b2pn_sa_backward": (ctypes.c_int, [ctypes.POINTER(SaArgs), ctypes.POINTER(SaGrads), _vp]),
    "b2pn_head_forward": (ctypes.c_int, [ctypes.POINTER(HeadArgs), _vp]),
    "b2pn_head_backward": (ctypes.c_int, [ctypes.POINTER(HeadArgs), ctypes.POINTER(HeadGrads), _vp]),
    "b2pn_tc_gemm_selftest": (ctypes.c_int, [_vp, _i32, _i32, _vp, _i32, _i64, _i64, _vp, _vp, _i64, _vp, _i64, _vp]),
}


def cuda_tool(name: str) -> str:
    """Path of a CUDA toolkit program: from PATH, else from $CUDA_HOME/bin (default /usr/local/cuda), since an ordinary
    user's PATH need not hold the toolkit."""
    return shutil.which(name) or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", name)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile libb2pn.so in-tree with nvcc for sm_100a (works without a GPU)."""
    cmd = ["make", "-C", CSRC, "-j8", f"NVCC={cuda_tool('nvcc')}"] + (["-B"] if force else [])
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout[-4000:], res.stderr[-4000:])
    if res.returncode != 0:
        raise RuntimeError("building libb2pn.so failed")
    return LIB_PATH


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: the B200 path has no fallback. Build it with "
                f"`make -C {CSRC}` (nvcc, sm_100a).")
        h = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(h, name)  # AttributeError if the ABI drifted
            fn.restype, fn.argtypes = res, args
        if h.b2pn_abi_version() != ABI_VERSION:
            raise ImportError("libb2pn.so ABI version mismatch; rebuild")
        _lib = h
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().b2pn_error_string(rc)
        raise RuntimeError(f"{what} failed (code {rc}): {msg.decode() if msg else '?'}")
