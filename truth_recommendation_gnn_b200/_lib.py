"""ctypes binding of ``lib/libtrg_b200.so`` (the C ABI in ``include/trg_b200.h``).

There is NO fallback: if the library has not been built, or a tensor is not on a CUDA device,
the call raises.  PyTorch is used only for device memory, streams and autograd plumbing.
"""
from __future__ import annotations

import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libtrg_b200.so")

TRG_F32, TRG_BF16, TRG_F8E4M3 = 0, 1, 2   # TRG_F8E4M3: trg_score_topk(_excluding) only
ABI_VERSION = 4    # TRG_ABI_VERSION of include/trg_b200.h

_vp, _i64, _i32, _sz, _int = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_size_t, ctypes.c_int


class TrgProjTerm(ctypes.Structure):
    _fields_ = [("a", _vp), ("w", _vp), ("k", _i32), ("alpha", ctypes.c_float)]


class TrgLongRows(ctypes.Structure):
    _fields_ = [("vrowptr", _vp), ("vinfo", _vp), ("n_vrows", _i64), ("long_rows", _vp), ("long_ptr", _vp),
                ("n_long", _i64), ("partial", _vp)]


class TrgProjBwdTerm(ctypes.Structure):
    _fields_ = [("w", _vp), ("k", _i32), ("alpha", ctypes.c_float), ("row_scale", _vp), ("d_a", _vp)]


class TrgProjDwTerm(ctypes.Structure):
    _fields_ = [("a", _vp), ("k", _i32), ("alpha", ctypes.c_float), ("d_w", _vp)]


#: every symbol ``include/trg_b200.h`` declares -> (restype, argtypes)
SIGNATURES = {
    "trg_abi_version": (_int, []),
    "trg_last_error": (ctypes.c_char_p, []),
    "trg_launch_count": (_i64, []),
    "trg_csr_workspace_bytes": (_sz, [_i64, _i64]),
    "trg_csr_build": (_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _sz, _vp]),
    "trg_select_range_workspace_bytes": (_sz, [_i64]),
    "trg_select_range": (_int, [_vp, _vp, _i64, _i64, _i64, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _sz, _vp]),
    "trg_sage_agg_fwd": (_int, [_vp, _vp, _vp, _i64, _i32, _int, _vp, _vp, ctypes.POINTER(TrgLongRows), _vp]),
    "trg_sage_agg_bwd": (_int, [_vp, _vp, _vp, _vp, _i64, _i32, _int, _vp, _int, _int, _vp,
                                ctypes.POINTER(TrgLongRows), _vp]),
    "trg_gather_wsum": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _int, _vp, _int, _int, _vp,
                               ctypes.POINTER(TrgLongRows), _vp]),
    "trg_rows_finish": (_int, [_vp, _int, _vp, _vp, _vp, _i64, _i32, _int, _vp, _vp]),
    "trg_peer_reduce_rows": (_int, [_vp, _i32, _i64, _int, _vp, _vp, _vp, _i64, _i32, _int, _vp, _i32, _vp]),
    "trg_edge_bce_workspace_bytes": (_sz, [_i64]),
    "trg_edge_bce_fwd": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _int, _vp, _vp,
                                _vp, _vp, _vp, _vp, _sz, _vp]),
    "trg_edge_anchor_loss": (_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _int, _int, _vp, _vp, _vp,
                                    _vp, _int, _int, _vp, _sz, _vp]),
    "trg_sage_proj_workspace_bytes": (_sz, [_i32, _i32, _int]),
    "trg_sage_proj_fwd": (_int, [ctypes.POINTER(TrgProjTerm), _i32, _vp, _i64, _i32, _int, _int, _vp,
                                 _vp, _sz, _vp]),
    "trg_sage_proj_bwd_input": (_int, [_vp, ctypes.POINTER(TrgProjBwdTerm), _i32, _i64, _i32, _int,
                                       _vp, _sz, _vp]),
    "trg_sage_proj_dw_workspace_bytes": (_sz, []),
    "trg_sage_proj_bwd_weight": (_int, [_vp, ctypes.POINTER(TrgProjDwTerm), _i32, _vp, _i64, _i32, _int,
                                        _vp, _sz, _vp]),
    "trg_score_topk_workspace_bytes": (_sz, [_i64, _i64, _i32, _i32]),
    "trg_score_topk": (_int, [_vp, _vp, _i64, _i64, _i32, _int, _i32, _i64, _vp, _vp, _vp, _sz, _vp]),
    "trg_score_topk_excluding": (_int, [_vp, _vp, _i64, _i64, _i32, _int, _i32, _i64, _vp, _vp, _vp, _vp, _vp,
                                        _vp, _sz, _vp]),
    "trg_topk_merge": (_int, [_vp, _vp, _i64, _i32, _i32, _i32, _vp, _vp, _vp]),
    "trg_rescore_topk_workspace_bytes": (_sz, [_i64, _i32]),
    "trg_rescore_topk": (_int, [_vp, _vp, _i64, _i64, _i32, _int, _vp, _i32, _i64, _i32, _vp, _vp, _vp, _sz,
                                _vp]),
}

_lib = None


class TrgError(RuntimeError):
    pass


def load():
    """Load the kernel library; raise (never fall back) when it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise TrgError(
                f"{LIB_PATH} is missing: build it with `python -m truth_recommendation_gnn_b200.build` "
                "(nvcc, sm_100a). There is no CPU or PyTorch fallback for the hot path.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        if lib.trg_abi_version() != ABI_VERSION:
            raise TrgError("libtrg_b200.so ABI version mismatch; rebuild")
        _lib = lib
    return _lib


def check(rc: int, what: str):
    if rc != 0:
        raise TrgError(f"{what} failed (rc={rc}): {load().trg_last_error().decode()}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL).  Refuses host tensors: no CPU path exists."""
    if t is None:
        return None
    if not t.is_cuda:
        raise TrgError("truth_recommendation_gnn_b200 runs on CUDA (sm_100a) tensors only; got a "
                       f"{t.device} tensor. There is no CPU fallback.")
    if not t.is_contiguous():
        raise TrgError("non-contiguous tensor passed to the C ABI")
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def dtype_code(dt: torch.dtype) -> int:
    if dt == torch.float32:
        return TRG_F32
    if dt == torch.bfloat16:
        return TRG_BF16
    raise TrgError(f"unsupported dtype {dt}: the hot path computes in fp32 or bf16 (fp32 accumulate)")


class Profiler:
    """Optional per-call CUDA-event timing of the C-ABI launches (used by bench.py to measure the
    dominant kernel live, on the launching stream).  Disabled by default: zero overhead."""

    def __init__(self):
        self.enabled = False
        self.records = []   # (name, algorithmic_bytes, start_event, end_event)

    def reset(self):
        self.records = []

    def summary(self):
        """name -> dict(calls, ms, bytes); call after torch.cuda.synchronize()."""
        out = {}
        for name, nbytes, s, e in self.records:
            d = out.setdefault(name, dict(calls=0, ms=0.0, bytes=0))
            d["calls"] += 1
            d["ms"] += s.elapsed_time(e)
            d["bytes"] += int(nbytes)
        return out


PROF = Profiler()


def call(name, nbytes, fn, *args):
    """Invoke a C-ABI function, check its return code, optionally time it with CUDA events."""
    if PROF.enabled:
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        rc = fn(*args)
        e.record()
        PROF.records.append((name, nbytes, s, e))
    else:
        rc = fn(*args)
    check(rc, name)


def launch_count() -> int:
    return int(load().trg_launch_count())
