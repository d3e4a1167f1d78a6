"""ctypes binding of ``librlctr_sm100a.so`` (the C ABI declared in ``include/rlctr.h``).

PyTorch is plumbing here: it owns device memory and streams; every hot-path computation is a
call into the library with raw device pointers and the current CUDA stream.  There is no
fallback: if the library is missing or a tensor is not on a CUDA device, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "librlctr_sm100a.so")

RLCTR_FM_TERM = 1
RLCTR_STAGED_PARTNER = 1
RLCTR_DZ_IN_SUMS = 2
RLCTR_EUNSUPPORTED = -2
RLCTR_REDUCE_WS_BYTES = 16640
RLCTR_DENSE_MAX = 24
RLCTR_MLP_RELU = 1
RLCTR_MLP_DROPOUT = 2
RLCTR_MLP_DX_MASK = 4
RLCTR_MLP_W_PRESPLIT = 16
RLCTR_MLP_FP32 = 8


class RlctrError(RuntimeError):
    pass


class Table(C.Structure):
    """struct rlctr_table"""
    _fields_ = [("data", C.c_void_p), ("n_rows", C.c_int64), ("row_stride", C.c_int32),
                ("lin_col", C.c_int32), ("emb_col", C.c_int32), ("dim", C.c_int32), ("row_pitch", C.c_int32),
                ("world", C.c_int32), ("peers", C.c_void_p * 8)]


class Adam(C.Structure):
    """struct rlctr_adam"""
    _fields_ = [("exp_avg", C.c_void_p), ("exp_avg_sq", C.c_void_p), ("stamp", C.c_void_p),
                ("sched", C.c_void_p), ("step", C.c_void_p), ("sched_len", C.c_int32), ("stamp_col", C.c_int32),
                ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double), ("weight_decay", C.c_double),
                ("stage", C.c_void_p)]


class Adagrad(C.Structure):
    """struct rlctr_adagrad"""
    _fields_ = [("state_sum", C.c_void_p), ("stamp", C.c_void_p), ("clr", C.c_void_p), ("step", C.c_void_p),
                ("sched_len", C.c_int32), ("stamp_col", C.c_int32), ("eps", C.c_double), ("weight_decay", C.c_double)]


class Lookup(C.Structure):
    """struct rlctr_lookup"""
    _fields_ = [("stage", C.c_void_p), ("world", C.c_int32), ("n_per_rank", C.c_uint32), ("gathered", C.c_void_p * 8)]


class RowGrad(C.Structure):
    """struct rlctr_rowgrad"""
    _fields_ = [("staged", C.c_void_p), ("dlogit", C.c_void_p), ("sums", C.c_void_p),
                ("extra", C.c_void_p), ("fields", C.c_int32), ("flags", C.c_int32),
                ("world", C.c_int32), ("n_per_rank", C.c_uint32), ("peer_staged", C.c_void_p * 8),
                ("peer_dlogit", C.c_void_p * 8), ("peer_sums", C.c_void_p * 8), ("peer_extra", C.c_void_p * 8)]


class Member(C.Structure):
    """struct rlctr_member: one model's view of a co-located record"""
    _fields_ = [("lin_col", C.c_int32), ("emb_col", C.c_int32), ("dim", C.c_int32), ("flags", C.c_int32),
                ("bias", C.c_void_p), ("logit", C.c_void_p), ("pctr", C.c_void_p), ("pctr_stride", C.c_int64),
                ("rows_out", C.c_void_p), ("rows_pitch", C.c_int64), ("dlogit", C.c_void_p), ("extra", C.c_void_p),
                ("extra_pitch", C.c_int64)]


RLCTR_GROUP_MAX = 4

_P, _I64, _I32, _SZ, _F = C.c_void_p, C.c_int64, C.c_int32, C.c_size_t, C.c_double
_TP, _AP, _GP, _LP = C.POINTER(Table), C.POINTER(Adam), C.POINTER(RowGrad), C.POINTER(Lookup)
_MP = C.POINTER(Member)
_AGP = C.POINTER(Adagrad)

# name -> (restype, argtypes); must list every symbol include/rlctr.h declares
SIGNATURES = {
    "rlctr_version": (C.c_int, []),
    "rlctr_strerror": (C.c_char_p, [C.c_int]),
    "rlctr_launch_count": (C.c_ulonglong, []),
    "rlctr_embed_fwd": (C.c_int, [_P, _TP, _P, _P, _P, _I64, _P, _P, _I64, _I64, _I32, _I32, _P]),
    "rlctr_pairdots_fwd": (C.c_int, [_P, _I64, _P, _I64, _I64, _I32, _I32, _I32, _P]),
    "rlctr_pairdots_bwd": (C.c_int, [_P, _I64, _P, _I64, _P, _I64, _I64, _I32, _I32, _I32, _P]),
    "rlctr_cross_ws_bytes": (_SZ, [_I64, _I32, _I32]),
    "rlctr_cross_fwd": (C.c_int, [_P, _I64, _P, _P, _I32, _P, _I64, _P, _I64, _I32, _P]),
    "rlctr_cross_bwd": (C.c_int, [_P, _I64, _P, _P, _P, _I32, _P, _I64, _P, _I64, _P, _P, _I64, _I32, _P, _SZ, _P]),
    "rlctr_fieldsq_fwd": (C.c_int, [_P, _I64, _P, _I64, _I64, _I32, _I32, _P]),
    "rlctr_fieldsq_bwd": (C.c_int, [_P, _I64, _P, _I64, _P, _I64, _I64, _I32, _I32, _P]),
    "rlctr_afm_ws_bytes": (_SZ, [_I64, _I32]),
    "rlctr_afm_fwd": (C.c_int, [_P, _I64, _P, _P, _I64, _I32, _I32, C.c_float, _P, _P, _P]),
    "rlctr_afm_bwd": (C.c_int, [_P, _I64, _P, _P, _P, _I64, _P, _I64, _I32, _I32, C.c_float, _P, _P, _P, _SZ, _P]),
    "rlctr_replay_store": (C.c_int, [_P, _I64, _I32, _I64, _P, _I64, _I64, _P]),
    "rlctr_replay_gather": (C.c_int, [_P, _I32, _P, _I64, _P, _P]),
    "rlctr_replay_update": (C.c_int, [_P, _I32, _P, _P, _I64, _P]),
    "rlctr_replay_sample_uniform": (C.c_int, [_I64, _I64, _P, _P, _P]),
    "rlctr_replay_per_ws_bytes": (_SZ, [_I64]),
    "rlctr_replay_sample_per": (C.c_int, [_P, _I32, _I64, C.c_float, C.c_float, C.c_float, _I32, _I64, _P, _P, _P, _P, _SZ, _P]),
    "rlctr_push_rows": (C.c_int, [_P, _I64, _I32, _I32, _I64, _P, _I32, _P, _P]),
    "rlctr_gae_ws_bytes": (_SZ, [_I64]),
    "rlctr_gae_scan": (C.c_int, [_P, _I64, _F, _P, _P, _SZ, _P]),
    "rlctr_gather_rows": (C.c_int, [_P, _I64, _TP, _P, _P]),
    "rlctr_ffm_fwd": (C.c_int, [_P, _TP, _P, _P, _P, _I64, _P, _I64, _I32, _I32, _P]),
    "rlctr_featemb_fwd": (C.c_int, [_P, _TP, _P, _I64, _I64, _I32, _P]),
    "rlctr_bn_relu_fwd": (C.c_int, [_P, _I64, _P, _P, _P, _P, C.c_float, C.c_float, _P, _I64, _P, _P, _I64, _I32, _I32, _P]),
    "rlctr_bn_relu_bwd": (C.c_int, [_P, _I64, _P, _I64, _P, _I64, _P, _P, _P, _P, _I64, _P, _P, _I64, _I32, _I32, _P]),
    "rlctr_bce_fwd_bwd": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _I64, _P]),
    "rlctr_sigmoid_bwd": (C.c_int, [_P, _P, _P, _P, _P, _I64, _P]),
    "rlctr_sort_ws_bytes": (_SZ, [_I64, _I64]),
    "rlctr_sort_ids": (C.c_int, [_P, _I64, _I64, _P, _P, _P, _SZ, _P]),
    "rlctr_sort_ids_sharded": (C.c_int, [_P, _I64, _I32, _I32, _I64, _P, _P, _P, _SZ, _P]),
    "rlctr_route_ws_bytes": (_SZ, [_I64, _I32]),
    "rlctr_route_ids": (C.c_int, [_P, _I64, _I32, _I32, _I64, _I64, _P, _P, _P, _P, _SZ, _P]),
    "rlctr_sort_routed": (C.c_int, [_P, _P, _I64, _I64, _P, _P, _P, _SZ, _P]),
    "rlctr_rows_ws_bytes": (_SZ, [_I64]),
    "rlctr_rows_adam": (C.c_int, [_P, _P, _I64, _GP, _TP, _AP, _P, _SZ, _P]),
    "rlctr_group_fwd": (C.c_int, [_P, _TP, _MP, _I32, _P, _I32, _I64, _I32, _P]),
    "rlctr_group_rows_adam": (C.c_int, [_P, _P, _I64, _TP, _AP, _MP, _I32, _P, _I32, _I32, _I32, _P, _P, _SZ, _P]),
    "rlctr_sort_routed_pos": (C.c_int, [_P, _I64, _I64, _P, _P, _P, _SZ, _P]),
    "rlctr_push_rows_routed": (C.c_int, [_P, _I64, _I32, _I32, _I64, _P, _I32, _P, _P]),
    "rlctr_push_rows_routed_multi": (C.c_int, [_P, _I64, _I32, _I32, _I64, _P, _P, _I32, _P, _P]),
    "rlctr_rows_grad_dense": (C.c_int, [_P, _P, _I64, _GP, _TP, _P, _P, _SZ, _P]),
    "rlctr_lookup_stage_floats": (_I64, [_TP]),
    "rlctr_rows_lookup": (C.c_int, [_P, _P, _I64, _TP, _AP, _LP, _P, _SZ, _P]),
    "rlctr_rows_catchup": (C.c_int, [_P, _I64, _TP, _AP, _P]),
    "rlctr_rows_claim_bytes": (_SZ, [_I64]),
    "rlctr_rows_catchup_ids": (C.c_int, [_P, _I64, _TP, _AP, _P, _SZ, _P]),
    "rlctr_adam_flush": (C.c_int, [_TP, _AP, _I64, _I64, _P]),
    "rlctr_dense_adam": (C.c_int, [_P, _P, _P, _P, _I64, _P, _P, _F, _F, _F, _F, _P]),
    "rlctr_dense_adam_multi": (C.c_int, [_P, _P, _P, _P, _P, _I32, _P, _P, _P, _F, _F, _F, _F, _P]),
    "rlctr_steps_advance": (C.c_int, [_P, _P, _I32, _P]),
    "rlctr_step_advance": (C.c_int, [_P, _I32, _P]),
    "rlctr_rows_adagrad": (C.c_int, [_P, _P, _I64, _GP, _TP, _AGP, _P, _SZ, _P]),
    "rlctr_group_rows_adagrad": (C.c_int, [_P, _P, _I64, _TP, _AGP, _MP, _I32, _P, _I32, _I32, _I32, _P, _P, _SZ, _P]),
    "rlctr_adagrad_catchup": (C.c_int, [_P, _I64, _TP, _AGP, _P]),
    "rlctr_adagrad_flush": (C.c_int, [_TP, _AGP, _I64, _I64, _P]),
    "rlctr_dense_adagrad_multi": (C.c_int, [_P, _P, _P, _P, _I32, _P, _P, _P, _F, _F, _P]),
    "rlctr_generate_preds": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _I64, _I32, _I32, _P]),
    "rlctr_generate_preds_v10_ws_bytes": (_SZ, [_I64]),
    "rlctr_generate_preds_v10": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _I64, _I32, _P, _SZ, _P]),
    "rlctr_reinforce_loss_bwd": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _I64, _I32, _I32, _P]),
    "rlctr_auc_ws_bytes": (_SZ, [_I64]),
    "rlctr_auc_logloss": (C.c_int, [_P, _P, _P, _I64, _P, _P, _SZ, _P]),
    "rlctr_mlp_ws_bytes": (_SZ, [_I64, _I32, _I32]),
    "rlctr_rng_advance": (C.c_int, [_P, C.c_uint64, _P]),
    "rlctr_linear_fwd": (C.c_int, [_P, _I64, _P, _P, _P, _I64, _I32, _I32, _I32, C.c_float, _P, _P, _SZ, _P]),
    "rlctr_linear_bwd": (C.c_int, [_P, _I64, _P, _P, _P, _P, _P, _P, _I64, _I32, _I32, _I32, C.c_float, C.c_float, _P, _SZ, _P]),
    "rlctr_bucket_ws_bytes": (_SZ, [_I64, _I32]),
    "rlctr_bucket_by_owner": (C.c_int, [_P, _I64, _I32, _I64, _P, _P, _P, _P, _P, _SZ, _P]),
}

_lib = None


def load() -> C.CDLL:
    """Load the library once; raise loudly if it was not built (no CPU or eager fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RlctrError(
            f"{LIB_PATH} is missing: build it with `python -m rl_ctr_prediction_b200.build` "
            "(nvcc, sm_100a). There is no fallback path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)            # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


# the shape limits behind RLCTR_EUNSUPPORTED of the entry points the field count F and the latent size D reach: every model serves
# 2 <= F <= 64 and 1 <= D <= 32 within these (AFM only up to F = 23, DCN and FFM only up to their per-row limits)
SHAPE_LIMITS = {
    "rlctr_pairdots_fwd": "InnerPNN pair dots: 2 <= F <= 64",
    "rlctr_pairdots_bwd": "InnerPNN pair dots: 2 <= F <= 64",
    "rlctr_ffm_fwd": "FFM: 2 <= F <= 64 (one sample's F rows in at most 227 KB of shared memory)",
    "rlctr_embed_fwd": "fused rows of at most 36 floats (D <= 32 with a first-order column, 36 without)",
    "rlctr_afm_fwd": "AFM: D <= 32, F <= 23",
    "rlctr_afm_bwd": "AFM: D <= 32, F <= 23",
    "rlctr_cross_fwd": "DCN: F*D <= 512, at most 8 cross layers",
    "rlctr_cross_bwd": "DCN: F*D <= 512, at most 6 cross layers",
    "rlctr_rows_adam": "fused rows of at most 512 floats (FFM: F*D + 1 <= 512)",
    "rlctr_group_fwd": "joint rows of at most 128 floats (four 128-byte lines), members' stand-alone rows of at most 36 floats; "
                       "one-line records: tower-member tiles of 48 KB per 8 samples (sum of F*D over tower members <= 1496)",
    "rlctr_group_rows_adam": "joint rows of at most 128 floats (four 128-byte lines), members' stand-alone rows of at most 36 floats",
    "rlctr_rows_catchup": "records with an in-record stamp: rows of at most 128 floats",
    "rlctr_adam_flush": "records with an in-record stamp: rows of at most 128 floats",
    "rlctr_rows_adagrad": "fused rows of at most 512 floats (FFM: F*D + 1 <= 512)",
    "rlctr_group_rows_adagrad": "joint rows of at most 128 floats (four 128-byte lines), members' stand-alone rows of at most 36 floats",
    "rlctr_adagrad_catchup": "records with an in-record stamp: rows of at most 128 floats",
    "rlctr_adagrad_flush": "records with an in-record stamp: rows of at most 128 floats",
    "rlctr_dense_adagrad_multi": "at most RLCTR_DENSE_MAX (24) tensors per call",
}


def check(code: int, what: str) -> None:
    if code != 0:
        msg = load().rlctr_strerror(code).decode()
        limit = SHAPE_LIMITS.get(what.split("[")[0]) if code == RLCTR_EUNSUPPORTED else None
        raise RlctrError(f"{what} failed: {msg} (code {code})" + (f"; supported: {limit}" if limit else ""))


def ptr(t):
    """Device pointer of a CUDA tensor (None -> NULL).  Refuses host tensors: no CPU path."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RlctrError("rlctr kernels need CUDA tensors (sm_100a); there is no CPU fallback")
    if not t.is_contiguous():
        raise RlctrError("rlctr kernels need contiguous tensors")
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


# ---------------------------------------------------------------------------------------------------
# optional per-kernel timing (bench.py): CUDA events on the launching stream around a C-ABI call
# ---------------------------------------------------------------------------------------------------
class KernelTimer:
    """Collects (start, stop) CUDA events per named call; ``summary(alg_fn)`` turns them into
    {name: (launches, mean ms, algorithmic bytes per launch)} after a synchronize."""

    def __init__(self):
        self.records = {}

    def add(self, key, e0, e1, meta):
        self.records.setdefault(key, []).append((e0, e1, meta))

    def summary(self, alg_fn=None):
        torch.cuda.synchronize()
        out = {}
        for key, recs in self.records.items():
            ms = [a.elapsed_time(b) for a, b, _ in recs]
            alg = 0.0
            if alg_fn is not None:
                alg = sum(alg_fn(key, m) for _, _, m in recs) / len(recs)
            out[key] = (len(recs), sum(ms) / len(ms), alg)
        return out


_timer = None


def set_timer(t):
    global _timer
    _timer = t


def timing() -> bool:
    return _timer is not None


def call(name, fn, *args, key=None, meta=None):
    """Invoke a C-ABI entry point, raise on a non-zero code; time it if a KernelTimer is installed."""
    t = _timer
    if t is None:
        check(fn(*args), name)
        return
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    rc = fn(*args)
    e1.record()
    check(rc, name)
    t.add(key or name, e0, e1, meta or {})
