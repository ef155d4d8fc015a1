"""ctypes binding of librank_b200.so (include/rank_b200.h).

There is exactly one compute path: the CUDA library.  If it cannot be loaded, every op raises —
there is no eager/CPU fallback.  Torch is used for device memory and streams only; tensors
cross the boundary as raw device pointers.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import torch

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "librank_b200.so"

RK_MAX_FIELDS = 24
RK_MAX_TABLES = 32
RK_MAX_LAYERS = 8
RK_DIRECT_MAX_N = 8192
RK_ADAM_MAX_TENSORS = 64
ABI_VERSION = 3


class RkField(C.Structure):
    _fields_ = [("weight", C.c_void_p), ("idx", C.c_void_p), ("rows", C.c_int64),
                ("dim", C.c_int32), ("out_off", C.c_int32)]


class RkGradTable(C.Structure):
    _fields_ = [("g", C.c_void_p), ("ld", C.c_int64), ("dw", C.c_void_p),
                ("dim", C.c_int32), ("field", C.c_int32)]


class RkDirectTable(C.Structure):
    _fields_ = [("idx", C.c_void_p), ("g", C.c_void_p), ("ld", C.c_int64), ("dw", C.c_void_p),
                ("rows", C.c_int64), ("n", C.c_int64), ("dim", C.c_int32), ("reserved", C.c_int32)]


class RkDinArgs(C.Structure):
    _fields_ = [("cat", C.c_void_p), ("n_cat", C.c_int32), ("n_dense", C.c_int32),
                ("dense_cols", C.c_void_p), ("dense_stride", C.c_int64),
                ("target", RkField), ("history", RkField), ("hist_len", C.c_void_p),
                ("T", C.c_int32), ("att_off", C.c_int32), ("width", C.c_int32),
                ("l2_from", C.c_int32), ("use_softmax", C.c_int32), ("precision", C.c_int32),
                ("mlp", C.c_void_p),
                ("B", C.c_int64),
                ("mlp_tiles", C.c_void_p)]


class RkBstBlock(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "pos", "wq", "bq", "wk", "bk", "wv", "bv", "wo", "bo", "ln1_g", "ln1_b", "w1", "b1", "w2", "b2",
        "ln2_g", "ln2_b", "rng")] + [("dropout_p", C.c_float), ("precision", C.c_int32)]


BST_FP32, BST_BF16_TENSOR = 0, 1


class RkAdamTensor(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "param", "exp_avg", "exp_avg_sq", "step", "grad", "touched_rows", "touched_values", "touched_count")] + [
        ("capacity", C.c_int64), ("rows", C.c_int64), ("dim", C.c_int32), ("lr", C.c_float),
        ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float), ("reserved", C.c_int32)]


LIVE_ALL, LIVE_PREFIX, LIVE_PREFIX_OR_EMPTY = 0, 1, 2

METRICS_NONFINITE, METRICS_BAD_LABEL, METRICS_BAD_GROUP, METRICS_OVERFLOW, METRICS_NOT_PROB = 1, 2, 4, 8, 16


class RkMetricsResult(C.Structure):
    _fields_ = [("pos", C.c_uint64), ("neg", C.c_uint64), ("u2", C.c_uint64), ("correct", C.c_uint64),
                ("logloss_sum", C.c_double), ("valid_groups", C.c_uint64), ("uauc_sum", C.c_double)]


RK_BATCH_MAX_COLS = 32
BATCH_WINDOW, BATCH_BAD_ROW, BATCH_SEQ_OVERFLOW = 1, 2, 4


class RkBatchCol(C.Structure):
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("row_bytes", C.c_int64)]


class RkBatchSeq(C.Structure):
    _fields_ = [("values", C.c_void_p), ("offsets", C.c_void_p), ("dst", C.c_void_p), ("dst_len", C.c_void_p),
                ("width", C.c_int32), ("reserved", C.c_int32)]


ENCODE_TABLE_FULL, ENCODE_SPLIT_COUNT = 1, 2


class RkVocab(C.Structure):
    _fields_ = [("bytes", C.c_void_p), ("offsets", C.c_void_p), ("pos", C.c_void_p), ("slots", C.c_void_p),
                ("n_keys", C.c_int64), ("n_slots", C.c_int64)]


class RkStrCol(C.Structure):
    _fields_ = [("bytes", C.c_void_p), ("offsets", C.c_void_p), ("valid", C.c_void_p), ("valid_bit0", C.c_int64),
                ("n", C.c_int64)]


_P = C.c_void_p
_I = C.c_int
_L = C.c_int64
_Z = C.c_size_t
_F = C.c_float

# name -> (restype, argtypes); mirrors include/rank_b200.h one to one
PROTOTYPES = {
    "rk_version": (_I, []),
    "rk_last_error": (C.c_char_p, []),
    "rk_device_sm_count": (_I, []),
    "rk_launch_count": (C.c_longlong, []),
    "rk_debug_spin": (_I, [_I, _P]),
    "rk_plan_workspace_bytes": (_Z, [_L]),
    "rk_plan_build": (_I, [_P, _P, _P, _I, _P, _P, _P, _P, _P, _P, _Z, _P, _P]),
    "rk_reduce_workspace_bytes": (_Z, [_P, _I, _P, _I]),
    "rk_embgrad_segment_reduce": (_I, [_P, _P, _P, _P, _I, _P, _I, _P, _Z, _P]),
    "rk_embgrad_direct_reduce": (_I, [_P, _I, _P, _P]),
    "rk_gather_concat_fwd": (_I, [_P, _I, _P, _I, _L, _P, _I, _P, _P]),
    "rk_deepfm_fwd": (_I, [_P, _P, _I, _L, _P, _P, _P, _P, _P]),
    "rk_deepfm_bwd": (_I, [_P, _P, _P, _I, _I, _L, _P, _P]),
    "rk_fwfm_fwd": (_I, [_P, _P, _P, _P, _I, _L, _P, _P, _P, _P]),
    "rk_fwfm_bwd_ctas": (_I, []),
    "rk_fwfm_bwd": (_I, [_P, _P, _P, _P, _I, _I, _L, _P, _P, _P, _P, _P]),
    "rk_crossnet_fwd": (_I, [_P, _I, _P, _I, _P, _P, _I, _L, _P, _P, _P, _P]),
    "rk_crossnet_bwd": (_I, [_P, _P, _P, _I, _I, _L, _P, _P, _P, _P]),
    "rk_cross_layer_fwd": (_I, [_P, _P, _P, _P, _I, _L, _P, _P]),
    "rk_cross_layer_bwd": (_I, [_P, _P, _P, _I, _L, _P, _P, _P, _P]),
    "rk_afm_bwd_ctas": (_I, [_L, _I]),
    "rk_afm_fwd": (_I, [_P, _I, _P, _P, _P, _P, _I, _L, _P, _P, _P]),
    "rk_afm_tile_bytes": (_I, []),
    "rk_afm_tc_fwd": (_I, [_P, _I, _P, _P, _P, _P, _I, _L, _P, _P, _P, _P]),
    "rk_afm_tc_bwd_ctas": (_I, [_L, _I]),
    "rk_afm_tc_bwd": (_I, [_P, _I, _P, _P, _P, _P, _I, _L, _P, _P, _P, _P, _P, _P, _P, _I, _P, _P, _P]),
    "rk_afm_bwd": (_I, [_P, _I, _P, _P, _P, _P, _I, _L, _P, _P, _P, _P, _P, _P, _P, _I, _P, _P]),
    "rk_dice_bn_max_batch": (_I, []),
    "rk_dice_bn_fwd": (_I, [_P, _L, _I, _P, _F, _P, _P, _F, _F, _P, _P, _P, _F, _P, _P, _P, _P, _P, _P]),
    "rk_dice_bn_bwd": (_I, [_P, _P, _L, _I, _P, _P, _P, _P, _P, _P, _P, _P]),
    "rk_bn_act_fwd": (_I, [_P, _L, _I, _P, _P, _F, _F, _P, _P, _P, _F, _P, _P, _P]),
    "rk_bn_act_bwd": (_I, [_P, _P, _L, _I, _P, _P, _F, _P, _P, _P, _P, _P]),
    "rk_linear_wgrad_scratch_floats": (_L, [_L, _I, _I]),
    "rk_linear_wgrad": (_I, [_P, _L, _P, _L, _L, _I, _I, _P, _P, _P, _P]),
    "rk_rowwise_adam": (_I, [_P, _P, _P, _P, _P, _L, _I, _L, _F, _F, _F, _F, _L, _P, _P]),
    "rk_shard_owner": (_I, [_P, _L, _L, _L, _P, _P, _P]),
    "rk_shard_route": (_I, [_P, _P, _P, _L, _L, _L, _I, _P, _P, _P, _P]),
    "rk_plan_compact_fields": (_I, [_P, _P, _P, _P, _I, _P, _P, _P, _P]),
    "rk_rowwise_adam_touched": (_I, [_P, _P, _P, _P, _P, _P, _L, _I, _L, _F, _F, _F, _F, _L, _P, _P]),
    "rk_resunit_pack_floats": (_I, [_I, _I]),
    "rk_resunits_fwd": (_I, [_P, _I, _P, _I, _P, _I, _I, _L, _P, _P, _P]),
    "rk_resunits_bwd": (_I, [_P, _P, _I, _I, _I, _L, _P, _P, _P]),
    "rk_bst_grad_floats": (_I, [_I]),
    "rk_bst_bwd_ctas": (_I, [_L, _I, _I]),
    "rk_bst_block_fwd": (_I, [_P, _I, _P, _P, _L, _P, _P, _L, _I, _P, _P, _I, _I, _P, _P]),
    "rk_bst_block_bwd": (_I, [_P, _I, _P, _P, _L, _P, _P, _L, _I, _P, _P, _I, _I, _P, _P, _P, _I, _P, _P]),
    "rk_din_mlp_floats": (_I, [_I]),
    "rk_din_tile_bytes": (_I, []),
    "rk_din_fwd": (_I, [_P, _P, _P, _P, _P, _P, _P]),
    "rk_din_bwd": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "rk_metrics_append": (_I, [_P, _P, _P, _L, _P, _P, _P, _L, _L, _P, _P, _P]),
    "rk_metrics_workspace_bytes": (_Z, [_L, _L]),
    "rk_metrics_compute": (_I, [_P, _P, _P, _L, _L, _P, _Z, _P, _P]),
    "rk_metrics_merge": (_I, [_P, _P, _P, _P, _L, _L, _P, _P, _P, _P, _P]),
    "rk_adam_step": (_I, [_P, _I, _P, _P]),
    "rk_batch_gather": (_I, [_P, _I, _P, _P, _L, _L, _P, _L, _L, _P, _P]),
    "rk_vocab_slots": (_L, [_L]),
    "rk_vocab_build": (_I, [_P, _P, _P]),
    "rk_encode_strings": (_I, [_P, _P, _P, _L, _P, _P]),
    "rk_encode_split_count": (_I, [_P, _P, _P]),
    "rk_encode_split": (_I, [_P, _P, _P, _P, _P, _P]),
}

_lib = None


class RankB200Error(RuntimeError):
    """A librank_b200 entry point returned non-zero."""


def library_path() -> Path:
    return LIB_PATH


def load() -> C.CDLL:
    """Load librank_b200.so (once).  Raises if it is absent or has the wrong ABI."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RankB200Error(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (needs nvcc, sm_100a).  There is no CPU fallback.")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.rk_version() != ABI_VERSION:
        raise RankB200Error(f"librank_b200 ABI {lib.rk_version()} != expected {ABI_VERSION}")
    _lib = lib
    return lib


class CallTimer:
    """Brackets every kernel-launching ABI call with CUDA events on the launching stream
    (bench.py's live per-call device times).  Use as a context manager; `summary()` after a
    synchronize gives {entry point: (calls, total ms)}."""

    NO_KERNEL = ("rk_resunit_pack_floats", "rk_din_mlp_floats", "rk_din_tile_bytes", "rk_afm_bwd_ctas", "rk_afm_tc_bwd_ctas", "rk_afm_tile_bytes", "rk_fwfm_bwd_ctas", "rk_dice_bn_max_batch", "rk_bst_grad_floats", "rk_bst_bwd_ctas", "rk_version", "rk_last_error", "rk_device_sm_count", "rk_launch_count", "rk_debug_spin",
                 "rk_vocab_slots", "rk_linear_wgrad_scratch_floats", "rk_plan_workspace_bytes", "rk_reduce_workspace_bytes", "rk_metrics_workspace_bytes")

    def __init__(self):
        self.records = []

    def __enter__(self):
        lib = load()
        self._saved = {}
        for name in PROTOTYPES:
            if name in self.NO_KERNEL:
                continue
            fn = getattr(lib, name)
            self._saved[name] = fn
            setattr(lib, name, self._wrap(name, fn))
        return self

    def _wrap(self, name, fn):
        def timed(*args):
            s = torch.cuda.Event(enable_timing=True)
            e = torch.cuda.Event(enable_timing=True)
            s.record()
            rc = fn(*args)
            e.record()
            self.records.append((name, s, e))
            return rc
        return timed

    def __exit__(self, *exc):
        lib = load()
        for name, fn in self._saved.items():
            setattr(lib, name, fn)
        return False

    def summary(self):
        torch.cuda.synchronize()
        out = {}
        for name, s, e in self.records:
            calls, ms = out.get(name, (0, 0.0))
            out[name] = (calls + 1, ms + s.elapsed_time(e))
        return out


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().rk_last_error().decode("utf-8", "replace")
        raise RankB200Error(f"{what} failed (rc={rc}): {msg}")


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def ptr(t: torch.Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


def require_cuda(t: torch.Tensor, name: str, dtype: torch.dtype) -> torch.Tensor:
    """The boundary takes contiguous CUDA tensors of one dtype; anything else is an error."""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a torch.Tensor, got {type(t).__name__}")
    if not t.is_cuda:
        raise RankB200Error(f"{name}: tensor is on {t.device}; the hot path runs on CUDA only "
                            "(no CPU fallback)")
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected {dtype}, got {t.dtype}")
    return t if t.is_contiguous() else t.contiguous()


_err_flags: dict[int, torch.Tensor] = {}


def err_flag(device: torch.device) -> torch.Tensor:
    """Per-device sticky int32 flag the kernels raise when an index is out of range."""
    key = device.index if device.index is not None else torch.cuda.current_device()
    flag = _err_flags.get(key)
    if flag is None:
        flag = torch.zeros(1, dtype=torch.int32, device=device)
        _err_flags[key] = flag
    return flag


def check_index_errors(device=None) -> None:
    """Synchronising check: raise IndexError if any kernel saw an out-of-range index since the
    last check (the reference raises IndexError from nn.Embedding on CPU)."""
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    flag = err_flag(dev)
    if int(flag.item()) != 0:
        flag.zero_()
        raise IndexError("index out of range in self")


CHECK_EVERY_CALL = os.environ.get("RANK_B200_CHECK_INDICES", "0") == "1"
