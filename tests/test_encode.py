"""Frame encoding on the device without a GPU: the argument checks of the encode entry points (refused with a
negative code before any CUDA call), the table sizing, the per-column path of DeviceWechat.from_frame, and
the reference's TypeError for a null string history, raised before any device is touched."""
import ctypes as C

import numpy as np
import pandas as pd
import pytest
import torch

import rank_b200
from rank_b200 import _lib, device_data
from rank_b200.device_data import _device_columns, classify_column
from rank_b200.loader import DIN_SEQ, KINDS, EncodedWechat
import loader_cases


def test_descriptor_layout_matches_header():
    assert C.sizeof(_lib.RkVocab) == 48 and _lib.RkVocab.n_slots.offset == 40
    assert C.sizeof(_lib.RkStrCol) == 40 and _lib.RkStrCol.n.offset == 32


@pytest.mark.parametrize("n_keys,slots", [(0, 1), (1, 2), (2, 4), (3, 8), (4, 8), (5, 16), (1 << 19, 1 << 20),
                                          ((1 << 19) + 1, 1 << 21), (10 ** 6, 1 << 21)])
def test_vocab_slots_is_the_smallest_power_of_two_at_twice_the_keys(n_keys, slots):
    assert _lib.load().rk_vocab_slots(n_keys) == slots


def test_vocab_slots_refuses_bad_counts():
    lib = _lib.load()
    assert lib.rk_vocab_slots(-1) == -1 and lib.rk_vocab_slots(2 ** 31 - 1) == -1


ADDR = 1 << 24          # placeholder device addresses: distinct, never dereferenced


def _vocab(n_keys=5, n_slots=16):
    return _lib.RkVocab(ADDR, ADDR * 2, ADDR * 3, ADDR * 4, n_keys, n_slots)


def _col(n=10):
    return _lib.RkStrCol(ADDR * 5, ADDR * 6, ADDR * 7, 0, n)


def _call(lib, entry, vocab, col, out, stride, status, offsets):
    v = None if vocab is None else C.byref(vocab)
    c = None if col is None else C.byref(col)
    if entry == "vocab_build":
        return lib.rk_vocab_build(v, status, None)
    if entry == "encode_strings":
        return lib.rk_encode_strings(v, c, out, stride, status, None)
    if entry == "encode_split_count":
        return lib.rk_encode_split_count(c, out, None)
    return lib.rk_encode_split(v, c, offsets, out, status, None)


CASES = {
    "vocab_build": ["null_vocab", "null_bytes", "null_offsets", "null_pos", "null_slots", "null_status", "n_keys",
                    "slots_not_pow2", "slots_below_2x", "slots_zero"],
    "encode_strings": ["null_vocab", "null_slots", "null_col", "null_col_bytes", "null_col_offsets", "null_out",
                       "null_status", "n_keys", "n", "valid_bit0", "slots_not_pow2", "slots_below_2x", "stride_0",
                       "stride_neg"],
    "encode_split_count": ["null_col", "null_col_bytes", "null_col_offsets", "null_out", "n"],
    "encode_split": ["null_vocab", "null_pos", "null_col", "null_col_offsets", "null_out", "null_offsets",
                     "null_status", "n_keys", "n", "slots_below_2x"],
}


@pytest.mark.skipif(torch.cuda.is_available(),
                    reason="placeholder device addresses: only run where no kernel can launch")
@pytest.mark.parametrize("entry,case", [(e, c) for e, cs in CASES.items() for c in cs])
def test_entry_points_refuse_bad_arguments_before_the_device(entry, case):
    lib = _lib.load()
    a = dict(vocab=_vocab(), col=_col(), out=ADDR * 8, stride=1, status=ADDR * 9, offsets=ADDR * 10)
    if case == "null_vocab":
        a["vocab"] = None
    elif case == "null_col":
        a["col"] = None
    elif case.startswith("null_col_"):
        setattr(a["col"], case[len("null_col_"):], None)
    elif case in ("null_bytes", "null_offsets", "null_pos", "null_slots") and not (entry == "encode_split" and
                                                                                  case == "null_offsets"):
        setattr(a["vocab"], case[5:], None)
    elif case in ("null_out", "null_status", "null_offsets"):
        a[case[5:]] = None
    elif case == "n_keys":
        a["vocab"].n_keys = -1
    elif case == "n":
        a["col"].n = -1
    elif case == "valid_bit0":
        a["col"].valid_bit0 = -3
    elif case == "slots_not_pow2":
        a["vocab"].n_slots = 12
    elif case == "slots_below_2x":
        a["vocab"].n_keys, a["vocab"].n_slots = 9, 16
    elif case == "slots_zero":
        a["vocab"].n_keys, a["vocab"].n_slots = 0, 0
    elif case == "stride_0":
        a["stride"] = 0
    elif case == "stride_neg":
        a["stride"] = -1
    rc = _call(lib, entry, **a)
    assert rc < 0, (entry, case, lib.rk_last_error())
    assert lib.rk_last_error().startswith(entry.encode()), (entry, case, lib.rk_last_error())


@pytest.mark.skipif(torch.cuda.is_available(),
                    reason="placeholder device addresses: only run where no kernel can launch")
def test_empty_columns_launch_nothing():
    lib = _lib.load()
    before = lib.rk_launch_count()
    empty = _col(n=0)
    assert lib.rk_encode_strings(C.byref(_vocab()), C.byref(empty), ADDR * 8, 1, ADDR * 9, None) == 0
    assert lib.rk_encode_split_count(C.byref(empty), ADDR * 8, None) == 0
    assert lib.rk_encode_split(C.byref(_vocab()), C.byref(empty), ADDR * 10, ADDR * 8, ADDR * 9, None) == 0
    assert lib.rk_launch_count() == before


def _paths(frame, kind):
    return {c: classify_column(frame, c, kind == "din" and c == DIN_SEQ)[0] for c in _device_columns(kind)}


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("history", ["string", "list"])
def test_each_column_of_the_loader_frames_takes_the_expected_path(kind, history):
    frame = loader_cases.make_frame(history)
    want = {c: "strings" for c in _device_columns(kind)}
    want["device"] = "zeros"                           # an integer column never equals a vocabulary line
    if kind == "din":
        want[DIN_SEQ] = "split" if history == "string" else "lists"
    assert _paths(frame, kind) == want


def test_other_column_types_take_the_host_path_or_zeros():
    frame = loader_cases.make_frame("string")
    frame["userid"] = frame["userid"].astype(object)                       # object, str only: device
    frame["authorid"] = pd.Series(["a1", 3] * (len(frame) // 2) + ["a1"], dtype=object)    # mixed: host
    frame["bgm_song_id"] = np.linspace(0, 1, len(frame))                   # float: zeros
    frame["manual_tag_list"] = pd.Series([None] * len(frame), dtype=object)   # no str at all: host
    frame = frame.drop(columns=["bgm_singer_id"])
    paths = _paths(frame, "dcn")
    assert paths == {"userid": "strings", "device": "zeros", "authorid": "host", "bgm_song_id": "zeros",
                     "bgm_singer_id": "absent", "manual_tag_list": "host"}
    bst = loader_cases.make_frame("string")
    bst["feedid"] = pd.Series([["f1", "f2"] if i % 7 == 0 else "f3" for i in range(len(bst))], dtype=object)
    assert _paths(bst, "bst")["feedid"] == "host"                           # BST's real Python lists
    din = loader_cases.make_frame("list")
    din[DIN_SEQ] = pd.Series([[1, 2]] * len(din), dtype=object)            # list items that are not str
    assert _paths(din, "din")[DIN_SEQ] == "host"
    din[DIN_SEQ] = pd.Series([["f1"], None] * (len(din) // 2) + [["f2"]], dtype=object)   # a null list row
    assert _paths(din, "din")[DIN_SEQ] == "host"


@pytest.mark.parametrize("storage", ["str", "object"])
def test_a_null_string_history_raises_the_reference_error_before_any_device(storage, tmp_path, monkeypatch):
    frame = loader_cases.make_frame("string")
    hist = frame[DIN_SEQ].astype(object)
    hist[4] = None if storage == "object" else np.nan
    frame[DIN_SEQ] = hist if storage == "object" else hist.astype("str")
    vocab = loader_cases.write_vocab(str(tmp_path / "vocab")) + "/"
    with pytest.raises(TypeError) as host:
        EncodedWechat(frame, vocab, "din")

    def no_device(*args, **kw):
        raise AssertionError("a device was touched")

    monkeypatch.setattr(device_data, "_FrameEncoder", no_device)
    monkeypatch.setattr(device_data, "_cuda_device", no_device)
    with pytest.raises(TypeError) as dev:
        rank_b200.DeviceWechat.from_frame(frame, vocab, "din", "cuda:0")
    assert str(dev.value) == str(host.value)
    assert str(dev.value) == ("'NoneType' object is not iterable" if storage == "object"
                              else "'float' object is not iterable")
