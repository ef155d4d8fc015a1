"""rank_b200.DeviceWechat and rk_batch_gather without a GPU: the batch and shard arithmetic against
EncodedWechat.batches + parallel.shard_batch, the seq_width and device checks, and the argument checks of
the entry point (refused with a negative code before any CUDA call)."""
import ctypes as C

import numpy as np
import pytest
import torch

import rank_b200
from rank_b200 import _lib
from rank_b200.device_data import windows
from rank_b200.loader import EncodedWechat
from rank_b200.parallel import shard_batch
import loader_cases
from test_loader import _same


def _enc(kind, tmp_path):
    vocab_dir = loader_cases.write_vocab(str(tmp_path / "vocab")) + "/"
    return EncodedWechat(loader_cases.make_frame("string"), vocab_dir, kind, max_seq_length=5)


@pytest.mark.parametrize("kind", ["dcn", "bst"])
@pytest.mark.parametrize("batch_size", [1, 7, 56, 57, 62])
@pytest.mark.parametrize("drop_last", [False, True])
@pytest.mark.parametrize("rank,world", [(0, 1), (0, 2), (1, 2), (2, 3)])
def test_windows_give_the_rows_of_batches_and_shard_batch(kind, batch_size, drop_last, rank, world, tmp_path):
    enc = _enc(kind, tmp_path)
    n = len(enc)
    order = torch.randperm(n, generator=torch.Generator().manual_seed(5)).numpy()
    want = list(enc.batches(batch_size, shuffle=True, generator=torch.Generator().manual_seed(5),
                            drop_last=drop_last))
    wins = list(windows(n, batch_size, drop_last, rank, world))
    assert len(wins) == len(want)
    for (start, size, row0, per), w in zip(wins, want):
        assert len(w["label"]) == size
        _same(enc.batch(order[start:start + size]), w)
        _same(enc.batch(order[start + row0:start + row0 + per]), shard_batch(w, rank, world))


@pytest.mark.parametrize("batch_size,world", [(0, 1), (4, 0)])
def test_windows_refuse_bad_splits(batch_size, world):
    with pytest.raises(ValueError):
        list(windows(10, batch_size, world=world))
    with pytest.raises(ValueError):
        list(windows(10, 4, rank=2, world=2))


def test_seq_width_is_checked_on_the_host(tmp_path):
    enc = _enc("din", tmp_path)
    longest = int(np.diff(enc.seq_offsets).max())
    with pytest.raises(ValueError, match="seq_width"):
        enc.to_device("cuda", seq_width=longest - 1)
    with pytest.raises(ValueError, match="DIN"):
        _enc("dcn", tmp_path).to_device("cuda", seq_width=8)


def test_cpu_device_is_refused(tmp_path):
    with pytest.raises(rank_b200.RankB200Error):
        _enc("deepfm", tmp_path).to_device("cpu")


def test_descriptor_layout_matches_header():
    assert C.sizeof(_lib.RkBatchCol) == 24                               # rk_batch_col_t
    assert C.sizeof(_lib.RkBatchSeq) == 40 and _lib.RkBatchSeq.width.offset == 32
    assert _lib.RK_BATCH_MAX_COLS == 32
    assert rank_b200.DeviceWechat is rank_b200.device_data.DeviceWechat


ADDR = 1 << 24          # placeholder device addresses: 16-byte aligned, distinct, never dereferenced


def _cols(k):
    return (_lib.RkBatchCol * max(k, 1))(*[_lib.RkBatchCol(ADDR * (2 * c + 1), ADDR * (2 * c + 2), 8)
                                           for c in range(k)])


def _seq(width=8, values=ADDR * 100):
    return _lib.RkBatchSeq(values, ADDR * 101, ADDR * 102, ADDR * 103, width, 0)


@pytest.mark.skipif(torch.cuda.is_available(),
                    reason="placeholder device addresses: only run where no kernel can launch")
@pytest.mark.parametrize("case", ["n_cols", "null_col", "row_bytes", "null_order", "null_cursor", "null_status",
                                  "B", "row0", "width", "null_values"])
def test_entry_point_refuses_bad_arguments_before_the_device(case):
    lib = _lib.load()
    args = dict(cols=_cols(3), n_cols=3, seq=_seq(), order=ADDR * 200, n_order=100, n_rows=100,
                cursor=ADDR * 201, row0=0, B=4, status=ADDR * 202)
    if case == "n_cols":
        args.update(cols=_cols(_lib.RK_BATCH_MAX_COLS + 1), n_cols=_lib.RK_BATCH_MAX_COLS + 1)
    elif case == "null_col":
        args["cols"][1].src = None
    elif case == "row_bytes":
        args["cols"][2].row_bytes = 0
    elif case in ("null_order", "null_cursor", "null_status"):
        args[case[5:]] = None
    elif case == "B":
        args["B"] = 0
    elif case == "row0":
        args["row0"] = -1
    elif case == "width":
        args["seq"] = _seq(width=0)
    elif case == "null_values":
        args["seq"] = _seq(values=None)
    rc = lib.rk_batch_gather(args["cols"], args["n_cols"], C.byref(args["seq"]), args["order"], args["n_order"],
                             args["n_rows"], args["cursor"], args["row0"], args["B"], args["status"], None)
    assert rc < 0, (case, lib.rk_last_error())
    assert lib.rk_last_error().startswith(b"batch_gather"), case
