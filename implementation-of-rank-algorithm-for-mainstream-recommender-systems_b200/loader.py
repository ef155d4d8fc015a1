"""Vectorised pre-encoding of the WeChat frames (SURVEY 8(f) item 4, "loader").

Every model script of the reference reads a parquet file into a DataFrame and encodes ONE ROW per
`__getitem__` — `DataFrame.iloc[idx]`, a dict lookup per categorical value, a 0-d tensor per
feature — and lets `DataLoader` collate them (DeepFM/deepfm.py:26-70, DCN/dcn.py:52-112,
DIN/din.py:86-222, BST/bst.py:94-159).  `EncodedWechat` encodes the whole frame once with
vectorised pandas/numpy operations into int64 / float32 arrays and slices batches out of them.
A batch has exactly the nested-dict structure, dtypes and values that
`DataLoader(WechatDataset(...), batch_size, collate_fn=...)` yields for the same rows — including
the reference's quirks, which are data-visible and therefore kept:

  * a categorical value is looked up by Python equality against the vocabulary LINES (strings):
    an integer-typed column never matches and encodes to 0; unknown / missing values encode to 0,
    the same id as the first vocabulary line; a duplicated line keeps its LAST position;
  * DIN: a history given as a string is split on ',' (so '' is a history of one unknown item,
    length 1), and a batch is padded with 0 to its own longest history (`din_collate_fn`);
  * BST: `feedid` that is not a Python list is a one-item sequence; sequences are cut / zero-padded
    to `max_seq_length`, the length is `min(len, max_seq_length)`.

`batches(..., packed=PackedBatch)` writes each batch straight into a pinned packed buffer
(`staging.py`), so a training step is: slice -> one H2D copy -> graph launch.
"""
from __future__ import annotations

import os

import numpy as np
import pandas as pd
import torch

DENSE_FEATURES = (
    "videoplayseconds", "u_read_comment_7d_sum", "u_like_7d_sum", "u_click_avatar_7d_sum",
    "u_forward_7d_sum", "u_comment_7d_sum", "u_follow_7d_sum", "u_favorite_7d_sum",
    "i_read_comment_7d_sum", "i_like_7d_sum", "i_click_avatar_7d_sum", "i_forward_7d_sum",
    "i_comment_7d_sum", "i_follow_7d_sum", "i_favorite_7d_sum", "c_user_author_read_comment_7d_sum",
)
VOCAB_FILES = {"userid": "userid.txt", "feedid": "feedid.txt", "device": "device.txt", "authorid": "authorid.txt",
               "bgm_song_id": "bgm_song_id.txt", "bgm_singer_id": "bgm_singer_id.txt",
               "manual_tag_list": "manual_tag_id.txt"}
SIX = ("userid", "feedid", "device", "authorid", "bgm_song_id", "bgm_singer_id")
SIDE = ("userid", "device", "authorid", "bgm_song_id", "bgm_singer_id", "manual_tag_list")
DIN_SEQ = "his_read_comment_7d_seq"
KINDS = ("deepfm", "dcn", "deepcrossing", "din", "bst")


def load_vocab_index(vocab_dir, filename):
    """{line: position} as every reference dataset builds it (a missing file is an empty vocabulary)."""
    path = os.path.join(vocab_dir, filename)
    if not os.path.exists(path):
        return {}
    with open(path, "r") as f:
        return {v: i for i, v in enumerate(line.strip() for line in f)}


def encode_column(values: pd.Series, index: dict) -> np.ndarray:
    """`index[v] if v in index else 0` for every v, by Python equality (no string conversion)."""
    if not index:
        return np.zeros(len(values), dtype=np.int64)
    mapped = values.map(index)                      # dict lookup per element; misses -> NaN
    return mapped.fillna(0).to_numpy(dtype=np.int64)


def category_columns(kind):
    """The `category` dict's columns of a batch of this kind."""
    return SIX if kind == "deepfm" else SIDE


def _float_column(frame, col, n):
    if col not in frame.columns:                    # row.get(col, 0.0)
        return np.zeros(n, dtype=np.float32)
    return frame[col].to_numpy(dtype=np.float64).astype(np.float32)   # torch.tensor(float64 value, dtype=float32)


def read_frame(data):
    """The DataFrame itself, or the parquet file at the path `data` read with pandas."""
    return pd.read_parquet(data) if isinstance(data, (str, os.PathLike)) else data


def encode_category(frame, col, index):
    """One categorical column encoded (`row.get(col)` is None for an absent column: every value unknown)."""
    if col not in frame.columns:
        return np.zeros(len(frame), dtype=np.int64)
    return encode_column(frame[col], index)


def din_history(frame, index):
    """Ragged encoding of `his_read_comment_7d_seq`: flat ids + offsets [N+1] (DIN/din.py:146-158)."""
    n = len(frame)
    if DIN_SEQ not in frame.columns:                # row.get(col, []) -> empty history
        return np.zeros(0, dtype=np.int64), np.zeros(n + 1, dtype=np.int64)
    col = frame[DIN_SEQ]
    is_str = col.map(lambda v: isinstance(v, str)).to_numpy(dtype=bool)
    lists = col.astype(object)                      # (an Arrow-backed string column cannot hold lists)
    if is_str.any():
        lists[is_str] = pd.Series([v.split(",") for v in col[is_str]], index=col.index[is_str], dtype=object)
    bad = [type(v).__name__ for v in lists[~is_str] if not hasattr(v, "__iter__")]
    if bad:                                         # the reference iterates the value: a float NaN raises there too
        raise TypeError(f"'{bad[0]}' object is not iterable")
    lengths = lists.map(len).to_numpy(dtype=np.int64)
    offsets = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(lengths, out=offsets[1:])
    flat = lists.explode()
    keep = np.repeat(lengths > 0, np.maximum(lengths, 1))     # explode keeps one NaN row per empty list
    items = flat.to_numpy(dtype=object)[keep]
    ids = pd.Series(items, dtype=object).map(index).fillna(0).to_numpy(dtype=np.int64) if len(items) else \
        np.zeros(0, dtype=np.int64)
    return ids, offsets


def bst_sequence(frame, index, T):
    """`feedid` as a sequence cut / padded to T = max_seq_length, and its lengths (BST/bst.py:139-148)."""
    n = len(frame)
    seq = np.zeros((n, T), dtype=np.int64)
    if "feedid" not in frame.columns:               # row.get("feedid", []) -> empty list
        return seq, np.zeros(n, dtype=np.int64)
    col = frame["feedid"]
    is_list = col.map(lambda v: isinstance(v, list)).to_numpy(dtype=bool)
    length = np.ones(n, dtype=np.int64)
    if (~is_list).any():
        seq[~is_list, 0] = encode_column(col[~is_list], index) if T > 0 else 0
    for row in np.nonzero(is_list)[0]:              # real python lists are rare (parquet yields arrays): plain loop
        items = col.iloc[row][:T]
        length[row] = len(items)
        if items:
            seq[row, :len(items)] = encode_column(pd.Series(items, dtype=object), index)
    length = np.minimum(length, T)
    if T == 0:
        seq = seq[:, :0]
    return seq, length


class EncodedWechat:
    """The whole frame encoded once; `batch(rows)` returns what the reference's DataLoader would."""

    def __init__(self, data, vocab_dir, kind, max_seq_length=50):
        if kind not in KINDS:
            raise ValueError(f"kind must be one of {KINDS}, got {kind!r}")
        frame = read_frame(data)
        self.kind, self.n, self.max_seq_length = kind, len(frame), max_seq_length
        vocab = {c: load_vocab_index(vocab_dir, f) for c, f in VOCAB_FILES.items()}
        self.label = _float_column(frame, "read_comment", self.n)
        self.category = {c: encode_category(frame, c, vocab[c]) for c in category_columns(kind)}
        if kind != "deepfm":
            self.dense = np.stack([_float_column(frame, c, self.n) for c in DENSE_FEATURES], axis=1)
        if kind == "din":
            self.target = {"feedid": encode_category(frame, "feedid", vocab["feedid"])}
            self.seq_flat, self.seq_offsets = din_history(frame, vocab["feedid"])
        if kind == "bst":
            self.seq, self.seq_length = bst_sequence(frame, vocab["feedid"], max_seq_length)

    def __len__(self):
        return self.n

    # ------------------------------------------------------------------ batches
    def batch(self, rows):
        """Nested dict of tensors for the given row numbers, as the reference's DataLoader collates them."""
        rows = np.asarray(rows, dtype=np.int64)
        t = torch.from_numpy
        out = {"category": {c: t(a[rows]) for c, a in self.category.items()}, "label": t(self.label[rows])}
        if self.kind == "deepfm":
            return out
        if self.kind == "din":
            dense = self.dense[rows]
            out["dense"] = {c: t(np.ascontiguousarray(dense[:, i])) for i, c in enumerate(DENSE_FEATURES)}
            out["target"] = {c: t(a[rows]) for c, a in self.target.items()}
            lengths = self.seq_offsets[rows + 1] - self.seq_offsets[rows]
            longest = int(lengths.max()) if len(rows) else 0
            padded = np.zeros((len(rows), longest), dtype=np.int64)
            if longest:
                pos = np.arange(longest)[None, :]
                live = pos < lengths[:, None]
                src = (self.seq_offsets[rows][:, None] + pos)[live]
                padded[live] = self.seq_flat[src]
            out["sequence"] = {DIN_SEQ: t(padded), DIN_SEQ + "_length": t(lengths)}
            return {k: out[k] for k in ("dense", "category", "sequence", "target", "label")}
        out["dense"] = t(self.dense[rows])
        if self.kind == "bst":
            out["seq_feedid"] = t(self.seq[rows])
            out["seq_length"] = t(self.seq_length[rows])
            return {k: out[k] for k in ("dense", "category", "seq_feedid", "seq_length", "label")}
        return {k: out[k] for k in ("dense", "category", "label")}

    def to_device(self, device, seq_width=None):
        """The encoded arrays uploaded once to `device` (plain copies), as a `device_data.DeviceWechat` whose
        batches are gathered there by one kernel launch each.  `seq_width` (DIN only) is the fixed history
        width of its graph-capturable feed: at least the longest history, which is the default."""
        from .device_data import DeviceWechat
        return DeviceWechat(self, device, seq_width)

    def batches(self, batch_size, shuffle=False, generator=None, drop_last=False, packed=None):
        """Iterate over the frame like `DataLoader(dataset, batch_size, shuffle)`.  With `packed`
        (a `PackedBatch` laid out for full batches) every full batch is written into its pinned buffer
        and the PackedBatch is yielded instead of a dict (call `.to_device()` on it)."""
        order = torch.randperm(self.n, generator=generator).numpy() if shuffle else np.arange(self.n)
        for start in range(0, self.n, batch_size):
            rows = order[start:start + batch_size]
            if len(rows) < batch_size and drop_last:
                return
            b = self.batch(rows)
            if packed is not None and len(rows) == batch_size and self.kind != "din":
                yield packed.fill(b)
            else:
                yield b
