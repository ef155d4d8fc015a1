"""The encoded WeChat frame kept in device memory, every batch assembled on the GPU.

`EncodedWechat.batches` builds each batch with numpy fancy indexing on one host thread, which is slower
than a B200 training step (the reference's per-row `WechatDataset.__getitem__` + `DataLoader` collation,
DIN/din.py:86-222, BST/bst.py:94-159, DCN/dcn.py:52-112, DeepFM/deepfm.py:26-70, is slower still).  The
encoded frame is small next to HBM, so `EncodedWechat.to_device(device)` uploads it once and a batch is
then one `rk_batch_gather` launch (csrc/batch.cu) that reads a slice of a device permutation:

    data = EncodedWechat(path, vocab_dir, "din").to_device("cuda")
    for batch in data.batches(8192, shuffle=True, generator=gen):          # eager, fresh tensors
        ...
    feed = data.feed(8192)                                                   # graph-capturable
    with torch.cuda.graph(g):
        batch = feed.next()                                                  # gather + cursor advance
        step(batch)
    for epoch in range(epochs):
        feed.start_epoch(shuffle=True, generator=gen)                        # one randperm, one copy
        for _ in range(len(feed)):
            g.replay()
        last = feed.tail()                                                   # the partial batch, or None
    feed.check()

Every batch holds the bytes `parallel.shard_batch(enc.batch(rows), rank, world)` holds, in the same nested
dicts, dtypes and shapes.  The eager form pads DIN's history to the batch's own longest history, as
`din_collate_fn` does; the lengths it needs stay on the host, so the eager loop never waits for the GPU.
The feed pads to the fixed `seq_width`, so its outputs keep their shapes and addresses from step to step.

`DeviceWechat.from_frame(parquet_or_frame, vocab_dir, kind, device)` builds the same arrays without encoding
on the host: string columns go to the GPU as their Arrow buffers and are looked up in device hash tables of
the vocabularies (csrc/encode.cu); DIN's comma-joined histories are split there too.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import pandas as pd
import pyarrow as pa
import torch

from . import _lib
from .loader import (DENSE_FEATURES, DIN_SEQ, KINDS, VOCAB_FILES, _float_column, bst_sequence, category_columns,
                     din_history, encode_category, load_vocab_index, read_frame)
from .staging import _build, _leaves

_LEN = DIN_SEQ + "_length"


def _upload(a, device):
    """One plain copy of a host array.  At least one row is allocated, so an empty array still has an address."""
    t = torch.from_numpy(np.require(a, requirements=("C", "W")))    # (a read-only array is copied first)
    buf = torch.zeros((max(t.shape[0], 1),) + tuple(t.shape[1:]), dtype=t.dtype, device=device)
    buf[:t.shape[0]].copy_(t)
    return buf[:t.shape[0]]


def _check_split(batch_size, rank, world):
    if int(batch_size) < 1:
        raise ValueError(f"batch_size={batch_size} must be >= 1")
    if int(world) < 1 or not 0 <= int(rank) < int(world):
        raise ValueError(f"rank={rank} must lie in [0, world={world})")


def windows(n, batch_size, drop_last=False, rank=0, world=1):
    """(start, size, row0, per) of every global batch of an epoch of n rows: the batch is rows
    order[start : start + size] (`EncodedWechat.batches`), this rank's shard is its rows [row0, row0 + per)
    (`parallel.shard_batch`)."""
    _check_split(batch_size, rank, world)
    for start in range(0, n, batch_size):
        size = min(batch_size, n - start)
        if size < batch_size and drop_last:
            return
        per = size // world
        yield start, size, rank * per, per


def _cuda_device(device):
    device = torch.device(device)
    if device.type != "cuda":
        raise _lib.RankB200Error(f"DeviceWechat: device {device}; batches are gathered on CUDA only "
                                 "(no CPU fallback)")
    return torch.device("cuda", torch.cuda.current_device()) if device.index is None else device


def _leaf_list(kind, dense, category, target, seq, seq_length, label):
    """(path, source [N, ...]) in the key order of EncodedWechat.batch; source None marks DIN's history pair,
    which is gathered from the ragged seq_flat / seq_offsets.  `dense` is DIN's list of columns, the [N, 16]
    matrix of the other kinds but DeepFM (None)."""
    leaves = []
    if kind == "din":
        leaves += [(("dense", c), t) for c, t in zip(DENSE_FEATURES, dense)]
    elif kind != "deepfm":
        leaves.append((("dense",), dense))
    leaves += [(("category", c), t) for c, t in category.items()]
    if kind == "din":
        leaves += [(("sequence", DIN_SEQ), None), (("sequence", _LEN), None)]
        leaves += [(("target", c), t) for c, t in target.items()]
    if kind == "bst":
        leaves += [(("seq_feedid",), seq), (("seq_length",), seq_length)]
    leaves.append((("label",), label))
    return leaves


def _device_columns(kind):
    """Every categorical column a batch of this kind reads."""
    extra = {"din": ("feedid", DIN_SEQ), "bst": ("feedid",)}.get(kind, ())
    return tuple(category_columns(kind)) + extra


def _is_str_list(t):
    return (pa.types.is_list(t) or pa.types.is_large_list(t)) and \
        (pa.types.is_string(t.value_type) or pa.types.is_large_string(t.value_type))


def _as_arrow(values, **kw):
    a = pa.array(values, **kw)
    return a.combine_chunks() if isinstance(a, pa.ChunkedArray) else a


def classify_column(frame, col, history=False):
    """(path, Arrow array or None) of one categorical column, from its type alone (see
    `DeviceWechat.from_frame`); `history` marks DIN's history.  A DIN string history with a null raises the
    reference's TypeError here, before any launch."""
    if col not in frame.columns:
        return "absent", None
    s = frame[col]
    dt = s.dtype
    is_str = isinstance(dt, pd.StringDtype) or (isinstance(dt, pd.ArrowDtype) and (
        pa.types.is_string(dt.pyarrow_dtype) or pa.types.is_large_string(dt.pyarrow_dtype)))
    if dt == object and pd.api.types.infer_dtype(s, skipna=True) == "string":
        is_str = True
    if is_str:
        arr = _as_arrow(s, type=pa.large_string(), from_pandas=True)
        if history and arr.null_count:              # the reference iterates the value (DIN/din.py:146-158)
            raise TypeError(f"'{type(s[s.isna()].iloc[0]).__name__}' object is not iterable")
        return ("split" if history else "strings"), arr
    if dt != object and pd.api.types.is_numeric_dtype(dt) and not history:
        return "zeros", None
    if history and (dt == object or isinstance(dt, pd.ArrowDtype)):
        try:
            arr = _as_arrow(s, from_pandas=True)
        except (pa.ArrowInvalid, pa.ArrowTypeError):
            return "host", None
        if _is_str_list(arr.type) and not arr.null_count:
            return "lists", arr
    return "host", None


class _FrameEncoder:
    """Device hash tables of the vocabularies, built on first use, and the column encodings of one frame.
    Every launch raises bits in one status word, which `check()` reads."""

    def __init__(self, frame, vocab_dir, device):
        self.frame, self.vocab_dir, self.device = frame, vocab_dir, device
        self.n = len(frame)
        self.lib = _lib.load()
        self.stream = torch.cuda.current_stream(device).cuda_stream
        self.status = torch.zeros(1, dtype=torch.int32, device=device)
        self._indices, self._tables = {}, {}

    def _alloc(self, shape, zero=False):
        """int64 device memory of `shape`, at least one row allocated so that even an empty array has an address."""
        buf = (torch.zeros if zero else torch.empty)((max(shape[0], 1),) + tuple(shape[1:]), dtype=torch.int64,
                                                     device=self.device)
        return buf[:shape[0]]

    def _buffer(self, a):
        """A device copy of the host array `a` in at least one element: an empty array still has an address."""
        t = torch.from_numpy(a)
        buf = torch.zeros(max(len(a), 1), dtype=t.dtype, device=self.device)
        buf[:len(a)].copy_(t)
        return buf

    def _index(self, col):
        if col not in self._indices:
            self._indices[col] = load_vocab_index(self.vocab_dir, VOCAB_FILES[col])
        return self._indices[col]

    def _table(self, col):
        """The rk_vocab_t of this column's vocabulary file, with the device buffers it points to."""
        name = VOCAB_FILES[col]
        if name not in self._tables:
            index = self._index(col)
            keys = self._strings(pa.array(list(index), type=pa.large_string()))
            pos = self._buffer(np.fromiter(index.values(), dtype=np.int64, count=len(index)))
            slots = torch.empty(int(self.lib.rk_vocab_slots(len(index))), dtype=torch.int64, device=self.device)
            desc = _lib.RkVocab(keys[0].bytes, keys[0].offsets, pos.data_ptr(), slots.data_ptr(), len(index),
                                slots.numel())
            _lib.check(self.lib.rk_vocab_build(C.byref(desc), self.status.data_ptr(), self.stream), "rk_vocab_build")
            self._tables[name] = (desc, keys, pos, slots)
        return self._tables[name][0]

    def _strings(self, arr):
        """(rk_str_col_t, its device buffers) of a large_string array: its offsets, bytes and validity bitmap,
        one copy each."""
        validity, offsets, data = arr.buffers()
        n = len(arr)
        offs = self._buffer(np.frombuffer(offsets, dtype=np.int64)[arr.offset:arr.offset + n + 1])
        data = self._buffer(np.frombuffer(data, dtype=np.uint8) if data is not None else np.zeros(0, np.uint8))
        valid = self._buffer(np.frombuffer(validity, dtype=np.uint8)) if arr.null_count else None
        col = _lib.RkStrCol(data.data_ptr(), offs.data_ptr(), None if valid is None else valid.data_ptr(),
                            arr.offset, n)
        return col, (offs, data, valid)

    def _lookup(self, col, arr, out, stride=1):
        if len(arr) == 0:                               # (an empty output has no address)
            return
        strings = self._strings(arr)
        _lib.check(self.lib.rk_encode_strings(C.byref(self._table(col)), C.byref(strings[0]), out.data_ptr(),
                                              stride, self.status.data_ptr(), self.stream), "rk_encode_strings")

    def category(self, col, plan):
        """One categorical column [N] (EncodedWechat's category / target columns)."""
        path, arr = plan
        if path == "strings":
            out = self._alloc((self.n,))
            self._lookup(col, arr, out)
            return out
        if path in ("zeros", "absent"):
            return self._alloc((self.n,), zero=True)
        return _upload(encode_category(self.frame, col, self._index(col)), self.device)

    def history(self, plan):
        """DIN's history: (seq_flat, seq_offsets) on the device and the lengths on the host."""
        path, arr = plan
        if path == "split" and self.n:
            strings = self._strings(arr)
            counts = self._alloc((self.n,))
            _lib.check(self.lib.rk_encode_split_count(C.byref(strings[0]), counts.data_ptr(), self.stream),
                       "rk_encode_split_count")
            offsets = self._alloc((self.n + 1,), zero=True)
            torch.cumsum(counts, 0, out=offsets[1:])
            lengths = counts.cpu().numpy()              # the one wait: the lengths stay on the host
            flat = self._alloc((int(lengths.sum()),))
            _lib.check(self.lib.rk_encode_split(C.byref(self._table("feedid")), C.byref(strings[0]),
                                                offsets.data_ptr(), flat.data_ptr(), self.status.data_ptr(),
                                                self.stream), "rk_encode_split")
            return flat, offsets, lengths
        if path == "lists":
            ends = np.asarray(arr.offsets, dtype=np.int64)
            lengths = np.diff(ends)
            offsets = np.zeros(self.n + 1, dtype=np.int64)
            np.cumsum(lengths, out=offsets[1:])
            items = arr.flatten().cast(pa.large_string())
            flat = self._alloc((len(items),))
            self._lookup("feedid", items, flat)
            return flat, _upload(offsets, self.device), lengths
        if path in ("absent", "split"):                 # (a "split" history of an empty frame)
            return self._alloc((0,)), self._alloc((self.n + 1,), zero=True), np.zeros(self.n, dtype=np.int64)
        flat, offsets = din_history(self.frame, self._index("feedid"))
        return _upload(flat, self.device), _upload(offsets, self.device), np.diff(offsets)

    def bst_sequence(self, plan, T):
        """BST's (seq [N, T], seq_length [N]): a value that is not a Python list is a one-item sequence."""
        path, arr = plan
        if path == "host":
            seq, length = bst_sequence(self.frame, self._index("feedid"), T)
            return _upload(seq, self.device), _upload(length, self.device)
        seq = self._alloc((self.n, T), zero=True)
        if path == "strings" and T > 0:
            self._lookup("feedid", arr, seq, stride=T)
        length = self._alloc((self.n,))
        length.fill_(0 if path == "absent" else min(1, T))
        return seq, length

    def check(self):
        """Waits for the device: the status bits of every encode launch."""
        bits = int(self.status.item())
        if bits:
            raise _lib.RankB200Error(f"DeviceWechat.from_frame: encode status bits {bits:#x} "
                                     "(1: a vocabulary table without an empty slot, 2: a history split miscounted)")


class DeviceWechat:
    """An encoded WeChat frame resident on one CUDA device: `EncodedWechat.to_device` uploads a frame encoded
    on the host, `DeviceWechat.from_frame` encodes the frame on the device."""

    def __init__(self, enc, device, seq_width=None):
        self._shape(enc.kind, enc.n, np.diff(enc.seq_offsets) if enc.kind == "din" else None, seq_width)
        device = _cuda_device(device)

        def up(a):
            return _upload(a, device)

        din, bst = enc.kind == "din", enc.kind == "bst"
        dense = None if enc.kind == "deepfm" else \
            [up(enc.dense[:, i]) for i in range(len(DENSE_FEATURES))] if din else up(enc.dense)
        self._place(device, _leaf_list(enc.kind, dense, {c: up(a) for c, a in enc.category.items()},
                                       {c: up(a) for c, a in enc.target.items()} if din else None,
                                       up(enc.seq) if bst else None, up(enc.seq_length) if bst else None,
                                       up(enc.label)),
                    (up(enc.seq_flat), up(enc.seq_offsets)) if din else None, None)

    @classmethod
    def from_frame(cls, data, vocab_dir, kind, device, max_seq_length=50, seq_width=None):
        """The frame (a DataFrame, or a parquet path read with pandas) encoded on `device`: every device array
        equals that of `EncodedWechat(data, vocab_dir, kind, max_seq_length).to_device(device, seq_width)` bit
        for bit, and the encoded frame never exists in host memory.  (BST with max_seq_length 0, which the host
        encoder refuses with an IndexError, gives width-0 sequences and zero lengths.)

        Each categorical column takes one path, chosen from its type alone before any launch, and recorded in
        `encode_paths` ({column: path}):
          "strings"  a string column (Arrow string / large_string, or object holding only str and nulls): one
                     host-to-device copy of its Arrow buffers and one `rk_encode_strings` launch;
          "split"    DIN's history as such a column: `rk_encode_split_count`, a cumsum, `rk_encode_split`;
          "lists"    DIN's history as lists of str without null rows (how parquet hands histories back): the
                     list offsets on the host, the items through `rk_encode_strings`;
          "zeros"    an integer-, float- or bool-typed column, which never equals a vocabulary line: zeros,
                     no launch;
          "absent"   a column the frame lacks: zeros (BST: zero lengths), no launch;
          "host"     anything else (mixed object columns, BST's Python lists, lists of non-str items): the
                     `loader` helper that EncodedWechat uses for that column, then one upload.
        Vocabularies are read by `loader.load_vocab_index` (its key semantics: stripped lines, a duplicated
        line keeps its last position) and built into device hash tables once per file.  A str item inside a
        list is compared as its UTF-8 bytes; a bytes item in such a list is read as those bytes.

        Dense and label columns are converted on the host as EncodedWechat converts them and uploaded.  DIN's
        history lengths stay on the host (the eager batches' widths, the `seq_width` check): a "split"
        history copies its lengths back once, the one point where construction waits for the device before
        the final check of the encode status bits."""
        if kind not in KINDS:
            raise ValueError(f"kind must be one of {KINDS}, got {kind!r}")
        frame = read_frame(data)
        n = len(frame)
        columns = _device_columns(kind)
        plan = {c: classify_column(frame, c, c == DIN_SEQ and kind == "din") for c in columns}
        self = cls.__new__(cls)
        if kind != "din":
            self._shape(kind, n, None, seq_width)
        device = _cuda_device(device)
        enc = _FrameEncoder(frame, vocab_dir, device)

        def up(a):
            return _upload(a, device)

        cat = {c: enc.category(c, plan[c]) for c in category_columns(kind)}
        target = seq = seq_length = history = None
        if kind == "din":
            target = {"feedid": enc.category("feedid", plan["feedid"])}
            seq_flat, seq_offsets, seq_len = enc.history(plan[DIN_SEQ])
            history = (seq_flat, seq_offsets)
            self._shape(kind, n, seq_len, seq_width)
        if kind == "bst":
            seq, seq_length = enc.bst_sequence(plan["feedid"], max_seq_length)
        dense = None
        if kind == "din":
            dense = [up(_float_column(frame, c, n)) for c in DENSE_FEATURES]
        elif kind != "deepfm":
            dense = up(np.stack([_float_column(frame, c, n) for c in DENSE_FEATURES], axis=1))
        label = up(_float_column(frame, "read_comment", n))
        enc.check()
        self._place(device, _leaf_list(kind, dense, cat, target, seq, seq_length, label), history,
                    {c: p for c, (p, _) in plan.items()})
        return self

    def _shape(self, kind, n, seq_len, seq_width):
        """Frame size and DIN's fixed feed width, checked against the host copy of the history lengths."""
        self.kind, self.n = kind, n
        self.seq_width = None
        if kind == "din":
            self._seq_len = seq_len                       # host copy: the eager form's widths, no sync
            longest = int(self._seq_len.max()) if self.n else 0
            if seq_width is None:
                seq_width = longest
            elif int(seq_width) < longest:
                raise ValueError(f"seq_width={seq_width} is smaller than the longest history ({longest})")
            self.seq_width = int(seq_width)
        elif seq_width is not None:
            raise ValueError(f"seq_width applies to DIN histories only, not to kind {kind!r}")

    def _place(self, device, leaves, history, encode_paths):
        """`encode_paths` is None for a frame encoded on the host."""
        self.device = device
        self._leaves = leaves
        if history is not None:
            self.seq_flat, self.seq_offsets = history
        self.encode_paths = encode_paths
        self._status = torch.zeros(1, dtype=torch.int32, device=device)

    def __len__(self):
        return self.n

    # ------------------------------------------------------------------ eager iteration
    def batches(self, batch_size, shuffle=False, generator=None, drop_last=False, rank=0, world=1):
        """Iterate like `EncodedWechat.batches` (same order for the same generator), each batch freshly
        allocated on the device and equal to `parallel.shard_batch(enc.batch(rows), rank, world)`.  The
        order is drawn on the host once per epoch and uploaded once; no call waits for the device."""
        wins = list(windows(self.n, batch_size, drop_last, rank, world))
        order_h = (torch.randperm(self.n, generator=generator) if shuffle else torch.arange(self.n)).numpy()
        order = _upload(order_h, self.device)
        cursor = torch.zeros(1, dtype=torch.int64, device=self.device)
        for start, size, row0, per in wins:
            yield self._eager(order, order_h[start:start + size], cursor, start, row0, per, self._status)

    def _eager(self, order, rows, cursor, start, row0, per, status):
        """This rank's rows [row0, row0 + per) of the global batch order[start : start + len(rows)] (whose host
        copy is `rows`), freshly allocated."""
        width = (int(self._seq_len[rows].max()) if len(rows) else 0) if self.kind == "din" else 0
        outs = self._outputs(per, width)
        if per:
            cursor.fill_(start)
            self._gather(outs, order, self.n, cursor, row0, per, width, status)
        return _build(outs)

    def _outputs(self, b, width):
        out = []
        for path, src in self._leaves:
            if src is not None:
                t = torch.empty((b,) + tuple(src.shape[1:]), dtype=src.dtype, device=self.device)
            elif path[-1] == DIN_SEQ:
                t = torch.empty((b, width), dtype=torch.int64, device=self.device)
            else:       # lengths: with width 0 every history is empty and no kernel writes them
                t = (torch.zeros if width == 0 else torch.empty)(b, dtype=torch.int64, device=self.device)
            out.append((path, t))
        return out

    def _gather(self, outs, order, n_order, cursor, row0, b, width, status):
        cols, seq = [], None
        for (path, src), (_, dst) in zip(self._leaves, outs):
            if src is not None:
                if dst.numel():                               # BST with max_seq_length 0 has empty rows
                    cols.append(_lib.RkBatchCol(src.data_ptr(), dst.data_ptr(), dst[0].numel() * dst.element_size()))
            elif path[-1] == DIN_SEQ:
                hist = dst
            else:
                hist_len = dst
        if self.kind == "din" and width > 0:
            seq = _lib.RkBatchSeq(self.seq_flat.data_ptr(), self.seq_offsets.data_ptr(), hist.data_ptr(),
                                  hist_len.data_ptr(), width, 0)
        arr = (_lib.RkBatchCol * max(len(cols), 1))(*cols)
        rc = _lib.load().rk_batch_gather(arr, len(cols), None if seq is None else C.byref(seq), order.data_ptr(),
                                         n_order, self.n, cursor.data_ptr(), row0, b, status.data_ptr(),
                                         torch.cuda.current_stream(self.device).cuda_stream)
        _lib.check(rc, "rk_batch_gather")

    # ------------------------------------------------------------------ graph-capturable form
    def feed(self, batch_size, rank=0, world=1, packed=None):
        """A `BatchFeed` of full batches (`batch_size` is the global batch; this rank gets
        batch_size // world rows of each), written into fixed device buffers: `packed.dev` when a
        `PackedBatch` laid out for such a batch is given."""
        return BatchFeed(self, batch_size, rank, world, packed)


class BatchFeed:
    """Full batches of an epoch into static device outputs, one launch per `next()`, capturable in a CUDA
    graph.  `start_epoch` draws the order; the feed starts on an unshuffled epoch."""

    def __init__(self, data: DeviceWechat, batch_size, rank, world, packed=None):
        _check_split(batch_size, rank, world)
        self.data, self.batch_size, self.rank, self.world = data, int(batch_size), int(rank), int(world)
        self.per = self.batch_size // self.world
        if self.per == 0:
            raise ValueError(f"batch_size={batch_size} gives no rows to each of {world} ranks")
        self.width = data.seq_width or 0
        dev = data.device
        outs = data._outputs(self.per, self.width)
        if packed is not None:
            have = list(_leaves(packed.device_views))
            want = [(p, t.dtype, tuple(t.shape)) for p, t in outs]
            if [(p, t.dtype, tuple(t.shape)) for p, t in have] != want or packed.dev.device != dev:
                raise ValueError(f"BatchFeed: the PackedBatch on {packed.dev.device} does not hold this feed's "
                                 f"batch on {dev}: want {want}")
            if data.kind == "din" and self.width == 0:
                dict(have)[("sequence", _LEN)].zero_()
            outs = have
            self.views = packed.device_views
        else:
            self.views = _build(outs)
        self._outs = outs
        self.n_full = data.n // self.batch_size
        self.order = torch.zeros(max(data.n, 1), dtype=torch.int64, device=dev)
        self._order_host = torch.empty(data.n, dtype=torch.int64, pin_memory=True)
        self._copied = None           # event behind the last copy out of the pinned order
        self.cursor = torch.zeros(1, dtype=torch.int64, device=dev)
        self._tail_cursor = torch.zeros(1, dtype=torch.int64, device=dev)
        self.status = torch.zeros(1, dtype=torch.int32, device=dev)
        self.start_epoch()

    def __len__(self):
        return self.n_full

    def start_epoch(self, shuffle=False, generator=None):
        """Draw the epoch's order on the host (`torch.randperm(n, generator=generator)`, the order
        `EncodedWechat.batches` uses), copy it into the fixed device buffer and reset the cursor."""
        if self._copied is not None:
            self._copied.synchronize()
        n = self.data.n
        self._order_host.copy_(torch.randperm(n, generator=generator) if shuffle else torch.arange(n))
        stream = torch.cuda.current_stream(self.data.device)
        self.order[:n].copy_(self._order_host, non_blocking=True)
        self._copied = torch.cuda.Event()
        self._copied.record(stream)
        self.cursor.zero_()

    def next(self):
        """Gather the cursor's batch into the static outputs and advance the cursor by the global batch;
        returns the static device views.  Past the last full batch it writes nothing and raises a
        status bit that `check()` reports."""
        self.data._gather(self._outs, self.order, self.n_full * self.batch_size, self.cursor,
                          self.rank * self.per, self.per, self.width, self.status)
        self.cursor.add_(self.batch_size)
        return self.views

    def tail(self):
        """The epoch's rows after the last full batch as a freshly allocated batch (this rank's shard,
        DIN padded to its own longest history), or None when the batches divide the epoch."""
        start = self.n_full * self.batch_size
        if start == self.data.n:
            return None
        ((_, size, row0, per),) = windows(self.data.n - start, self.batch_size, False, self.rank, self.world)
        return self.data._eager(self.order, self._order_host[start:].numpy(), self._tail_cursor, start, row0, per,
                                self.status)

    def check(self):
        """Synchronising check of the status bits raised since the last check."""
        bits = int(self.status.item())
        if bits:
            self.status.zero_()
        if bits & _lib.BATCH_WINDOW:
            raise IndexError(f"BatchFeed.next() was called more than len(feed) = {self.n_full} times in an epoch")
        if bits & _lib.BATCH_BAD_ROW:
            raise IndexError(f"an order entry is outside [0, {self.data.n})")
        if bits & _lib.BATCH_SEQ_OVERFLOW:
            raise ValueError(f"a history is longer than seq_width = {self.width}")
