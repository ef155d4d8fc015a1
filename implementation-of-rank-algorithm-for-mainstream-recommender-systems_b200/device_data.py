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
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .loader import DENSE_FEATURES, DIN_SEQ
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


class DeviceWechat:
    """An `EncodedWechat` frame resident on one CUDA device (build it with `EncodedWechat.to_device`)."""

    def __init__(self, enc, device, seq_width=None):
        self.kind, self.n = enc.kind, enc.n
        self.seq_width = None
        if enc.kind == "din":
            self._seq_len = np.diff(enc.seq_offsets)          # host copy: the eager form's widths, no sync
            longest = int(self._seq_len.max()) if self.n else 0
            if seq_width is None:
                seq_width = longest
            elif int(seq_width) < longest:
                raise ValueError(f"seq_width={seq_width} is smaller than the longest history ({longest})")
            self.seq_width = int(seq_width)
        elif seq_width is not None:
            raise ValueError(f"seq_width applies to DIN histories only, not to kind {enc.kind!r}")
        device = torch.device(device)
        if device.type != "cuda":
            raise _lib.RankB200Error(f"DeviceWechat: device {device}; batches are gathered on CUDA only "
                                     "(no CPU fallback)")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = device

        def up(a):
            return _upload(a, device)

        # (path, source [N, ...]) in the key order of EncodedWechat.batch; source None marks DIN's history
        # pair, which is gathered from the ragged seq_flat / seq_offsets
        leaves = []
        if enc.kind == "din":
            leaves += [(("dense", c), up(enc.dense[:, i])) for i, c in enumerate(DENSE_FEATURES)]
        elif enc.kind != "deepfm":
            leaves.append((("dense",), up(enc.dense)))
        leaves += [(("category", c), up(a)) for c, a in enc.category.items()]
        if enc.kind == "din":
            self.seq_flat, self.seq_offsets = up(enc.seq_flat), up(enc.seq_offsets)
            leaves += [(("sequence", DIN_SEQ), None), (("sequence", _LEN), None)]
            leaves += [(("target", c), up(a)) for c, a in enc.target.items()]
        if enc.kind == "bst":
            leaves += [(("seq_feedid",), up(enc.seq)), (("seq_length",), up(enc.seq_length))]
        leaves.append((("label",), up(enc.label)))
        self._leaves = leaves
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
