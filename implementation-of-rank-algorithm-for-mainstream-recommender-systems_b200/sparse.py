"""Host side of the sparse-field machinery shared by all six models.

* `field_array`     packs (table, index column, offset) triples into the C `rk_field_t[]`.
* `OccurrencePlan`  = rk_plan_build: the stable (field,row) order of every index occurrence of
                      the batch, computed once in forward (it depends on the indices only).
* `reduce_to_dense` = rk_embgrad_segment_reduce: per-occurrence gradient rows -> the dense
                      `[V, D]` gradients `optim.Adam` expects (the reference's nn.Embedding is
                      sparse=False, e.g. DeepFM/deepfm.py:90-98), deterministic, no atomics.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import torch

from . import _lib


def field_array(weights, indices, offsets):
    """rk_field_t[F] for tables `weights[f]` read through `indices[f]`, landing at column
    `offsets[f]` of the concatenated row.  Returns (ctypes array, keep-alive list)."""
    F = len(weights)
    if F > _lib.RK_MAX_FIELDS:
        raise ValueError(f"{F} sparse fields exceed RK_MAX_FIELDS={_lib.RK_MAX_FIELDS}")
    arr = (_lib.RkField * max(F, 1))()
    keep = []
    for f in range(F):
        w = _lib.require_cuda(weights[f], f"table[{f}]", torch.float32)
        i = _lib.require_cuda(indices[f], f"index[{f}]", torch.int64)
        if w.dim() != 2:
            raise ValueError(f"table[{f}] must be [rows, dim], got {tuple(w.shape)}")
        keep += [w, i]
        arr[f].weight = w.data_ptr()
        # an empty batch has no index storage (data_ptr() == 0) but the ABI wants non-NULL pointers:
        # any valid device address will do, it is never dereferenced when B == 0
        arr[f].idx = i.data_ptr() if i.numel() else w.data_ptr()
        arr[f].rows = w.shape[0]
        arr[f].dim = w.shape[1]
        arr[f].out_off = int(offsets[f])
    return arr, keep


def _i64_array(values):
    return (C.c_int64 * max(len(values), 1))(*values)


PLAN_ON_SIDE_STREAM = True          # False: plans and reductions run on the caller's stream (timing, debugging)
_side_streams: dict = {}


def _side_stream(device, priority):
    """A per-device side stream of the given priority (None when PLAN_ON_SIDE_STREAM is off).  The occurrence
    plans are built on the high-priority one (-1): the sort is short and something (the segment reduce) always
    ends up waiting for it, while the kernels it shares the GPU with (forward / backward of the hot path, the
    tower) are long.  The one-launch direct reduction runs on the default-priority one (0) when a sorted
    reduction runs next to it: it depends on the backward kernel only, not on the plan."""
    if not PLAN_ON_SIDE_STREAM:
        return None
    key = (device.index if device.index is not None else torch.cuda.current_device(), priority)
    stream = _side_streams.get(key)
    if stream is None:
        stream = _side_streams[key] = torch.cuda.Stream(device=device, priority=priority)
    return stream


@dataclass
class GradSource:
    """Per-occurrence gradient rows of one table: row o lives at base[o*ld : o*ld+dim]."""
    base: torch.Tensor   # any fp32 CUDA tensor; `offset` is in floats from its data_ptr
    offset: int
    ld: int
    dim: int
    rows: int
    field: int           # which plan field's occurrences feed this table
    param: object = None  # the table tensor itself (where a touched-rows gradient is attached)


def check_table_gradients(tables, what):
    """Refuse, before the forward launches anything, a layout whose table gradients the backward's
    reductions (rk_embgrad_direct_reduce, rk_embgrad_segment_reduce) would refuse.  `tables` lists the
    (dim, offset, ld) of every GradSource the backward will hand to OccurrencePlan.reduce_to_dense.
    * at most RK_MAX_TABLES gradient tables in one reduction;
    * a reduction lane carries 4, 2 or 1 floats, the widest that divides the row's dim, its offset and
      the row pitch ld, and a row has at most 32 lanes: dim <= 32 * that width."""
    if len(tables) > _lib.RK_MAX_TABLES:
        raise _lib.RankB200Error(f"{what}: the backward reduces {len(tables)} gradient tables "
                                 f"(at most RK_MAX_TABLES={_lib.RK_MAX_TABLES})")
    for t, (dim, offset, ld) in enumerate(tables):
        vec = 4
        while vec > 1 and (dim % vec or offset % vec or ld % vec):
            vec //= 2
        if dim > 32 * vec:
            raise _lib.RankB200Error(
                f"{what}: table {t} is {dim} floats wide at column {offset} of a {ld}-float row; its gradient "
                f"reduction moves {vec} float(s) per lane, 32 lanes, so at most {32 * vec} columns")


# ---- opt-in sparse gradients of the replicated tables (SURVEY 8(f) item 3) ---------------------
# "dense"  : every table receives a dense [V, D] .grad, as the reference's nn.Embedding(sparse=False)
#            does (DeepFM/deepfm.py:90-98) and dense optim.Adam needs (:226) — the default.
# "touched": no dense slab is written.  Each table gets `table.touched_grad = TouchedRows(...)` — the
#            distinct rows the batch touched and one summed gradient row each, count on the device,
#            no host synchronisation — and `.grad` stays None.  optim.RowwiseAdam consumes it.
_TABLE_GRADIENTS = "dense"


def set_table_gradients(mode: str) -> None:
    global _TABLE_GRADIENTS
    if mode not in ("dense", "touched"):
        raise ValueError(f"table gradients are 'dense' or 'touched', got {mode!r}")
    _TABLE_GRADIENTS = mode


def table_gradients() -> str:
    return _TABLE_GRADIENTS


# Where the dense-gradient slabs come from: None = torch.empty; parallel.GradientAllReducer installs its
# own so that the table gradients are born inside the buffer the all-reduce reads (no pack copy).
_slab_provider = None


def set_slab_provider(fn) -> None:
    """fn(n_floats, device, params) -> 1-D fp32 tensor of n_floats, or None to fall back to torch.empty;
    `params` are the tables whose gradients the slab will hold (a provider serves its own model only)."""
    global _slab_provider
    _slab_provider = fn


def _new_slab(n_floats, device, params):
    if _slab_provider is not None:
        t = _slab_provider(n_floats, device, params)
        if t is not None:
            return t
    return torch.empty(n_floats, dtype=torch.float32, device=device)


@dataclass
class TouchedRows:
    """Sparse gradient of one table, sized without a host sync: `capacity = min(occurrences, table rows)`."""
    rows: torch.Tensor      # [capacity] int64: the first `count` entries are the distinct touched rows, ascending
    values: torch.Tensor    # [capacity, dim]: values[i] = summed gradient of rows[i]; zero from `count` on
    count: torch.Tensor     # [1] int64, on the device
    shape: tuple            # (table rows, dim)

    def to_dense(self) -> torch.Tensor:
        """The dense gradient it stands for (synchronises; tests and debugging)."""
        n = int(self.count.item())
        out = torch.zeros(self.shape, dtype=self.values.dtype, device=self.values.device)
        out[self.rows[:n]] = self.values[:n]
        return out

    def to_sparse_coo(self) -> torch.Tensor:
        """A coalesced torch sparse gradient (synchronises on the count)."""
        n = int(self.count.item())
        return torch.sparse_coo_tensor(self.rows[:n].unsqueeze(0), self.values[:n], self.shape, is_coalesced=True)


class OccurrencePlan:
    """How the embedding gradients of a batch's index columns will be reduced (one entry per field).

    * per-sample columns (n <= RK_DIRECT_MAX_N occurrences, all live): nothing to prepare — their dense
      gradients come from rk_embgrad_direct_reduce in one launch, which also writes the zeros;
    * longer columns (DIN / BST histories, batches beyond 8192) and padded sequence fields: the stable
      (field, row) order of rk_plan_build, computed here (it depends on the indices only) on a side
      stream while the forward runs, consumed by rk_embgrad_segment_reduce.
    `direct=None` reduces directly where the field allows it, unless the table gradients are in the touched-rows
    mode (set_table_gradients), which needs every field sorted; `direct=False` sorts every field (the order is
    then available as sorted_keys / perm)."""

    def __init__(self, indices: list[torch.Tensor], rows: list[int], seq_len=None, live_mode=None, direct=None):
        """`seq_len[f]` (int64 [B]) and `live_mode[f]` (_lib.LIVE_*) mark field f as a padded
        sequence field whose dead positions are left out of the reduction.  Create the plan BEFORE queueing
        the forward kernel: its side stream waits for everything on the current stream at this point."""
        lib = _lib.load()
        self.F = len(indices)
        if not 1 <= self.F <= _lib.RK_MAX_FIELDS:
            raise ValueError(f"plan over {self.F} fields (max {_lib.RK_MAX_FIELDS})")
        self.indices = [_lib.require_cuda(i, f"index[{k}]", torch.int64)
                        for k, i in enumerate(indices)]
        self.n = [int(i.numel()) for i in self.indices]
        self.rows = [int(r) for r in rows]
        dev = self.indices[0].device
        self.device = dev
        modes_all = [_lib.LIVE_ALL] * self.F if live_mode is None else [int(m) for m in live_mode]
        self.touched = _TABLE_GRADIENTS == "touched" and direct is None
        self._compact = None
        use_direct = not self.touched if direct is None else bool(direct)
        self.direct = [use_direct and self.n[f] <= _lib.RK_DIRECT_MAX_N and modes_all[f] == _lib.LIVE_ALL
                       for f in range(self.F)]
        # ---- the fields that need the sorted order
        self.sort_fields = [f for f in range(self.F) if not self.direct[f]]
        self.sort_pos = {f: k for k, f in enumerate(self.sort_fields)}
        self._event = None
        self._ws = None
        self.sorted_keys = self.perm = None
        if not self.sort_fields:
            self.total = 0
            return
        S = len(self.sort_fields)
        s_idx = [self.indices[f] for f in self.sort_fields]
        self.s_n = [self.n[f] for f in self.sort_fields]
        self.s_rows = [self.rows[f] for f in self.sort_fields]
        total = sum(self.s_n)
        self.total = total
        self.sorted_keys = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
        self.perm = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
        ws_bytes = lib.rk_plan_workspace_bytes(total)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        idx_ptrs = (C.c_void_p * S)(*[i.data_ptr() for i in s_idx])
        len_ptrs = seq_T = modes = None
        lens = []
        s_modes = [modes_all[f] for f in self.sort_fields]
        if any(s_modes):
            lens = [None if m == _lib.LIVE_ALL else _lib.require_cuda(seq_len[f], f"seq_len[{f}]", torch.int64)
                    for f, m in zip(self.sort_fields, s_modes)]
            self._lens = lens
            len_ptrs = (C.c_void_p * S)(*[None if l is None else l.data_ptr() for l in lens])
            seq_T = (C.c_int32 * S)(*[0 if l is None else self.s_n[k] // max(int(l.numel()), 1)
                                      for k, l in enumerate(lens)])
            modes = (C.c_int32 * S)(*s_modes)
        # The order depends on the indices only, so it is built on a side stream while the main
        # stream runs the forward kernel and the tower; reduce_to_dense() joins.  Every buffer the
        # side stream touches is recorded on it, so the caching allocator cannot hand a block back to the
        # main stream while rk_plan_build may still be using it, even if the plan is dropped without a join
        # (a grad-enabled forward that never runs backward); inside a CUDA-graph capture the fork/join is
        # captured.
        main = torch.cuda.current_stream(dev)
        side = _side_stream(dev, -1)
        self._ws = ws
        if side is None:
            rc = lib.rk_plan_build(idx_ptrs, _i64_array(self.s_n), _i64_array(self.s_rows), S,
                                   len_ptrs, seq_T, modes, self.sorted_keys.data_ptr(), self.perm.data_ptr(),
                                   ws.data_ptr(), ws_bytes, _lib.err_flag(dev).data_ptr(), main.cuda_stream)
        else:
            side.wait_stream(main)
            with torch.cuda.stream(side):
                rc = lib.rk_plan_build(idx_ptrs, _i64_array(self.s_n), _i64_array(self.s_rows), S,
                                       len_ptrs, seq_T, modes, self.sorted_keys.data_ptr(), self.perm.data_ptr(),
                                       ws.data_ptr(), ws_bytes, _lib.err_flag(dev).data_ptr(), side.cuda_stream)
                self._event = side.record_event()
            if not torch.cuda.is_current_stream_capturing():
                for t in [ws, self.sorted_keys, self.perm, *s_idx, *[l for l in lens if l is not None]]:
                    t.record_stream(side)
        _lib.check(rc, "rk_plan_build")

    def join(self):
        """Make the current stream wait for the plan (no-op when it was built in-stream)."""
        if self._event is not None:
            torch.cuda.current_stream(self.device).wait_event(self._event)
            self._event = None
        self._ws = None

    def reduce_to_dense(self, sources: list[GradSource]) -> list[torch.Tensor]:
        """One dense `[rows, dim]` gradient per source, summed over duplicate indices.  In the opt-in
        "touched" mode (set_table_gradients) nothing dense is written: every source's table receives
        a `touched_grad` and the returned gradients are None."""
        if self.touched:
            return self._reduce_touched(sources)
        lib = _lib.load()
        T = len(sources)
        if not 1 <= T <= _lib.RK_MAX_TABLES:
            raise ValueError(f"{T} gradient tables (max {_lib.RK_MAX_TABLES})")
        dev = self.device
        for s in sources:
            if s.rows != self.rows[s.field]:
                raise ValueError("gradient table height does not match its plan field")
        # one slab for all dense gradients (contiguous for the data-parallel all-reduce), carved per table:
        # the tables reduced directly first (their kernel writes the zeros too), then the sorted ones, whose
        # part of the slab is zero-filled by one memset
        order = [t for t, s in enumerate(sources) if self.direct[s.field]] + \
                [t for t, s in enumerate(sources) if not self.direct[s.field]]
        n_direct = sum(self.direct[s.field] for s in sources)
        starts, acc, sorted_from = {}, 0, 0
        for k, t in enumerate(order):
            if k == n_direct:
                sorted_from = acc
            starts[t] = acc
            acc += (sources[t].rows * sources[t].dim + 3) // 4 * 4          # keep every table 16-byte aligned
        if n_direct == T:
            sorted_from = acc
        slab = _new_slab(acc, dev, [s.param for s in sources])
        if sorted_from < acc:
            slab[sorted_from:].zero_()
        grads = [slab[starts[t]:starts[t] + s.rows * s.dim].view(s.rows, s.dim) for t, s in enumerate(sources)]
        direct_event = None
        if n_direct:
            tabs = (_lib.RkDirectTable * n_direct)()
            for k, t in enumerate(order[:n_direct]):
                s, g = sources[t], grads[t]
                tabs[k].idx = self.indices[s.field].data_ptr() if self.n[s.field] else None
                tabs[k].g = s.base.data_ptr() + 4 * s.offset if self.n[s.field] else None
                tabs[k].ld = s.ld
                tabs[k].dw = g.data_ptr()
                tabs[k].rows = s.rows
                tabs[k].n = self.n[s.field]
                tabs[k].dim = s.dim
            # the two reductions write disjoint parts of the slab: when both exist, the one-launch direct
            # reduction runs on the side stream next to the sorted one (forked and joined here)
            side = _side_stream(dev, 0) if n_direct < T else None
            if side is None:
                rc = lib.rk_embgrad_direct_reduce(tabs, n_direct, _lib.err_flag(dev).data_ptr(), _lib.stream_ptr())
            else:
                main = torch.cuda.current_stream(dev)
                side.wait_stream(main)
                with torch.cuda.stream(side):
                    rc = lib.rk_embgrad_direct_reduce(tabs, n_direct, _lib.err_flag(dev).data_ptr(), side.cuda_stream)
                    direct_event = side.record_event()
                if not torch.cuda.is_current_stream_capturing():
                    for t in [slab, *{id(sources[t].base): sources[t].base for t in order[:n_direct]}.values(),
                              *[self.indices[sources[t].field] for t in order[:n_direct]]]:
                        t.record_stream(side)
            _lib.check(rc, "rk_embgrad_direct_reduce")
        self.join()                 # only the sorted reduction needs the plan; the direct one is already queued
        if n_direct < T:
            S = T - n_direct
            tabs = (_lib.RkGradTable * S)()
            for k, t in enumerate(order[n_direct:]):
                s, g = sources[t], grads[t]
                tabs[k].g = s.base.data_ptr() + 4 * s.offset
                tabs[k].ld = s.ld
                tabs[k].dw = g.data_ptr()
                tabs[k].dim = s.dim
                tabs[k].field = self.sort_pos[s.field]
            n_arr = _i64_array(self.s_n)
            F = len(self.sort_fields)
            ws_bytes = lib.rk_reduce_workspace_bytes(n_arr, F, tabs, S)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            rc = lib.rk_embgrad_segment_reduce(self.sorted_keys.data_ptr(), self.perm.data_ptr(),
                                               n_arr, _i64_array(self.s_rows), F, tabs, S,
                                               ws.data_ptr(), ws_bytes, _lib.stream_ptr())
            _lib.check(rc, "rk_embgrad_segment_reduce")
        if direct_event is not None:
            torch.cuda.current_stream(dev).wait_event(direct_event)
        return grads


def _reduce_touched_impl(plan, sources):
    lib = _lib.load()
    T = len(sources)
    if not 1 <= T <= _lib.RK_MAX_TABLES:
        raise ValueError(f"{T} gradient tables (max {_lib.RK_MAX_TABLES})")
    plan.join()
    dev = plan.device
    F = len(plan.sort_fields)
    n_arr, rows_arr = _i64_array(plan.s_n), _i64_array(plan.s_rows)
    if plan._compact is None:
        # ranks of the distinct rows of every field + the rows themselves, one launch, no host sync
        caps = [max(1, min(n, r)) for n, r in zip(plan.s_n, plan.s_rows)]
        rank_keys = torch.empty(max(plan.total, 1), dtype=torch.int32, device=dev)
        uniq = torch.empty(max(plan.total, 1), dtype=torch.int64, device=dev)
        n_uniq = torch.empty(F, dtype=torch.int64, device=dev)
        rc = lib.rk_plan_compact_fields(plan.sorted_keys.data_ptr(), n_arr, rows_arr, _i64_array(caps), F,
                                        rank_keys.data_ptr(), uniq.data_ptr(), n_uniq.data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "rk_plan_compact_fields")
        starts, acc = [], 0
        for n in plan.s_n:
            starts.append(acc)
            acc += n
        plan._compact = (caps, rank_keys, uniq, n_uniq, starts)
    caps, rank_keys, uniq, n_uniq, starts = plan._compact
    offs, acc = [], 0
    for s in sources:
        if s.param is None:
            raise RuntimeError("touched-rows gradients need GradSource.param (the table tensor)")
        if s.rows != plan.rows[s.field]:
            raise ValueError("gradient table height does not match its plan field")
        offs.append(acc)
        acc += (caps[plan.sort_pos[s.field]] * s.dim + 3) // 4 * 4
    slab = torch.zeros(max(acc, 1), dtype=torch.float32, device=dev)
    tabs = (_lib.RkGradTable * T)()
    for t, s in enumerate(sources):
        tabs[t].g = s.base.data_ptr() + 4 * s.offset
        tabs[t].ld = s.ld
        tabs[t].dw = slab.data_ptr() + 4 * offs[t]
        tabs[t].dim = s.dim
        tabs[t].field = plan.sort_pos[s.field]
    if plan.total:
        ws_bytes = lib.rk_reduce_workspace_bytes(n_arr, F, tabs, T)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        rc = lib.rk_embgrad_segment_reduce(rank_keys.data_ptr(), plan.perm.data_ptr(), n_arr, _i64_array(caps), F,
                                           tabs, T, ws.data_ptr(), ws_bytes, _lib.stream_ptr())
        _lib.check(rc, "rk_embgrad_segment_reduce")
    else:
        n_uniq.zero_()
    for t, s in enumerate(sources):
        k = plan.sort_pos[s.field]
        cap = caps[k]
        touched = TouchedRows(uniq[starts[k]:starts[k] + cap] if plan.s_n[k] else uniq[:0],
                              slab[offs[t]:offs[t] + cap * s.dim].view(cap, s.dim) if plan.s_n[k]
                              else slab[:0].view(0, s.dim),
                              n_uniq[k:k + 1], (s.rows, s.dim))
        if getattr(s.param, "touched_grad", None) is not None:
            raise RuntimeError("a touched-rows gradient is already attached to this table: run the optimizer step "
                               "(or clear table.touched_grad) between backward passes")
        s.param.touched_grad = touched
    return [None] * T


OccurrencePlan._reduce_touched = _reduce_touched_impl


class GatherConcat(torch.autograd.Function):
    """(dense[B,n] or None, idx_0.., table_0..) -> [dense | table_0[idx_0] | ...], differentiable
    w.r.t. dense and the tables (dense gradients through the sorted segment reduction)."""

    @staticmethod
    def forward(ctx, F, dense, *args):
        idx, tables = args[:F], args[F:2 * F]
        offsets, off = [], 0 if dense is None else int(dense.shape[1])
        n_dense = off
        for t in tables:
            offsets.append(off)
            off += int(t.shape[1])
        out = gather_concat(tables, idx, offsets, dense)
        ctx.set_materialize_grads(False)
        ctx.meta = (F, n_dense, offsets, off, [int(t.shape[0]) for t in tables], [int(t.shape[1]) for t in tables])
        if any(ctx.needs_input_grad[2 + F:]):
            ctx.plan = OccurrencePlan(list(idx), ctx.meta[4])
            ctx.tables = list(tables)
        return out

    @staticmethod
    def backward(ctx, g_out):
        F, n_dense, offsets, width, rows, dims = ctx.meta
        if g_out is None:
            return (None,) * (2 + 2 * F)
        g_out = _lib.require_cuda(g_out, "g_out", torch.float32)
        g_dense = g_out[:, :n_dense] if (n_dense and ctx.needs_input_grad[1]) else None
        g_tables = [None] * F
        if any(ctx.needs_input_grad[2 + F:]):
            g_tables = ctx.plan.reduce_to_dense(
                [GradSource(g_out, offsets[f], width, dims[f], rows[f], f, ctx.tables[f]) for f in range(F)])
        return (None, g_dense, *([None] * F), *g_tables)


def gather_concat(weights, indices, offsets, dense=None, width=None) -> torch.Tensor:
    """[dense | W_0[idx_0] | W_1[idx_1] | ...] in one launch (no autograd)."""
    lib = _lib.load()
    arr, keep = field_array(weights, indices, offsets)
    B = int(indices[0].shape[0]) if indices else int(dense.shape[0])
    n_dense = 0
    if dense is not None:
        dense = _lib.require_cuda(dense, "dense", torch.float32)
        n_dense = int(dense.shape[1])
    d = max([n_dense] + [int(o) + int(w.shape[1]) for w, o in zip(weights, offsets)])
    width = d if width is None else width
    dev = keep[0].device if keep else dense.device
    out = torch.empty(B, width, dtype=torch.float32, device=dev)
    if B == 0:                      # nothing to launch; empty tensors have no storage to point at
        return out
    rc = lib.rk_gather_concat_fwd(arr, len(weights), _lib.ptr(dense), n_dense, B, out.data_ptr(),
                                  width, _lib.err_flag(dev).data_ptr(), _lib.stream_ptr())
    _lib.check(rc, "rk_gather_concat_fwd")
    return out
