"""DCN (Deep & Cross) with gather + concat + CrossNet on the B200 hot path.

Drop-in for `DCNModel` and `cross_layer` of the reference (DCN/dcn.py:25-50,114-180): same
constructor, `forward(dense, category) -> (probability, logit)`, `state_dict` keys.  The six
lookups, the concat with the dense block and all `num_cross_layer` cross layers are one kernel
(csrc/concat_cross.cu); the backward is one kernel for d/dx0 plus the sorted segment
reduction.  The DNN, `output_layer` and sigmoid stay torch.

Reference quirk kept on purpose: every cross layer draws a fresh `w_l ~ xavier_normal`,
`b_l = 0` on the CPU generator inside each call (DCN/dcn.py:37-41) and never registers them,
so they are not trained and not in the state_dict.  `draw_cross_weights` replays exactly those
draws; only d(out)/d(x0) is observable, which is all the backward kernel computes.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _lib
from .ephemeral import EphemeralBuffer
from .sparse import GradSource, OccurrencePlan, check_table_gradients, field_array
from .tower import run_tower
from .vocab import table_heights

SIDE_COLUMNS = ("userid", "feedid", "device", "authorid", "bgm_song_id", "bgm_singer_id",
                "manual_tag_list")
# (column, embedding dim) in ModuleDict order — shared by DCN, DeepCrossing, DIN and BST
SIDE_TABLES = (("userid", 16), ("device", 2), ("authorid", 4), ("bgm_song_id", 4),
               ("bgm_singer_id", 4), ("manual_tag_list", 4))
NUM_DENSE = 16


def draw_cross_weights(dimension, num_layers):
    """The CPU-generator draws of `num_layers` consecutive cross_layer calls, in order."""
    ws, bs = [], []
    for _ in range(num_layers):
        wl = nn.Parameter(torch.zeros(dimension, 1), requires_grad=True)
        bl = nn.Parameter(torch.zeros(dimension, 1), requires_grad=True)
        nn.init.xavier_normal_(wl)
        nn.init.zeros_(bl)
        ws.append(wl.detach().reshape(1, dimension))
        bs.append(bl.detach().reshape(1, dimension))
    if not ws:
        return torch.zeros(0, dimension), torch.zeros(0, dimension)
    return torch.cat(ws, 0), torch.cat(bs, 0)


class _CrossNet(torch.autograd.Function):
    """(dense, w[L,d], b[L,d], idx_0.., table_0..) -> concat_all[B,d], cross_vec[B,d]."""

    @staticmethod
    def forward(ctx, F, offsets, dense, w, b, *args):
        lib = _lib.load()
        idx, tables = args[:F], args[F:2 * F]
        fields, keep = field_array(tables, idx, offsets)
        dense = _lib.require_cuda(dense, "dense", torch.float32)
        w = _lib.require_cuda(w, "cross w", torch.float32)
        b = _lib.require_cuda(b, "cross b", torch.float32)
        B, n_dense = int(dense.shape[0]), int(dense.shape[1])
        d = max([n_dense] + [o + int(t.shape[1]) for o, t in zip(offsets, tables)])
        L = int(w.shape[0])
        if w.shape != (L, d) or b.shape != (L, d):
            raise ValueError(f"cross weights must be [{L}, {d}]")
        for i in idx:
            if i.shape != (B,):
                raise ValueError("every category column must be [batch]")
        if any(ctx.needs_input_grad[5 + F:]):
            check_table_gradients([(int(t.shape[1]), o, d) for o, t in zip(offsets, tables)], "CrossNet")
        dev = dense.device
        concat_all = torch.empty(B, d, dtype=torch.float32, device=dev)
        cross_vec = torch.empty(B, d, dtype=torch.float32, device=dev)
        rc = lib.rk_crossnet_fwd(fields, F, dense.data_ptr(), n_dense, w.data_ptr(), b.data_ptr(),
                                 L, B, concat_all.data_ptr(), cross_vec.data_ptr(),
                                 _lib.err_flag(dev).data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "rk_crossnet_fwd")
        if _lib.CHECK_EVERY_CALL:
            _lib.check_index_errors(dev)
        ctx.meta = (F, tuple(offsets), L, d, B, n_dense, [int(t.shape[0]) for t in tables],
                    [int(t.shape[1]) for t in tables])
        ctx.set_materialize_grads(False)
        if any(ctx.needs_input_grad):
            if any(ctx.needs_input_grad[5 + F:]):
                ctx.plan = OccurrencePlan([keep[2 * f + 1] for f in range(F)],
                                          [int(t.shape[0]) for t in tables])
                ctx.tables = list(tables)
            ctx.save_for_backward(concat_all, w, b)
        return concat_all, cross_vec

    @staticmethod
    def backward(ctx, g_concat, g_cross):
        lib = _lib.load()
        F, offsets, L, d, B, n_dense, rows, dims = ctx.meta
        concat_all, w, b = ctx.saved_tensors
        none = (None,) * (5 + 2 * F)
        if g_concat is None and g_cross is None:
            return none
        g_concat = None if g_concat is None else _lib.require_cuda(g_concat, "g_concat", torch.float32)
        g_cross = None if g_cross is None else _lib.require_cuda(g_cross, "g_cross", torch.float32)
        g_x0 = torch.empty(B, d, dtype=torch.float32, device=concat_all.device)
        rc = lib.rk_crossnet_bwd(concat_all.data_ptr(), w.data_ptr(), b.data_ptr(), L, d, B,
                                 _lib.ptr(g_concat), _lib.ptr(g_cross), g_x0.data_ptr(),
                                 _lib.stream_ptr())
        _lib.check(rc, "rk_crossnet_bwd")
        g_dense = g_x0[:, :n_dense] if ctx.needs_input_grad[2] else None
        g_tables = [None] * F
        if any(ctx.needs_input_grad[5 + F:]):
            src = [GradSource(g_x0, offsets[f], d, dims[f], rows[f], f, ctx.tables[f]) for f in range(F)]
            g_tables = ctx.plan.reduce_to_dense(src)
        return (None, None, g_dense, None, None, *([None] * F), *g_tables)


class _CrossLayer(torch.autograd.Function):
    """One cross layer with distinct anchor x0 and input xl: out = x0 * (xl . w) + b + xl."""

    @staticmethod
    def forward(ctx, x0, xl, w, b):
        lib = _lib.load()
        x0 = _lib.require_cuda(x0, "x0", torch.float32)
        xl = _lib.require_cuda(xl, "xl", torch.float32)
        if x0.dim() != 2 or x0.shape != xl.shape:
            raise ValueError("cross_layer: x0 and xl must both be [batch, d]")
        B, d = int(xl.shape[0]), int(xl.shape[1])
        out = torch.empty_like(xl)
        rc = lib.rk_cross_layer_fwd(x0.data_ptr(), xl.data_ptr(), w.data_ptr(), b.data_ptr(), d, B,
                                    out.data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "rk_cross_layer_fwd")
        ctx.save_for_backward(x0, xl, w)
        return out

    @staticmethod
    def backward(ctx, g_out):
        lib = _lib.load()
        x0, xl, w = ctx.saved_tensors
        B, d = int(xl.shape[0]), int(xl.shape[1])
        g_out = _lib.require_cuda(g_out, "g_out", torch.float32)
        g_x0, g_xl = torch.empty_like(x0), torch.empty_like(xl)
        rc = lib.rk_cross_layer_bwd(x0.data_ptr(), xl.data_ptr(), w.data_ptr(), d, B,
                                    g_out.data_ptr(), g_x0.data_ptr(), g_xl.data_ptr(),
                                    _lib.stream_ptr())
        _lib.check(rc, "rk_cross_layer_bwd")
        return g_x0, g_xl, None, None


def cross_layer(x0, xl, index):
    """One cross layer with freshly drawn, unregistered weights (DCN/dcn.py:25-50).  Stand-alone
    form of the op; `DCNModel.forward` runs the fused gather + L-layer chain instead."""
    w, b = draw_cross_weights(x0.shape[-1], 1)
    w, b = EphemeralBuffer().upload([w, b], x0.device)
    return _CrossLayer.apply(x0, xl, w, b)


class DCNModel(nn.Module):
    def __init__(self, vocab_dir, hidden_units=[512, 256, 128], num_cross_layer=1):
        super().__init__()
        self.vocab_sizes = table_heights(vocab_dir, SIDE_COLUMNS)
        self.num_dense_features = NUM_DENSE
        self.embeddings = nn.ModuleDict(
            {col: nn.Embedding(self.vocab_sizes[col], dim) for col, dim in SIDE_TABLES})
        self.input_dim = self.num_dense_features + sum(dim for _, dim in SIDE_TABLES)
        self.num_cross_layer = num_cross_layer
        layers, width = [], self.input_dim
        for hidden in hidden_units:
            layers += [nn.Linear(width, hidden), nn.ReLU()]
            width = hidden
        self.dnn = nn.Sequential(*layers)
        self.output_layer = nn.Linear(self.input_dim + hidden_units[-1], 1)
        self._ephemeral = EphemeralBuffer()
        self.ephemeral_frozen = False   # True: reuse the weights of the last draw_ephemeral()

    def draw_ephemeral(self, device=None, width=None, fresh=False):
        """Replay one forward's CPU-generator draws (DCN/dcn.py:37-41, once per cross layer) and
        ship them to the GPU.  Returns device views (w[L,d], b[L,d]) — of the fixed-address buffer a
        frozen (CUDA-graph) forward reads, or of a new tensor when `fresh` (every eager forward)."""
        device = self.output_layer.weight.device if device is None else device
        w, b = draw_cross_weights(self.input_dim if width is None else width, self.num_cross_layer)
        return self._ephemeral.upload([w, b], device, fresh=fresh)

    def hot_path(self, dense, category):
        """The part of forward that runs in librank_b200: (concat_all, cross_vec)."""
        cols = [c for c in self.embeddings if c in category]
        offsets, off = [], int(dense.shape[1])
        for c in cols:
            offsets.append(off)
            off += self.embeddings[c].embedding_dim
        if self.ephemeral_frozen and self._ephemeral.ready:
            w, b = self._ephemeral.views([(self.num_cross_layer, off)] * 2)
        else:
            w, b = self.draw_ephemeral(dense.device, off, fresh=True)
        return _CrossNet.apply(
            len(cols), offsets, dense, w, b, *[category[c] for c in cols],
            *[self.embeddings[c].weight for c in cols])

    def forward(self, dense, category):
        concat_all, cross_vec = self.hot_path(dense, category)
        dnn_vec = run_tower(list(self.dnn), concat_all)      # = self.dnn(concat_all), Linear weight gradients in librank
        logit = self.output_layer(torch.cat([cross_vec, dnn_vec], dim=1))
        probability = torch.sigmoid(logit)
        return probability, logit
