"""DeepFM with the FM part on the B200 hot path.

Drop-in for the reference class `DeepFM` (DeepFM/deepfm.py:73-151): same constructor, same
`forward(category)` 5-tuple, same `state_dict` keys and parameter creation order.  The 12
embedding lookups, the first-order sum, the sum-square second-order term and the `deep_input`
concat run in one CUDA kernel (csrc/fm.cu); their backward is one kernel for the
per-occurrence gradients plus the sorted segment reduction (csrc/segment_reduce.cu).  The DNN
tower, `final_layer` and the sigmoid stay torch modules, as in the reference.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn as nn

from . import _lib
from .sparse import GradSource, OccurrencePlan, check_table_gradients, field_array
from .tower import run_tower
from .vocab import table_heights

DEEPFM_COLUMNS = ("userid", "feedid", "device", "authorid", "bgm_song_id", "bgm_singer_id")


class _FMInteraction(torch.autograd.Function):
    """(idx_0..idx_F-1, first_0.., second_0..) -> deep_input[B,F*D], first[B,1], second[B,1]."""

    @staticmethod
    def forward(ctx, F, *args):
        lib = _lib.load()
        idx, first, second = args[:F], args[F:2 * F], args[2 * F:3 * F]
        fields, keep = field_array(second, idx, [f * second[0].shape[1] for f in range(F)])
        first = [_lib.require_cuda(w, f"first_order[{f}]", torch.float32) for f, w in enumerate(first)]
        for f, w in enumerate(first):
            if w.shape != (second[f].shape[0], 1):
                raise ValueError(f"first-order table {f} must be [{second[f].shape[0]}, 1]")
        B, D = int(idx[0].shape[0]), int(second[0].shape[1])
        if any(ctx.needs_input_grad):
            # the backward reduces the F second-order and the F first-order gradients together
            check_table_gradients([(D, f * D, F * D) for f in range(F)] + [(1, 0, 1)] * F, "FM part")
        dev = second[0].device
        deep_input = torch.empty(B, F * D, dtype=torch.float32, device=dev)
        fm_first = torch.empty(B, 1, dtype=torch.float32, device=dev)
        fm_second = torch.empty(B, 1, dtype=torch.float32, device=dev)
        first_ptrs = (C.c_void_p * F)(*[w.data_ptr() for w in first])
        rc = lib.rk_deepfm_fwd(fields, first_ptrs, F, B, deep_input.data_ptr(),
                               fm_first.data_ptr(), fm_second.data_ptr(),
                               _lib.err_flag(dev).data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "rk_deepfm_fwd")
        if _lib.CHECK_EVERY_CALL:
            _lib.check_index_errors(dev)
        ctx.F, ctx.D, ctx.B = F, D, B
        ctx.rows = [int(w.shape[0]) for w in second]
        ctx.set_materialize_grads(False)
        if any(ctx.needs_input_grad):
            # the occurrence order depends on the indices only: build it while the tower runs
            ctx.plan = OccurrencePlan([keep[2 * f + 1] for f in range(F)], ctx.rows)
            ctx.tables = (list(args[F:2 * F]), list(second))
            ctx.save_for_backward(deep_input)
        return deep_input, fm_first, fm_second

    @staticmethod
    def backward(ctx, g_deep, g_first, g_second):
        lib = _lib.load()
        F, D, B = ctx.F, ctx.D, ctx.B
        (deep_input,) = ctx.saved_tensors
        dev = deep_input.device
        grads_first = [None] * F
        grads_second = [None] * F
        sources = []
        if g_deep is not None or g_second is not None:
            g_deep = None if g_deep is None else _lib.require_cuda(g_deep, "g_deep", torch.float32)
            g_second = None if g_second is None else _lib.require_cuda(g_second, "g_second", torch.float32)
            g_rows = torch.empty(B, F * D, dtype=torch.float32, device=dev)
            rc = lib.rk_deepfm_bwd(deep_input.data_ptr(), _lib.ptr(g_deep), _lib.ptr(g_second), F, D, B,
                                   g_rows.data_ptr(), _lib.stream_ptr())
            _lib.check(rc, "rk_deepfm_bwd")
            sources += [GradSource(g_rows, f * D, F * D, D, ctx.rows[f], f, ctx.tables[1][f]) for f in range(F)]
        n_second = len(sources)
        if g_first is not None:
            g_first = _lib.require_cuda(g_first, "g_first", torch.float32)
            # every field's first-order weight receives the same per-sample scalar
            sources += [GradSource(g_first, 0, 1, 1, ctx.rows[f], f, ctx.tables[0][f]) for f in range(F)]
        if sources:
            dense = ctx.plan.reduce_to_dense(sources)
            if n_second:
                grads_second = dense[:n_second]
            if g_first is not None:
                grads_first = dense[n_second:]
        return (None, *([None] * F), *grads_first, *grads_second)


class DeepFM(nn.Module):
    def __init__(self, vocab_dir, embedding_dim=8, hidden_units=None, dropout_rate=0.1, batch_norm=True):
        super().__init__()
        hidden_units = [512, 256, 128] if hidden_units is None else hidden_units
        self.vocab_sizes = table_heights(vocab_dir, DEEPFM_COLUMNS)
        self.num_categories = len(self.vocab_sizes)
        # creation order = the reference's (first-order tables, second-order tables, tower)
        self.first_order_embeddings = nn.ModuleDict(
            {col: nn.Embedding(rows, 1) for col, rows in self.vocab_sizes.items()})
        self.second_order_embeddings = nn.ModuleDict(
            {col: nn.Embedding(rows, embedding_dim) for col, rows in self.vocab_sizes.items()})
        self.deep_layers = nn.ModuleList()
        width = self.num_categories * embedding_dim
        for unit in hidden_units:
            self.deep_layers.append(nn.Linear(width, unit))
            if batch_norm:
                self.deep_layers.append(nn.BatchNorm1d(unit))
            self.deep_layers.append(nn.ReLU())
            if dropout_rate > 0:
                self.deep_layers.append(nn.Dropout(dropout_rate))
            width = unit
        self.deep_output_layer = nn.Linear(width, 1)
        self.final_layer = nn.Linear(3, 1)

    def hot_path(self, category):
        """The part of forward that runs in librank_b200: (deep_input, fm_first, fm_second)."""
        cols = [c for c in self.first_order_embeddings if c in category]
        F = len(cols)
        args = ([category[c] for c in cols]
                + [self.first_order_embeddings[c].weight for c in cols]
                + [self.second_order_embeddings[c].weight for c in cols])
        return _FMInteraction.apply(F, *args)

    def forward(self, category):
        deep_input, fm_first_order_logit, fm_second_order_logit = self.hot_path(category)
        deep_output = run_tower(self.deep_layers, deep_input)     # the reference's layer loop
        deep_logit = self.deep_output_layer(deep_output)
        total_logit = self.final_layer(
            torch.cat([fm_first_order_logit, fm_second_order_logit, deep_logit], dim=1))
        probability = torch.sigmoid(total_logit)
        return probability, total_logit, fm_first_order_logit, fm_second_order_logit, deep_logit
