"""Field-weighted FM on the B200 hot path.

Drop-in for the reference class `FwFM` (FwFM/fwfm.py:87-139): same constructor
`FwFM(field_dims, embed_dim)`, same parameter names and creation order (`linear.{i}.weight`,
`embedding.{i}.weight` re-initialised with xavier_uniform_, `field_weight`, `bias`), same
`forward(x)` taking the dict of six index tensors and returning `y[B]`.  The 12 lookups, the
F(F-1)/2 weighted pair products, the bias and the sigmoid run in one CUDA kernel (csrc/fwfm.cu);
the backward is one kernel for the per-occurrence row gradients and the field_weight / bias sums
plus the sorted segment reduction shared with every other model (csrc/segment_reduce.cu).
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn as nn

from . import _lib
from .sparse import GradSource, OccurrencePlan, check_table_gradients, field_array

FWFM_COLUMNS = ("userid", "feedid", "device", "authorid", "bgm_song_id", "bgm_singer_id")


class _FwFMInteraction(torch.autograd.Function):
    """(idx_0.., linear_0.., embedding_0.., field_weight, bias) -> y[B]."""

    @staticmethod
    def forward(ctx, F, *args):
        lib = _lib.load()
        idx, first, second = args[:F], args[F:2 * F], args[2 * F:3 * F]
        field_weight, bias = args[3 * F], args[3 * F + 1]
        fields, keep = field_array(second, idx, [f * second[0].shape[1] for f in range(F)])
        first = [_lib.require_cuda(w, f"linear[{f}]", torch.float32) for f, w in enumerate(first)]
        for f, w in enumerate(first):
            if w.shape != (second[f].shape[0], 1):
                raise ValueError(f"linear table {f} must be [{second[f].shape[0]}, 1]")
        P = F * (F - 1) // 2
        field_weight = _lib.require_cuda(field_weight, "field_weight", torch.float32)
        bias = _lib.require_cuda(bias, "bias", torch.float32)
        if field_weight.numel() != P or bias.numel() != 1:
            raise ValueError(f"field_weight must have {P} entries and bias 1")
        B, D = int(idx[0].shape[0]), int(second[0].shape[1])
        if any(ctx.needs_input_grad):
            # the backward reduces the F embedding and the F linear-table gradients together
            check_table_gradients([(D, f * D, F * D) for f in range(F)] + [(1, 0, 1)] * F, "FwFM")
        dev = second[0].device
        emb = torch.empty(B, F * D, dtype=torch.float32, device=dev)
        y = torch.empty(B, dtype=torch.float32, device=dev)
        first_ptrs = (C.c_void_p * F)(*[w.data_ptr() for w in first])
        rc = lib.rk_fwfm_fwd(fields, first_ptrs, field_weight.data_ptr(), bias.data_ptr(), F, B,
                             emb.data_ptr(), y.data_ptr(), _lib.err_flag(dev).data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "rk_fwfm_fwd")
        if _lib.CHECK_EVERY_CALL:
            _lib.check_index_errors(dev)
        ctx.F, ctx.D, ctx.B = F, D, B
        ctx.rows = [int(w.shape[0]) for w in second]
        if any(ctx.needs_input_grad):
            # the occurrence order depends on the indices only: built on the side stream
            ctx.plan = OccurrencePlan([keep[2 * f + 1] for f in range(F)], ctx.rows)
            ctx.tables = (list(args[F:2 * F]), list(second))
            ctx.save_for_backward(emb, y, field_weight)
        return y

    @staticmethod
    def backward(ctx, g_y):
        lib = _lib.load()
        F, D, B = ctx.F, ctx.D, ctx.B
        emb, y, field_weight = ctx.saved_tensors
        dev = emb.device
        P = F * (F - 1) // 2
        g_y = _lib.require_cuda(g_y, "g_y", torch.float32)
        g_rows = torch.empty(B, F * D, dtype=torch.float32, device=dev)
        g_z = torch.empty(B, 1, dtype=torch.float32, device=dev)
        partials = torch.empty(lib.rk_fwfm_bwd_ctas(), P + 1, dtype=torch.float32, device=dev)
        g_pair = torch.empty(P + 1, dtype=torch.float32, device=dev)
        rc = lib.rk_fwfm_bwd(emb.data_ptr(), y.data_ptr(), g_y.data_ptr(), field_weight.data_ptr(), F, D, B,
                             g_rows.data_ptr(), g_z.data_ptr(), partials.data_ptr(), g_pair.data_ptr(),
                             _lib.stream_ptr())
        _lib.check(rc, "rk_fwfm_bwd")
        sources = [GradSource(g_rows, f * D, F * D, D, ctx.rows[f], f, ctx.tables[1][f]) for f in range(F)]
        # every field's first-order weight receives the same per-sample scalar g_z
        sources += [GradSource(g_z, 0, 1, 1, ctx.rows[f], f, ctx.tables[0][f]) for f in range(F)]
        dense = ctx.plan.reduce_to_dense(sources)
        grads_second, grads_first = dense[:F], dense[F:]
        g_fw = g_pair[:P] if ctx.needs_input_grad[1 + 3 * F] else None
        g_bias = g_pair[P:] if ctx.needs_input_grad[2 + 3 * F] else None
        return (None, *([None] * F), *grads_first, *grads_second, g_fw, g_bias)


class FwFM(nn.Module):
    def __init__(self, field_dims, embed_dim):
        super().__init__()
        self.field_dims = field_dims
        self.num_fields = len(field_dims)
        self.embed_dim = embed_dim
        # creation (and RNG) order = the reference's: linear tables, embedding tables, xavier, randn
        self.linear = nn.ModuleList([nn.Embedding(rows, 1) for rows in field_dims])
        self.embedding = nn.ModuleList([nn.Embedding(rows, embed_dim) for rows in field_dims])
        for table in self.embedding:
            nn.init.xavier_uniform_(table.weight)
        self.num_pairs = self.num_fields * (self.num_fields - 1) // 2
        self.field_weight = nn.Parameter(torch.randn(self.num_pairs), requires_grad=True)
        self.bias = nn.Parameter(torch.zeros(1))

    def hot_path(self, x):
        """FwFM has no torch tower: the whole forward runs in librank_b200."""
        return (self.forward(x),)

    def forward(self, x):
        F = self.num_fields
        if F > len(FWFM_COLUMNS):     # the reference indexes a list of six columns (fwfm.py:118-121)
            raise IndexError("list index out of range")
        cols = FWFM_COLUMNS[:F]
        args = ([x[c] for c in cols]
                + [t.weight for t in self.linear]
                + [t.weight for t in self.embedding]
                + [self.field_weight, self.bias])
        return _FwFMInteraction.apply(F, *args)
