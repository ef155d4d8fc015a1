"""DeepCrossing with gather + concat + residual units on the B200 hot path.

Drop-in for the reference's `DeepCrossingModel` and `residual_unit`
(DeepCrossing/deepcrossing.py:25-42,106-163): same constructor, `forward(dense, category) ->
(probability, logit)`, same `state_dict` keys (embeddings + `output_layer` only).  One kernel
(csrc/residual.cu) gathers the six rows, concatenates them with the dense block and runs all
`residual_network_num` residual units with activations resident in shared memory; the backward
is one kernel for d/d(concat row) plus the sorted segment reduction.

Reference quirk kept on purpose: each unit's two `nn.Linear` layers are constructed inside the
call on the CPU generator and never registered (DeepCrossing/deepcrossing.py:37,39).
`draw_residual_units` makes the same constructor calls in the same order.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as Fn

from . import _lib
from .dcn import NUM_DENSE, SIDE_COLUMNS, SIDE_TABLES
from .ephemeral import EphemeralBuffer
from .sparse import GradSource, OccurrencePlan, check_table_gradients, field_array
from .vocab import table_heights


def draw_residual_units(dim, internal_dim, num_units):
    """CPU-generator draws of `num_units` consecutive residual_unit calls, packed per unit as
    rk_resunits_fwd expects: [W1^T][b1][W2^T][b2][W2][W1], zero padded to Hp / dp."""
    hp = (internal_dim + 7) // 8 * 8
    dp = (dim + 3) // 4 * 4
    packs = []
    for _ in range(num_units):
        first = nn.Linear(dim, internal_dim)
        second = nn.Linear(internal_dim, dim)
        w1, b1 = first.weight.detach(), first.bias.detach()      # [H, d], [H]
        w2, b2 = second.weight.detach(), second.bias.detach()    # [d, H], [d]
        packs += [
            Fn.pad(w1.t(), (0, hp - internal_dim)).reshape(-1),                      # W1^T  [d][Hp]
            Fn.pad(b1, (0, hp - internal_dim)),
            Fn.pad(w2.t(), (0, dp - dim, 0, hp - internal_dim)).reshape(-1),         # W2^T  [Hp][dp]
            Fn.pad(b2, (0, dp - dim)),
            Fn.pad(w2, (0, hp - internal_dim)).reshape(-1),                          # W2    [d][Hp]
            Fn.pad(w1, (0, dp - dim, 0, hp - internal_dim)).reshape(-1),             # W1    [Hp][dp]
        ]
    return torch.cat(packs) if packs else torch.zeros(0)


class _ResidualStack(torch.autograd.Function):
    """(dense, packed units, idx_0.., table_0..) -> output of the last unit [B, d]."""

    @staticmethod
    def forward(ctx, F, offsets, internal_dim, n_units, dense, units, *args):
        lib = _lib.load()
        idx, tables = args[:F], args[F:2 * F]
        fields, keep = field_array(tables, idx, offsets)
        dense = _lib.require_cuda(dense, "dense", torch.float32)
        B, n_dense = int(dense.shape[0]), int(dense.shape[1])
        d = max([n_dense] + [o + int(t.shape[1]) for o, t in zip(offsets, tables)])
        if any(ctx.needs_input_grad[6 + F:]):
            check_table_gradients([(int(t.shape[1]), o, d) for o, t in zip(offsets, tables)], "residual units")
        dev = dense.device
        if n_units:
            units = _lib.require_cuda(units, "residual weights", torch.float32)
            if units.numel() != n_units * lib.rk_resunit_pack_floats(d, internal_dim):
                raise ValueError("packed residual-unit weights have the wrong size")
        nets = torch.empty(n_units + 1, B, d, dtype=torch.float32, device=dev)
        rc = lib.rk_resunits_fwd(fields, F, dense.data_ptr(), n_dense, units.data_ptr() if n_units else None,
                                 n_units, internal_dim, B, nets.data_ptr(), _lib.err_flag(dev).data_ptr(),
                                 _lib.stream_ptr())
        _lib.check(rc, "rk_resunits_fwd")
        if _lib.CHECK_EVERY_CALL:
            _lib.check_index_errors(dev)
        ctx.set_materialize_grads(False)
        if any(ctx.needs_input_grad):
            ctx.meta = (F, tuple(offsets), internal_dim, n_units, B, d, n_dense,
                        [int(t.shape[0]) for t in tables], [int(t.shape[1]) for t in tables])
            if any(ctx.needs_input_grad[6 + F:]):
                ctx.plan = OccurrencePlan([keep[2 * f + 1] for f in range(F)], ctx.meta[7])
                ctx.tables = list(tables)
            ctx.save_for_backward(nets, units if n_units else None)
        return nets[n_units]

    @staticmethod
    def backward(ctx, g_out):
        lib = _lib.load()
        F, offsets, internal_dim, n_units, B, d, n_dense, rows, dims = ctx.meta
        if g_out is None:
            return (None,) * (6 + 2 * F)
        nets, units = ctx.saved_tensors
        g_out = _lib.require_cuda(g_out, "g_out", torch.float32)
        g_x0 = torch.empty(B, d, dtype=torch.float32, device=nets.device)
        rc = lib.rk_resunits_bwd(nets.data_ptr(), _lib.ptr(units), n_units, internal_dim, d, B,
                                 g_out.data_ptr(), g_x0.data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "rk_resunits_bwd")
        g_dense = g_x0[:, :n_dense] if ctx.needs_input_grad[4] else None
        g_tables = [None] * F
        if any(ctx.needs_input_grad[6 + F:]):
            g_tables = ctx.plan.reduce_to_dense(
                [GradSource(g_x0, offsets[f], d, dims[f], rows[f], f, ctx.tables[f]) for f in range(F)])
        return (None, None, None, None, g_dense, None, *([None] * F), *g_tables)


def residual_unit(input_tensor, internal_dim, index):
    """One residual unit with freshly drawn, unregistered weights
    (DeepCrossing/deepcrossing.py:25-42): relu(x + W2 relu(W1 x + b1) + b2)."""
    dim = int(input_tensor.size(-1))
    (units,) = EphemeralBuffer().upload([draw_residual_units(dim, internal_dim, 1)], input_tensor.device)
    return _ResidualStack.apply(0, (), internal_dim, 1, input_tensor, units)


class DeepCrossingModel(nn.Module):
    def __init__(self, vocab_dir, residual_internal_dim=128, residual_network_num=1):
        super().__init__()
        self.vocab_sizes = table_heights(vocab_dir, SIDE_COLUMNS)
        self.num_dense_features = NUM_DENSE
        self.embeddings = nn.ModuleDict(
            {col: nn.Embedding(self.vocab_sizes[col], dim) for col, dim in SIDE_TABLES})
        self.input_dim = self.num_dense_features + sum(dim for _, dim in SIDE_TABLES)
        self.residual_internal_dim = residual_internal_dim
        self.residual_network_num = residual_network_num
        self.output_layer = nn.Linear(self.input_dim, 1)
        self._ephemeral = EphemeralBuffer()
        self.ephemeral_frozen = False

    def draw_ephemeral(self, device=None, width=None, fresh=False):
        """Replay one forward's CPU-generator draws (two nn.Linear per unit) onto the GPU (`fresh`: into a
        new tensor instead of the fixed-address buffer of the frozen / CUDA-graph path)."""
        device = self.output_layer.weight.device if device is None else device
        pack = draw_residual_units(self.input_dim if width is None else width, self.residual_internal_dim,
                                   self.residual_network_num)
        self._pack_numel = int(pack.numel())
        if not pack.numel():
            return torch.zeros(0, device=device)
        return self._ephemeral.upload([pack], device, fresh=fresh)[0]

    def hot_path(self, dense, category):
        """The part of forward that runs in librank_b200: the output of the residual stack."""
        cols = [c for c in self.embeddings if c in category]
        offsets, off = [], int(dense.shape[1])
        for c in cols:
            offsets.append(off)
            off += self.embeddings[c].embedding_dim
        if self.ephemeral_frozen and self._ephemeral.ready:
            units = self._ephemeral.views([(self._pack_numel,)])[0]
        else:
            units = self.draw_ephemeral(dense.device, off, fresh=True)
        return (_ResidualStack.apply(len(cols), tuple(offsets), self.residual_internal_dim,
                                     self.residual_network_num, dense, units, *[category[c] for c in cols],
                                     *[self.embeddings[c].weight for c in cols]),)

    def forward(self, dense, category):
        (net,) = self.hot_path(dense, category)
        logit = self.output_layer(net)
        probability = torch.sigmoid(logit)
        return probability, logit
