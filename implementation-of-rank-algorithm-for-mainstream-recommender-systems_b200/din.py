"""DIN with every gather, the local activation unit and the masked pooling on the B200 hot path.

Drop-in for the reference's `DIN`, `din_attention`, `Dice` and `din_collate_fn`
(DIN/din.py:26-36,42-84,176-222,225-323): same constructor, same
`forward(dense, category, sequence, target) -> (probability, logit, l2_reg)`, same `state_dict`
keys.  One kernel (csrc/din.cu) gathers the category / target / history rows, runs the
activation-unit MLP 4D->64->32->1 on the history positions t < len, applies the raw-masked or
scaled-softmax weights, pools, builds the concat row and the per-sample L2 norm; its backward is
one kernel plus the sorted segment reduction.  The Dice/PReLU tower stays torch.

Reference quirk kept on purpose: the activation unit's weights are created inside every call on
the CPU generator (nn.Sequential of three nn.Linear, DIN/din.py:61-67) and never registered.
`draw_attention_mlp` makes the very same constructor calls; only d/d(inputs) is observable.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn as nn

from . import _lib
from .dcn import NUM_DENSE, SIDE_COLUMNS, SIDE_TABLES
from .ephemeral import EphemeralBuffer
from .sparse import GradSource, OccurrencePlan, field_array
from .tower import run_tower
from .vocab import table_heights

SEQ = "his_read_comment_7d_seq"
SEQ_LEN = "his_read_comment_7d_seq_length"

_PRECISION = "fp32"
_TC_MAX_T = 128          # widest history of the tensor-core activation unit (fp32 takes any width)


def set_activation_unit_precision(mode):
    """'fp32': the activation-unit MLP in fp32 on the FMA pipe (parity 1e-5, the default).
    'bf16': the MLP on tcgen05 tensor cores, bf16 operands, fp32 accumulation (parity 2e-2)."""
    global _PRECISION
    if mode not in ("fp32", "bf16"):
        raise ValueError("precision must be 'fp32' or 'bf16'")
    _PRECISION = mode


def get_activation_unit_precision():
    return _PRECISION


class Dice(nn.Module):
    """Data-adaptive activation of the DIN tower (DIN/din.py:26-36) — torch, not on the hot path."""

    def __init__(self, num_features, eps=1e-9):
        super().__init__()
        self.eps = eps
        self.alpha = nn.Parameter(torch.zeros(num_features))
        self.bn = nn.BatchNorm1d(num_features, affine=False)

    def forward(self, x):
        x_p = torch.sigmoid(self.bn(x))
        return self.alpha * (1.0 - x_p) * x + x_p * x


def din_collate_fn(batch):
    """Pads every history to the batch maximum with index 0 (DIN/din.py:176-222)."""
    def stack(group):
        return {col: torch.stack([item[group][col] for item in batch]) for col in batch[0][group]}

    longest = max([len(item["sequence"][c]) for item in batch for c in item["sequence"]
                   if not c.endswith("_length")] + [0])
    sequence = {}
    for col in batch[0]["sequence"]:
        if col.endswith("_length"):
            sequence[col] = torch.stack([item["sequence"][col] for item in batch])
        else:
            rows = torch.zeros(len(batch), longest, dtype=torch.long)
            for r, item in enumerate(batch):
                seq = item["sequence"][col]
                rows[r, :len(seq)] = seq
            sequence[col] = rows
    return {"dense": stack("dense"), "category": stack("category"), "sequence": sequence,
            "target": stack("target"), "label": torch.stack([item["label"] for item in batch])}


def draw_attention_mlp(embedding_dim):
    """The CPU-generator draws of one din_attention call, packed for rk_din_fwd/bwd:
    [W1^T][b1][W2^T][b2][w3][b3,0,0,0][W1][W2]  (layout of rk_din_mlp_floats)."""
    att_net = nn.Sequential(
        nn.Linear(4 * embedding_dim, 64), nn.ReLU(), nn.Linear(64, 32), nn.ReLU(), nn.Linear(32, 1))
    w1, b1 = att_net[0].weight.detach(), att_net[0].bias.detach()
    w2, b2 = att_net[2].weight.detach(), att_net[2].bias.detach()
    w3, b3 = att_net[4].weight.detach(), att_net[4].bias.detach()
    return torch.cat([w1.t().reshape(-1), b1, w2.t().reshape(-1), b2, w3.reshape(-1), b3,
                      torch.zeros(3), w1.reshape(-1), w2.reshape(-1)])


def _din_args(cat_tables, cat_idx, cat_offsets, dense_cols, target_w, target_idx, tgt_off, his_w,
              his_idx, his_len, att_off, width, l2_from, use_softmax, mlp, precision=None):
    """rk_din_args_t + the objects that must outlive the call."""
    fields, keep = field_array(cat_tables, cat_idx, cat_offsets)
    a = _lib.RkDinArgs()
    a.cat = C.addressof(fields)
    a.n_cat = len(cat_tables)
    cols = [_lib.require_cuda(c, "dense column", torch.float32) for c in dense_cols]
    strides = {c.stride(0) if c.dim() else 1 for c in cols}
    if len(strides) > 1:
        cols = [c.contiguous() for c in cols]
    a.n_dense = len(cols)
    col_ptrs = (C.c_void_p * max(len(cols), 1))(*[c.data_ptr() for c in cols])
    a.dense_cols = C.addressof(col_ptrs)
    a.dense_stride = cols[0].stride(0) if cols and cols[0].numel() > 1 else 1
    tw = _lib.require_cuda(target_w, "target table", torch.float32)
    ti = _lib.require_cuda(target_idx, "target index", torch.int64)
    hw = _lib.require_cuda(his_w, "history table", torch.float32)
    hi = _lib.require_cuda(his_idx, "history index", torch.int64)
    hl = _lib.require_cuda(his_len, "history length", torch.int64)
    if hi.dim() != 2 or hl.shape != (hi.shape[0],) or ti.shape != (hi.shape[0],):
        raise ValueError("history index must be [B, T], lengths and target index [B]")
    a.target = _lib.RkField(tw.data_ptr(), ti.data_ptr(), tw.shape[0], tw.shape[1], tgt_off)
    a.history = _lib.RkField(hw.data_ptr(), hi.data_ptr(), hw.shape[0], hw.shape[1], 0)
    a.hist_len = hl.data_ptr()
    a.T = int(hi.shape[1])
    a.att_off, a.width, a.l2_from, a.use_softmax = att_off, width, l2_from, int(bool(use_softmax))
    precision = _PRECISION if precision is None else precision
    if precision not in ("fp32", "bf16"):
        raise ValueError("activation-unit precision must be 'fp32' or 'bf16'")
    if precision == "bf16" and int(his_w.shape[1]) != 16:
        # the tensor-core unit is built for D = 16 (the model's dim): no silent fp32 fallback
        raise _lib.RankB200Error(f"the tcgen05 activation unit needs embedding dim 16, got {int(his_w.shape[1])}; "
                                 "use precision 'fp32' for other dims")
    if precision == "bf16" and a.T > _TC_MAX_T:
        # the tensor-core unit packs whole histories into 128-row tiles: no silent fp32 fallback either
        raise _lib.RankB200Error(f"the tcgen05 activation unit takes histories of at most {_TC_MAX_T} positions, "
                                 f"got {a.T}; use precision 'fp32' for longer ones")
    a.precision = 1 if precision == "bf16" else 0
    mlp = _lib.require_cuda(mlp, "attention mlp", torch.float32)
    if mlp.numel() != _lib.load().rk_din_mlp_floats(int(hw.shape[1])):
        raise ValueError("packed attention weights have the wrong size")
    a.mlp = mlp.data_ptr()
    a.B = int(hi.shape[0])
    tiles = None
    if precision == "bf16":
        # scratch for the operand tiles the forward's prologue makes and both directions fetch by bulk (TMA) copy
        tiles = torch.empty(_lib.load().rk_din_tile_bytes(), dtype=torch.uint8, device=hw.device)
        a.mlp_tiles = tiles.data_ptr()
    return a, (fields, keep, cols, col_ptrs, tw, ti, hw, hi, hl, mlp, tiles)


class _DinHotPath(torch.autograd.Function):
    """(mlp, dense cols.., cat idx.., target idx, hist idx, hist len, cat tables.., target table,
    history table) -> concat_all[B,width], norm[B]."""

    @staticmethod
    def forward(ctx, cfg, mlp, *args):
        lib = _lib.load()
        n_dense, F, offsets, use_softmax, precision = cfg
        dense_cols = args[:n_dense]
        cat_idx = args[n_dense:n_dense + F]
        tgt_idx, his_idx, his_len = args[n_dense + F:n_dense + F + 3]
        cat_tabs = args[n_dense + F + 3:n_dense + 2 * F + 3]
        tgt_w, his_w = args[n_dense + 2 * F + 3:]
        D = int(his_w.shape[1])
        tgt_off = (offsets[-1] + int(cat_tabs[-1].shape[1])) if F else n_dense
        att_off, width = tgt_off + D, tgt_off + 2 * D
        a, keep = _din_args(cat_tabs, cat_idx, offsets, dense_cols, tgt_w, tgt_idx, tgt_off, his_w, his_idx,
                            his_len, att_off, width, n_dense, use_softmax, mlp, precision)
        B, T = int(a.B), int(a.T)
        dev = his_w.device
        need_grad = any(ctx.needs_input_grad)
        concat_all = torch.empty(B, width, dtype=torch.float32, device=dev)
        norm = torch.empty(B, dtype=torch.float32, device=dev)
        att_w = torch.empty(B, T, dtype=torch.float32, device=dev)
        masks = torch.empty(B, T, 3, dtype=torch.int32, device=dev) if need_grad else None
        plan = rows = None
        if need_grad:
            # forked BEFORE the forward kernel is queued: the plan's side stream waits for what is on the main
            # stream at this point (the indices), so the sort of the history ids overlaps the forward kernel
            idx_cols = [keep[1][2 * f + 1] for f in range(F)] + [keep[5], keep[7]]
            rows = [int(t.shape[0]) for t in cat_tabs] + [int(tgt_w.shape[0]), int(his_w.shape[0])]
            mode = _lib.LIVE_PREFIX_OR_EMPTY if use_softmax else _lib.LIVE_PREFIX
            if T == 0:
                mode = _lib.LIVE_ALL      # no positions at all: nothing to mask
            plan = OccurrencePlan(idx_cols, rows, seq_len=[None] * (F + 1) + [keep[8]],
                                  live_mode=[_lib.LIVE_ALL] * (F + 1) + [mode])
        rc = lib.rk_din_fwd(C.byref(a), concat_all.data_ptr(), norm.data_ptr(), att_w.data_ptr(),
                            _lib.ptr(masks), _lib.err_flag(dev).data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "rk_din_fwd")
        if _lib.CHECK_EVERY_CALL:
            _lib.check_index_errors(dev)
        ctx.set_materialize_grads(False)
        if need_grad:
            ctx.cfg = cfg
            ctx.args, ctx.keep = a, keep
            ctx.shape = (B, T, D, width, tgt_off)
            ctx.plan = plan
            ctx.dims = [int(t.shape[1]) for t in cat_tabs]
            ctx.rows = rows
            ctx.tables = [*cat_tabs, tgt_w, his_w]
            ctx.save_for_backward(concat_all, norm, att_w, masks, mlp)
        return concat_all, norm

    @staticmethod
    def backward(ctx, g_concat, g_norm):
        lib = _lib.load()
        n_dense, F, offsets = ctx.cfg[:3]
        concat_all, norm, att_w, masks, mlp = ctx.saved_tensors      # mlp: version-checked by autograd
        B, T, D, width, tgt_off = ctx.shape
        n_in = 2 + n_dense + 2 * F + 5
        if g_concat is None and g_norm is None:
            return (None,) * n_in
        dev = concat_all.device
        g_concat = None if g_concat is None else _lib.require_cuda(g_concat, "g_concat", torch.float32)
        g_norm = None if g_norm is None else _lib.require_cuda(g_norm, "g_norm", torch.float32)
        g_row = torch.empty(B, width, dtype=torch.float32, device=dev)
        # never a NULL pointer, even with T == 0: the reduction takes the history gradient's address
        g_hist = torch.empty(max(B * T * D, 1), dtype=torch.float32, device=dev)[:B * T * D].view(B, T, D)
        rc = lib.rk_din_bwd(C.byref(ctx.args), concat_all.data_ptr(), norm.data_ptr(), att_w.data_ptr(),
                            masks.data_ptr(), _lib.ptr(g_concat), _lib.ptr(g_norm), g_row.data_ptr(),
                            g_hist.data_ptr(), _lib.err_flag(dev).data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "rk_din_bwd")
        src = [GradSource(g_row, offsets[f], width, ctx.dims[f], ctx.rows[f], f, ctx.tables[f]) for f in range(F)]
        src.append(GradSource(g_row, tgt_off, width, D, ctx.rows[F], F, ctx.tables[F]))
        src.append(GradSource(g_hist, 0, D, D, ctx.rows[F + 1], F + 1, ctx.tables[F + 1]))
        dense = ctx.plan.reduce_to_dense(src)
        g_dense = [g_row[:, c] if ctx.needs_input_grad[2 + c] else None for c in range(n_dense)]
        return (None, None, *g_dense, *([None] * (F + 3)), *dense)


class _DinAttention(torch.autograd.Function):
    """din_attention on already-gathered tensors: the same kernels with identity index columns."""

    @staticmethod
    def forward(ctx, query, keys, keys_length, mlp, use_softmax):
        lib = _lib.load()
        B, T, D = keys.shape
        dev = keys.device
        q = _lib.require_cuda(query, "query", torch.float32)
        k = _lib.require_cuda(keys, "keys", torch.float32).view(B * T, D)
        length = _lib.require_cuda(keys_length.to(torch.int64), "keys_length", torch.int64)
        ti = torch.arange(B, dtype=torch.int64, device=dev)
        hi = torch.arange(B * T, dtype=torch.int64, device=dev).view(B, T)
        a, keep = _din_args([], [], [], [], q, ti, 0, k, hi, length, D, 2 * D, 2 * D, use_softmax, mlp)
        out = torch.empty(B, 2 * D, dtype=torch.float32, device=dev)
        att_w = torch.empty(B, T, dtype=torch.float32, device=dev)
        masks = torch.empty(B, T, 3, dtype=torch.int32, device=dev)
        rc = lib.rk_din_fwd(C.byref(a), out.data_ptr(), None, att_w.data_ptr(), masks.data_ptr(),
                            _lib.err_flag(dev).data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "rk_din_fwd")
        ctx.args, ctx.keep, ctx.shape = a, keep, (B, T, D)
        ctx.save_for_backward(out, att_w, masks, mlp)
        return out[:, D:].contiguous()

    @staticmethod
    def backward(ctx, g_out):
        lib = _lib.load()
        out, att_w, masks, mlp = ctx.saved_tensors
        B, T, D = ctx.shape
        dev = out.device
        g_concat = torch.zeros(B, 2 * D, dtype=torch.float32, device=dev)
        g_concat[:, D:] = g_out
        g_row = torch.empty(B, 2 * D, dtype=torch.float32, device=dev)
        g_hist = torch.zeros(B, T, D, dtype=torch.float32, device=dev)   # dead positions stay 0
        rc = lib.rk_din_bwd(C.byref(ctx.args), out.data_ptr(), None, att_w.data_ptr(), masks.data_ptr(),
                            g_concat.data_ptr(), None, g_row.data_ptr(), g_hist.data_ptr(),
                            _lib.err_flag(dev).data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "rk_din_bwd")
        return g_row[:, :D].contiguous(), g_hist, None, None, None


def din_attention(query, keys, keys_length, is_softmax=False):
    """Local activation unit with freshly drawn, unregistered weights (DIN/din.py:42-84):
    query [B,D], keys [B,T,D], keys_length [B] -> [B,D]."""
    mlp = draw_attention_mlp(keys.shape[-1])
    (mlp,) = EphemeralBuffer().upload([mlp], keys.device)
    return _DinAttention.apply(query, keys, keys_length, mlp, is_softmax)


class DIN(nn.Module):
    def __init__(self, vocab_dir, hidden_units=None, activation='dice', dropout_rate=0.1, batch_norm=True,
                 use_softmax=False, l2_lambda=0.2, mini_batch_aware_regularization=True):
        super().__init__()
        hidden_units = [512, 256, 128] if hidden_units is None else hidden_units
        self.activation = activation
        self.dropout_rate = dropout_rate
        self.batch_norm = batch_norm
        self.use_softmax = use_softmax
        self.l2_lambda = l2_lambda
        self.mini_batch_aware_regularization = mini_batch_aware_regularization
        self.vocab_sizes = table_heights(vocab_dir, SIDE_COLUMNS)
        self.num_dense_features = NUM_DENSE
        tables = {col: nn.Embedding(self.vocab_sizes[col], dim) for col, dim in SIDE_TABLES}
        tables["feedid"] = nn.Embedding(self.vocab_sizes["feedid"], 16)
        tables[SEQ] = nn.Embedding(self.vocab_sizes["feedid"], 16)
        self.embeddings = nn.ModuleDict(tables)
        width = (self.num_dense_features + sum(dim for _, dim in SIDE_TABLES)
                 + self.embeddings["feedid"].embedding_dim + self.embeddings[SEQ].embedding_dim)
        self.fcn = nn.ModuleList()
        for unit in hidden_units:
            self.fcn.append(nn.Linear(width, unit))
            self.fcn.append(Dice(unit) if activation == 'dice' else nn.PReLU())
            if batch_norm:
                self.fcn.append(nn.BatchNorm1d(unit))
            if dropout_rate > 0:
                self.fcn.append(nn.Dropout(dropout_rate))
            width = unit
        self.output_layer = nn.Linear(width, 1)
        self._ephemeral = EphemeralBuffer()
        self.ephemeral_frozen = False
        self.activation_unit_precision = None     # None: follow set_activation_unit_precision()

    def draw_ephemeral(self, device=None, fresh=False):
        """Replay one forward's CPU-generator draws (att_net, DIN/din.py:61-67) onto the GPU (`fresh`:
        into a new tensor instead of the fixed-address buffer of the frozen / CUDA-graph path)."""
        device = self.output_layer.weight.device if device is None else device
        mlp = draw_attention_mlp(self.embeddings[SEQ].embedding_dim)
        return self._ephemeral.upload([mlp], device, fresh=fresh)[0]

    def hot_path(self, dense, category, sequence, target):
        """The part of forward that runs in librank_b200: (concat_all[B,82], per-sample L2 norm[B])."""
        dense_cols = [dense[c] for c in dense]
        cols = [c for c in self.embeddings if c in category]
        offsets, off = [], len(dense_cols)
        for c in cols:
            offsets.append(off)
            off += self.embeddings[c].embedding_dim
        dev = self.output_layer.weight.device
        if self.ephemeral_frozen and self._ephemeral.ready:
            mlp = self._ephemeral.views([(_lib.load().rk_din_mlp_floats(self.embeddings[SEQ].embedding_dim),)])[0]
        else:
            mlp = self.draw_ephemeral(dev, fresh=True)
        cfg = (len(dense_cols), len(cols), tuple(offsets), bool(self.use_softmax), self.activation_unit_precision)
        return _DinHotPath.apply(
            cfg, mlp, *dense_cols, *[category[c] for c in cols], target['feedid'], sequence[SEQ],
            sequence[SEQ_LEN], *[self.embeddings[c].weight for c in cols],
            self.embeddings['feedid'].weight, self.embeddings[SEQ].weight)

    def forward(self, dense, category, sequence, target):
        concat_all, norm = self.hot_path(dense, category, sequence, target)
        net = run_tower(self.fcn, concat_all)      # the reference's `for layer in self.fcn` loop
        logit = self.output_layer(net)
        probability = torch.sigmoid(logit)
        l2_reg = 0.0
        if self.mini_batch_aware_regularization and self.l2_lambda > 0:
            l2_reg = self.l2_lambda * norm.mean()
        return probability, logit, l2_reg
