"""BST with the sequence gather, the transformer block(s) and the pooling on the B200 hot path.

Drop-in for the reference's `BSTModel`, `BSTTransformer`, `leakyrelu` and `load_vocabulary`
(BST/bst.py:27-39,42-91,162-247): same constructors, `forward(dense, category, seq_feedid,
seq_length) -> (probabilities, logits)`, same `state_dict` keys.  Each transformer block is one
kernel (csrc/bst.cu): the first one gathers the feedid rows itself, the last one also pools over
all T positions; the side-information gathers + concat are one more launch.  The backward of a
block is one persistent kernel (in-kernel recompute, no saved [B,heads,T,T] tensor) plus a
fixed-order reduction of the per-CTA partial gradients of the block's registered weights.  The
DNN stays torch.

Dropout inside the block (BST/bst.py:57,62,86,90): in training mode with dropout > 0 the kernels
apply inverted dropout at the reference's three sites (w_o output, inside the FFN, FFN output)
with keep-bits from an in-kernel counter-based generator (Philox4x32-10 keyed by a per-block seed
drawn from torch's CPU generator, an offset advanced on the device once per forward, the row and
the site); the backward regenerates the same bits, nothing is stored.  The reference's own draws
(torch generators) cannot be replayed, so parity with the reference is defined at dropout 0 /
eval mode, and the dropout path is checked against the oracle run with the very same masks.

`set_block_precision("bf16")` runs the block's projections, FFN and weight gradients on tcgen05
tensor cores (bf16 operands, fp32 accumulation in TMEM; the north star's 2e-2 bar); the default
"fp32" is the SIMT block held to 1e-5.
"""
from __future__ import annotations

import ctypes as C
import os

import torch
import torch.nn as nn

from . import _lib
from .dcn import NUM_DENSE, SIDE_COLUMNS, SIDE_TABLES
from .sharded import RowShardedEmbedding
from .sparse import GatherConcat, GradSource, OccurrencePlan
from .tower import run_tower

D_MODEL = 16
_PARAM_ORDER = ("position_embedding.weight", "w_q.weight", "w_q.bias", "w_k.weight", "w_k.bias", "w_v.weight",
                "w_v.bias", "w_o.weight", "w_o.bias", "norm1.weight", "norm1.bias", "ffn.0.weight", "ffn.0.bias",
                "ffn.3.weight", "ffn.3.bias", "norm2.weight", "norm2.bias")
_FIELD_ORDER = ("pos", "wq", "bq", "wk", "bk", "wv", "bv", "wo", "bo", "ln1_g", "ln1_b", "w1", "b1", "w2", "b2",
                "ln2_g", "ln2_b")
_PRECISION = "fp32"
_TC_MAX_T = 128          # longest sequence of the tensor-core block (fp32 takes any length)


def set_block_precision(precision: str) -> None:
    """"fp32" (default): fp32 SIMT block, 1e-5 parity.  "bf16": the projections / FFN / weight
    gradients on tcgen05 tensor cores, tested at the north star's 2e-2 bar."""
    global _PRECISION
    if precision not in ("fp32", "bf16"):
        raise ValueError(f"precision must be 'fp32' or 'bf16', got {precision!r}")
    _PRECISION = precision


def block_precision() -> str:
    return _PRECISION


def load_vocabulary(vocab_file):
    """Lines of a vocabulary file, [] if it does not exist (BST/bst.py:27-33)."""
    if not os.path.exists(vocab_file):
        return []
    with open(vocab_file, 'r') as f:
        return [line.strip() for line in f]


def leakyrelu(x, leak=0.01):
    """max(x, leak*x) written as in the reference (BST/bst.py:36-39); unused by the model."""
    return 0.5 * (1 + leak) * x + 0.5 * (1 - leak) * torch.abs(x)


def _block_struct(params, dropout_p, rng, precision):
    blk = _lib.RkBstBlock()
    keep = []
    for name, t in zip(_FIELD_ORDER, params):
        t = _lib.require_cuda(t, name, torch.float32)
        keep.append(t)
        setattr(blk, name, t.data_ptr())
    blk.dropout_p = float(dropout_p)
    blk.precision = _lib.BST_BF16_TENSOR if precision == "bf16" else _lib.BST_FP32
    if rng is not None:
        rng = _lib.require_cuda(rng, "dropout rng state", torch.int64)
        keep.append(rng)
        blk.rng = rng.data_ptr()
    return blk, keep


def _check_length(T, precision):
    """The tensor-core block tiles whole sequences into 128 rows: refused above that, before any launch
    (no silent fp32 fallback)."""
    if precision == "bf16" and T > _TC_MAX_T:
        raise _lib.RankB200Error(f"the tcgen05 BST block takes sequences of at most {_TC_MAX_T} positions, "
                                 f"got {T}; use block precision 'fp32' for longer ones")


class _BstBlock(torch.autograd.Function):
    """One transformer block.  source = table (with idx) for the first block, else x[B,T,16].
    Returns y[B,T,16], or the pooled [B,16] when `pool` is 'sum' / 'mean'."""

    @staticmethod
    def forward(ctx, cfg, seq_len, idx, source, *params):
        lib = _lib.load()
        nhead, pool, dropout_p, rng, precision = cfg
        seq_len = _lib.require_cuda(seq_len, "seq_length", torch.int64)
        source = _lib.require_cuda(source, "sequence input", torch.float32)
        from_table = idx is not None
        if from_table:
            idx = _lib.require_cuda(idx, "seq_feedid", torch.int64)
            B, T = int(idx.shape[0]), int(idx.shape[1])
        else:
            B, T = int(source.shape[0]), int(source.shape[1])
        if source.shape[-1] != D_MODEL or D_MODEL % nhead:
            raise RuntimeError(f"shape '[{B}, {T}, {nhead}, -1]' is invalid for d_model {source.shape[-1]}")
        if params[0].shape[0] < T:
            raise IndexError("index out of range in self")      # position_embedding(arange(T))
        _check_length(T, precision)
        blk, keep = _block_struct(params, dropout_p, rng, precision)
        dev = source.device
        y = pooled = None
        if pool is None:
            y = torch.empty(B, T, D_MODEL, dtype=torch.float32, device=dev)
        else:
            pooled = torch.empty(B, D_MODEL, dtype=torch.float32, device=dev)
        plan = None
        if from_table and ctx.needs_input_grad[3]:
            # forked before the forward kernel is queued, so the sort of the sequence ids overlaps it
            plan = OccurrencePlan([idx], [int(source.shape[0])])
        rc = lib.rk_bst_block_fwd(C.byref(blk), nhead, source.data_ptr() if from_table else None,
                                  _lib.ptr(idx), int(source.shape[0]) if from_table else 0,
                                  None if from_table else source.data_ptr(), seq_len.data_ptr(), B, T,
                                  _lib.ptr(y), _lib.ptr(pooled), D_MODEL, int(pool == "mean"),
                                  _lib.err_flag(dev).data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "rk_bst_block_fwd")
        if _lib.CHECK_EVERY_CALL:
            _lib.check_index_errors(dev)
        ctx.set_materialize_grads(False)
        if any(ctx.needs_input_grad):
            ctx.cfg, ctx.shape, ctx.from_table = cfg, (B, T), from_table
            ctx.blk, ctx.keep = blk, keep
            ctx.max_len = int(params[0].shape[0])
            if plan is not None:
                ctx.plan = plan
                ctx.table = source
            ctx.save_for_backward(seq_len, idx if from_table else None, source)
        return y if pool is None else pooled

    @staticmethod
    def backward(ctx, g):
        lib = _lib.load()
        n_in = 4 + len(_PARAM_ORDER)
        if g is None:
            return (None,) * n_in
        nhead, pool = ctx.cfg[:2]
        B, T = ctx.shape
        seq_len, idx, source = ctx.saved_tensors
        dev = source.device
        g = _lib.require_cuda(g, "g_out", torch.float32)
        g_x = torch.empty(B, T, D_MODEL, dtype=torch.float32, device=dev)
        n_par = lib.rk_bst_grad_floats(T)
        g_par = torch.empty(n_par, dtype=torch.float32, device=dev)
        n_ctas = lib.rk_bst_bwd_ctas(B, T, ctx.blk.precision)
        partials = torch.empty(n_ctas * n_par, dtype=torch.float32, device=dev)
        rc = lib.rk_bst_block_bwd(C.byref(ctx.blk), nhead, source.data_ptr() if ctx.from_table else None,
                                  _lib.ptr(idx), int(source.shape[0]) if ctx.from_table else 0,
                                  None if ctx.from_table else source.data_ptr(), seq_len.data_ptr(), B, T,
                                  g.data_ptr() if pool is None else None, None if pool is None else g.data_ptr(),
                                  D_MODEL, int(pool == "mean"), g_x.data_ptr(), g_par.data_ptr(),
                                  partials.data_ptr(), n_ctas, _lib.err_flag(dev).data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "rk_bst_block_bwd")
        # split the flat gradient: position table first (rows >= T of the table get no gradient)
        g_pos = torch.zeros(ctx.max_len, D_MODEL, dtype=torch.float32, device=dev)
        g_pos[:T] = g_par[:T * D_MODEL].view(T, D_MODEL)
        grads, pos = [g_pos], T * D_MODEL
        for name in _PARAM_ORDER[1:]:
            if name.endswith("bias") or name.startswith("norm"):
                grads.append(g_par[pos:pos + D_MODEL])
                pos += D_MODEL
            else:
                grads.append(g_par[pos:pos + D_MODEL * D_MODEL].view(D_MODEL, D_MODEL))
                pos += D_MODEL * D_MODEL
        g_source = None
        if ctx.needs_input_grad[3]:
            if ctx.from_table:
                (g_source,) = ctx.plan.reduce_to_dense(
                    [GradSource(g_x, 0, D_MODEL, D_MODEL, int(source.shape[0]), 0, ctx.table)])
            else:
                g_source = g_x
        return (None, None, None, g_source, *grads)


class BSTTransformer(nn.Module):
    """Parameters and names of the reference block (BST/bst.py:42-64); forward runs the kernel."""

    def __init__(self, d_model, nhead, max_len, dropout=0.1):
        super().__init__()
        self.d_model = d_model
        self.nhead = nhead
        self.position_embedding = nn.Embedding(max_len, d_model)
        self.w_q = nn.Linear(d_model, d_model)
        self.w_k = nn.Linear(d_model, d_model)
        self.w_v = nn.Linear(d_model, d_model)
        self.w_o = nn.Linear(d_model, d_model)
        self.norm1 = nn.LayerNorm(d_model)
        self.norm2 = nn.LayerNorm(d_model)
        self.dropout = nn.Dropout(dropout)
        self.ffn = nn.Sequential(nn.Linear(d_model, d_model), nn.LeakyReLU(negative_slope=0.01),
                                 nn.Dropout(dropout), nn.Linear(d_model, d_model))

    def _params(self):
        named = dict(self.named_parameters())
        return [named[n] for n in _PARAM_ORDER]

    def _dropout_state(self, device):
        """(p, rng) of this forward: rng = a snapshot [seed, offset] of the block's device-side
        generator state, whose offset is then advanced in-stream (capturable in a CUDA graph: every
        replay draws new masks).  The seed comes from torch's CPU generator the first time, so
        torch.manual_seed makes the masks reproducible."""
        p = float(self.dropout.p)
        if not self.training or p <= 0.0:
            return 0.0, None
        if p >= 1.0:
            raise NotImplementedError("dropout = 1 zeroes the block; use the reference module for that")
        state = getattr(self, "_rng_state", None)
        if state is None or state.device != device:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())
            state = torch.tensor([seed, 0], dtype=torch.int64, device=device)
            self._rng_state = state
        snap = state.clone()
        state[1:2] += 1
        self._last_rng = snap          # what this forward's masks were drawn from (tests read it)
        return p, snap

    def resolve_precision(self, precision=None):
        """The block precision of a call: `precision`, else this block's, else set_block_precision's."""
        return precision or getattr(self, "block_precision", None) or _PRECISION

    def run(self, source, seq_len, idx=None, pool=None, precision=None):
        """Fused path used by BSTModel: rows from `source[idx]` (first block) or `source[B,T,16]`.
        precision: "fp32" / "bf16" for this call, None = set_block_precision's global setting."""
        if self.d_model != D_MODEL:
            raise NotImplementedError(f"the fused BST block is built for d_model = {D_MODEL}")
        p, rng = self._dropout_state(source.device)
        precision = self.resolve_precision(precision)
        return _BstBlock.apply((self.nhead, pool, p, rng, precision), seq_len, idx, source, *self._params())

    def forward(self, queries, keys, values, key_padding_mask=None):
        """Self-attention form of the reference signature: queries, keys and values must be the
        same tensor and the mask a key-padding PREFIX mask (True from position len on), which is
        what BSTModel builds (BST/bst.py:226-236)."""
        if not (queries is keys and keys is values):
            raise NotImplementedError("the fused BST block implements self-attention (queries is keys is values)")
        B, T = queries.shape[0], queries.shape[1]
        if key_padding_mask is None:
            seq_len = torch.full((B,), T, dtype=torch.int64, device=queries.device)
        else:
            seq_len = (~key_padding_mask).sum(dim=1).to(torch.int64)
        return self.run(queries, seq_len)


class BSTModel(nn.Module):
    def __init__(self, vocab_dir, hidden_units=[512, 256, 128], dropout_rate=0.1, batch_norm=True,
                 d_model=16, nhead=4, num_transformer_blocks=1, max_seq_length=50, pooling_method='sum'):
        super().__init__()
        self.vocab_sizes = {
            col: len(load_vocabulary(os.path.join(vocab_dir, fname))) + 1
            for col, fname in (("userid", "userid.txt"), ("feedid", "feedid.txt"), ("device", "device.txt"),
                               ("authorid", "authorid.txt"), ("bgm_song_id", "bgm_song_id.txt"),
                               ("bgm_singer_id", "bgm_singer_id.txt"), ("manual_tag_list", "manual_tag_id.txt"))}
        self.num_dense_features = NUM_DENSE
        tables = {col: nn.Embedding(self.vocab_sizes[col], dim) for col, dim in SIDE_TABLES}
        tables["feedid"] = nn.Embedding(self.vocab_sizes["feedid"], 16)
        self.embeddings = nn.ModuleDict(tables)
        self.transformer_blocks = nn.ModuleList([
            BSTTransformer(d_model=16, nhead=nhead, max_len=max_seq_length + 1, dropout=dropout_rate)
            for _ in range(num_transformer_blocks)])
        self.batch_norm = batch_norm
        self.dropout_rate = dropout_rate
        self.pooling_method = pooling_method
        self.block_precision = None       # "fp32" | "bf16" for this model; None = bst.set_block_precision's setting
        width = self.num_dense_features + sum(dim for _, dim in SIDE_TABLES) + 16
        layers = []
        for hidden in hidden_units:
            layers.append(nn.Linear(width, hidden))
            if batch_norm:
                layers.append(nn.BatchNorm1d(hidden))
            layers.append(nn.LeakyReLU(negative_slope=0.01))
            if dropout_rate > 0:
                layers.append(nn.Dropout(dropout_rate))
            width = hidden
        layers.append(nn.Linear(width, 1))
        self.dnn = nn.Sequential(*layers)

    def hot_path(self, dense, category, seq_feedid, seq_length):
        """The part of forward that runs in librank_b200: (side features [B,50], pooled sequence [B,16])."""
        for block in self.transformer_blocks:
            _check_length(int(seq_feedid.shape[1]), block.resolve_precision(self.block_precision))
        cols = [c for c in self.embeddings if c in category]
        side = GatherConcat.apply(len(cols), dense, *[category[c] for c in cols],
                                  *[self.embeddings[c].weight for c in cols])
        pool = 'sum' if self.pooling_method == 'sum' else 'mean'
        blocks = list(self.transformer_blocks)
        if not blocks:      # no transformer: the reference pools the raw sequence embeddings
            raise NotImplementedError("BSTModel needs at least one transformer block on the fused path")
        feed = self.embeddings['feedid']
        if isinstance(feed, RowShardedEmbedding):
            # scaled configuration: the table is row-sharded over the ranks; the rows arrive
            # owner-sorted through the all-to-all and idx becomes the inverse permutation
            x, idx = feed.exchange(seq_feedid)
        else:
            x, idx = feed.weight, seq_feedid
        for i, block in enumerate(blocks):
            last = i == len(blocks) - 1
            x = block.run(x, seq_length, idx=idx, pool=pool if last else None, precision=self.block_precision)
            idx = None
        return side, x

    def forward(self, dense, category, seq_feedid, seq_length):
        side, x = self.hot_path(dense, category, seq_feedid, seq_length)
        all_features = torch.cat([side, x], dim=1)
        logits = run_tower(list(self.dnn), all_features)      # = self.dnn(all_features), BatchNorm1d+LeakyReLU fused
        probabilities = torch.sigmoid(logits)
        return probabilities, logits
