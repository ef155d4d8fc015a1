"""Data parallelism for the hot path: one process per GPU, batch split by sample, every rank
holds all tables (SURVEY.md §8e).  The only exchange of a step is the gradient all-reduce.

The reference is single-process (no torch.distributed anywhere); this is new plumbing, kept to
what the path needs: all registered gradients — the dense `[V, D]` table gradients produced by
the segment reduction and the tower gradients — live in ONE flat fp32 buffer (the table gradients
are written there by the reduction kernels themselves, the tower gradients are copied in), which is
averaged with a single NCCL all-reduce over NVLink/NVSwitch (gloo on CPU in the tests) and handed
back as views of that buffer (no copy back).
"""
from __future__ import annotations

import torch
import torch.distributed as dist


class GradientAllReducer:
    """All registered gradients of a replica in ONE all-reduce per step, with no pack copy for the tables.

    The flat buffer has two regions: [tower | tables].  While the reducer is attached (`attach()`, done by
    the constructor) the embedding-gradient reductions of rank_b200.sparse allocate their dense `[V, D]`
    slabs straight out of the table region, so the big gradients are already where the collective reads
    them; only the small tower gradients are copied (one `_foreach_copy_`).  The average is taken by NCCL
    itself (ReduceOp.AVG; gloo: SUM then one scale).  Every call is stream-ordered device work — the whole
    step including the collective can be captured in a CUDA graph (bench.py does)."""

    # bench.py reports it; the collective is always torch.distributed's (NCCL, or gloo in the CPU tests)
    symmetric = None

    def __init__(self, model: torch.nn.Module, group=None, attach=True):
        self.group = group
        # row-sharded tables are owned by one rank each: their gradients are not replicated
        self.params = [p for p in model.parameters()
                       if p.requires_grad and not getattr(p, "_rank_local", False)]
        if not self.params:
            raise ValueError("model has no trainable parameters")
        dev, dtype = self.params[0].device, self.params[0].dtype
        sizes = [p.numel() for p in self.params]
        self.n_staging = (sum(sizes) + 31) // 32 * 32          # the table region starts 128-byte aligned
        # table region: every parameter could be a table, each slab padded to 16 bytes per table
        self.n_slab = sum(sizes) + 4 * len(sizes)
        self.flat = torch.zeros(self.n_staging + self.n_slab, dtype=dtype, device=dev)
        self.views, pos = [], 0
        for p, n in zip(self.params, sizes):
            self.views.append(self.flat[pos:pos + n].view_as(p))
            pos += n
        self._cursor = 0
        self._param_ids = {id(p) for p in self.params}
        self._avg = None
        if attach:
            self.attach()

    @property
    def world_size(self):
        return dist.get_world_size(self.group)

    # ---- slab provider of rank_b200.sparse ------------------------------------------------------
    def attach(self):
        from . import sparse
        sparse.set_slab_provider(self._take)

    def detach(self):
        from . import sparse
        sparse.set_slab_provider(None)

    def _take(self, n_floats, device, params):
        """A chunk of the table region for one backward's dense gradients (None: allocate normally).  Only for
        this reducer's own parameters: another model's backward in the same process must not land here."""
        if device != self.flat.device or self._cursor + n_floats > self.n_slab:
            return None
        if not params or any(p is None or id(p) not in self._param_ids for p in params):
            return None
        lo = self.n_staging + self._cursor
        self._cursor += (n_floats + 3) // 4 * 4
        return self.flat[lo:lo + n_floats]

    def _in_slab(self, g):
        lo = self.flat.data_ptr() + 4 * self.n_staging
        return g is not None and g.device == self.flat.device and lo <= g.data_ptr() < lo + 4 * self.n_slab

    def allreduce(self, grads=None):
        """Average every parameter's gradient over the ranks (call after backward).  `grads`
        (default: each parameter's .grad) lets a CUDA-graph step pass its static tensors.
        Afterwards every parameter's .grad is a view of the reduced buffer."""
        grads = [p.grad for p in self.params] if grads is None else list(grads)
        in_slab = [self._in_slab(g) for g in grads]
        staged = sum(p.numel() for p, s_ in zip(self.params, in_slab) if not s_)
        # the copied gradients sit right below the table region: [n_staging - staged, n_staging + used) is ONE range
        pos = self.n_staging - staged
        lo = pos
        copy_dst, copy_src, zero, out_views = [], [], [], []
        for p, g, s_ in zip(self.params, grads, in_slab):
            if s_:
                out_views.append(g)              # already in the reduced range
                continue
            n = p.numel()
            v = self.flat[pos:pos + n].view_as(p)
            pos += n
            out_views.append(v)
            if g is None:
                zero.append(v)
            elif g.data_ptr() != v.data_ptr():
                copy_dst.append(v)
                copy_src.append(g)
        if copy_dst:
            torch._foreach_copy_(copy_dst, copy_src)
        for v in zero:
            v.zero_()
        lo = lo // 4 * 4                                       # 16-byte aligned start (a few stale floats ride along)
        r = self.flat[lo:self.n_staging + self._cursor]
        if self._avg is None:
            self._avg = dist.get_backend(self.group) == "nccl"
        if self._avg:
            dist.all_reduce(r, op=dist.ReduceOp.AVG, group=self.group)
        else:
            dist.all_reduce(r, op=dist.ReduceOp.SUM, group=self.group)
            r.mul_(1.0 / self.world_size)
        self.reduced_floats = int(r.numel())
        self._cursor = 0
        for v, p in zip(out_views, self.params):
            p.grad = v
        return None

    def flat_gradients(self):
        """All reduced gradients in parameter order, concatenated (a copy; tests and diagnostics)."""
        return torch.cat([p.grad.reshape(-1) for p in self.params])


def shard_batch(batch, rank: int, world: int):
    """Rows [rank*B/world, (rank+1)*B/world) of every tensor of a (nested dict) batch."""
    if torch.is_tensor(batch):
        n = batch.shape[0]
        per = n // world
        return batch[rank * per:(rank + 1) * per]
    return {k: shard_batch(v, rank, world) for k, v in batch.items()}
