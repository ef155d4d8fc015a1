"""Row-wise Adam for embedding tables with sparse (COO) gradients (SURVEY 8(f) item 3, opt-in).

`RowwiseAdam` has the arithmetic and state of `torch.optim.SparseAdam` — moments and weights of the
rows a step does not touch are left alone, the bias correction uses the global step — but one CUDA
kernel (csrc/optim.cu) updates weight, exp_avg and exp_avg_sq of the touched rows in place instead
of SparseAdam's dozen sparse-tensor kernels.  It consumes (a) coalesced sparse gradients — what
`RowShardedEmbedding` produces for the row-sharded BST table (sharded.py) and what
`nn.Embedding(sparse=True)` produces — and (b) the `touched_grad` the REPLICATED tables of every
model receive after `rank_b200.sparse.set_table_gradients("touched")`: distinct rows + summed
gradient rows with the count on the device, so no dense `[V, D]` slab is written by the backward,
no dense Adam sweeps the tables, and nothing synchronises with the host.  The reference itself uses dense `optim.Adam`; dense Adam also
decays the moments of untouched rows, so this is a different optimizer, not a drop-in.

`Adam` is the drop-in: the reference's dense Adam (bit-identical to torch's fused Adam) over every parameter in
one launch, fed by dense `.grad`s or by the same `touched_grad`s, where the untouched rows take a zero gradient.
"""
from __future__ import annotations

import torch

from . import _lib


class RowwiseAdam(torch.optim.Optimizer):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8):
        if lr <= 0 or eps <= 0 or not (0 <= betas[0] < 1) or not (0 <= betas[1] < 1):
            raise ValueError("RowwiseAdam: invalid lr / eps / betas")
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps))

    def _state(self, p):
        state = self.state[p]
        if not state:
            state["step"] = 0
            state["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
            state["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
        return state

    def _step_touched(self, lib, group, p, touched):
        """A `sparse.TouchedRows` gradient (set_table_gradients("touched")): the count stays on the device."""
        if p.dim() != 2 or tuple(touched.shape) != tuple(p.shape):
            raise RuntimeError("RowwiseAdam: touched-rows gradient does not match its table")
        w = _lib.require_cuda(p.data, "table", torch.float32)
        if w.data_ptr() != p.data.data_ptr():
            raise RuntimeError("RowwiseAdam: the table must be contiguous")
        state = self._state(p)
        state["step"] += 1
        cap = int(touched.rows.numel())
        if cap == 0:
            return
        beta1, beta2 = group["betas"]
        rc = lib.rk_rowwise_adam_touched(w.data_ptr(), state["exp_avg"].data_ptr(), state["exp_avg_sq"].data_ptr(),
                                         touched.rows.data_ptr(), touched.values.data_ptr(), touched.count.data_ptr(),
                                         cap, int(p.shape[1]), int(p.shape[0]), group["lr"], beta1, beta2,
                                         group["eps"], state["step"], _lib.err_flag(p.device).data_ptr(),
                                         _lib.stream_ptr())
        _lib.check(rc, "rk_rowwise_adam_touched")

    def zero_grad(self, set_to_none: bool = True):
        super().zero_grad(set_to_none)
        for group in self.param_groups:
            for p in group["params"]:
                if getattr(p, "touched_grad", None) is not None:
                    p.touched_grad = None

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        lib = _lib.load()
        for group in self.param_groups:
            beta1, beta2 = group["betas"]
            for p in group["params"]:
                touched = getattr(p, "touched_grad", None)
                if p.grad is None and touched is None:
                    continue
                if touched is not None:
                    if p.grad is not None:
                        raise RuntimeError("RowwiseAdam: a table carries both .grad and .touched_grad")
                    self._step_touched(lib, group, p, touched)
                    p.touched_grad = None
                    continue
                if not p.grad.is_sparse:
                    raise RuntimeError("RowwiseAdam takes sparse gradients (rows, values); use torch.optim.Adam "
                                       "for dense ones")
                if p.dim() != 2:
                    raise RuntimeError("RowwiseAdam updates 2-D tables")
                w = _lib.require_cuda(p.data, "table", torch.float32)
                if w.data_ptr() != p.data.data_ptr():
                    raise RuntimeError("RowwiseAdam: the table must be contiguous")
                state = self._state(p)
                state["step"] += 1
                grad = p.grad.coalesce()            # one summed row per touched row, as SparseAdam requires
                rows = grad.indices()[0].contiguous()
                vals = _lib.require_cuda(grad.values(), "gradient rows", torch.float32)
                rc = lib.rk_rowwise_adam(w.data_ptr(), state["exp_avg"].data_ptr(), state["exp_avg_sq"].data_ptr(),
                                         rows.data_ptr(), vals.data_ptr(), int(rows.numel()), int(p.shape[1]),
                                         int(p.shape[0]), group["lr"], beta1, beta2, group["eps"], state["step"],
                                         _lib.err_flag(p.device).data_ptr(), _lib.stream_ptr())
                _lib.check(rc, "rk_rowwise_adam")
        return loss


# torch.optim.Adam's group keys, with the only values this optimizer implements.  Kept in every group so that a
# state_dict moves between the two in either direction: torch.optim.Adam reads weight_decay / amsgrad / maximize
# from the group, and fused=True makes a torch.optim.Adam that loads our state continue with the same arithmetic.
_TORCH_ADAM_FLAGS = dict(weight_decay=0.0, amsgrad=False, maximize=False, foreach=None, capturable=True,
                         differentiable=False, fused=True, decoupled_weight_decay=False)


def _check_hyper(lr, betas, eps, weight_decay=0.0, amsgrad=False, maximize=False):
    if weight_decay != 0:
        raise ValueError("rank_b200.Adam has no weight decay (weight_decay must be 0)")
    if amsgrad:
        raise ValueError("rank_b200.Adam has no amsgrad")
    if maximize:
        raise ValueError("rank_b200.Adam has no maximize")
    for name, x in (("lr", lr), ("eps", eps), ("betas[0]", betas[0]), ("betas[1]", betas[1])):
        if isinstance(x, bool) or not isinstance(x, (int, float)):
            raise ValueError(f"rank_b200.Adam: {name} must be a number, got {type(x).__name__}")
    if not lr >= 0.0:
        raise ValueError(f"Invalid learning rate: {lr}")
    if not eps >= 0.0:
        raise ValueError(f"Invalid epsilon value: {eps}")
    if not (0.0 <= betas[0] < 1.0 and 0.0 <= betas[1] < 1.0):
        raise ValueError(f"Invalid beta parameters: {tuple(betas)}")


class Adam(torch.optim.Optimizer):
    """Dense Adam, bit-identical to `torch.optim.Adam(params, lr, betas, eps, fused=True)`: the drop-in for the
    reference's `optim.Adam(model.parameters(), lr)`.

    One launch of `rk_adam_step` (csrc/optim.cu) updates every parameter, after one `torch._foreach_add_` of the
    step counts, with nothing synchronising with the host, so `step()` can be captured in a CUDA graph together
    with the forward and backward.  A parameter's gradient is its dense `.grad`, or the `touched_grad` a table
    receives after `rank_b200.sparse.set_table_gradients("touched")`: the rows a batch did not touch take a zero
    gradient, so their moments decay exactly as in dense Adam, but no dense gradient is ever written.  Parameters
    with neither are skipped, as torch skips them.

    State keys and formats are torch's fused ones (`step` a 0-d float32 tensor on the parameter's device,
    `exp_avg`, `exp_avg_sq`): a state_dict saved by `torch.optim.Adam` (fused or foreach) loads here, and ours
    loads into `torch.optim.Adam`.  Weight decay, amsgrad and maximize are not implemented and are refused."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, amsgrad=False, *,
                 maximize=False):
        _check_hyper(lr, betas, eps, weight_decay, amsgrad, maximize)
        super().__init__(params, dict(lr=lr, betas=tuple(betas), eps=eps, **_TORCH_ADAM_FLAGS))

    def __setstate__(self, state):
        super().__setstate__(state)
        for group in self.param_groups:
            _check_hyper(group["lr"], group["betas"], group["eps"], group.get("weight_decay", 0.0),
                         group.get("amsgrad", False), group.get("maximize", False))
            group.update(_TORCH_ADAM_FLAGS)
            for p in group["params"]:
                st = self.state.get(p)
                if st and "step" in st:
                    st["step"] = self._step_tensor(st["step"], p)

    @staticmethod
    def _step_tensor(step, p):
        """torch's fused format: a 0-d float32 tensor on the parameter's device (foreach keeps it on the host)."""
        if not torch.is_tensor(step):
            return torch.tensor(float(step), dtype=torch.float32, device=p.device)
        if step.device != p.device or step.dtype != torch.float32 or step.dim() != 0:
            return step.detach().reshape(()).to(device=p.device, dtype=torch.float32)
        return step

    @staticmethod
    def _check(p, touched):
        """Every refusal happens here, for all parameters, before anything is launched."""
        if not p.is_cuda:
            raise _lib.RankB200Error(f"rank_b200.Adam: a parameter is on {p.device}; the update runs on CUDA only "
                                     "(no CPU fallback)")
        if p.dtype != torch.float32:
            raise TypeError(f"rank_b200.Adam updates float32 parameters, got {p.dtype}")
        if not p.is_contiguous():
            raise RuntimeError("rank_b200.Adam: parameters must be contiguous")
        if touched is not None:
            if p.grad is not None:
                raise RuntimeError("rank_b200.Adam: a parameter carries both .grad and .touched_grad (a touched-rows "
                                   "model whose gradients were also made dense, e.g. by GradientAllReducer); keep "
                                   "one of them")
            if p.dim() != 2 or tuple(touched.shape) != tuple(p.shape):
                raise RuntimeError(f"rank_b200.Adam: touched-rows gradient of shape {tuple(touched.shape)} does not "
                                   f"match its table {tuple(p.shape)}")
            cap = touched.rows.numel()
            if (touched.rows.dtype != torch.int64 or touched.count.dtype != torch.int64 or touched.count.numel() < 1
                    or tuple(touched.values.shape) != (cap, p.shape[1]) or touched.values.dtype != torch.float32
                    or not (touched.rows.is_contiguous() and touched.values.is_contiguous())
                    or any(t.device != p.device for t in (touched.rows, touched.values, touched.count))):
                raise RuntimeError("rank_b200.Adam: malformed touched-rows gradient (rows int64 [capacity], values "
                                   "float32 [capacity, dim], count int64, contiguous, on the table's device)")
            return
        g = p.grad
        if g.is_sparse:
            raise RuntimeError("rank_b200.Adam takes dense or touched-rows gradients, not sparse ones; "
                               "RowwiseAdam consumes sparse gradients")
        if g.dtype != torch.float32 or g.device != p.device or g.shape != p.shape:
            raise RuntimeError("rank_b200.Adam: the gradient must be float32 and match its parameter")

    def _state(self, p):
        state = self.state[p]
        if not state:
            state["step"] = torch.zeros((), dtype=torch.float32, device=p.device)
            state["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
            state["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
        else:
            state["step"] = self._step_tensor(state["step"], p)
            for k in ("exp_avg", "exp_avg_sq"):
                if state[k].shape != p.shape or state[k].dtype != torch.float32 or state[k].device != p.device \
                        or not state[k].is_contiguous():
                    raise RuntimeError(f"rank_b200.Adam: state {k!r} does not match its parameter")
        return state

    def zero_grad(self, set_to_none: bool = True):
        super().zero_grad(set_to_none)
        for group in self.param_groups:
            for p in group["params"]:
                if getattr(p, "touched_grad", None) is not None:
                    p.touched_grad = None

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        work = []
        for group in self.param_groups:
            for p in group["params"]:
                touched = getattr(p, "touched_grad", None)
                if p.grad is None and touched is None:
                    continue
                self._check(p, touched)
                work.append((group, p, touched))
        if not work:
            return loss
        lib = _lib.load()
        by_device = {}
        for group, p, touched in work:
            state = self._state(p)
            g = None if touched is not None else p.grad.contiguous()
            by_device.setdefault(p.device, []).append((group, p, touched, g, state))
        for dev, items in by_device.items():
            with torch.cuda.device(dev):
                torch._foreach_add_([it[4]["step"] for it in items], 1)
                stream = torch.cuda.current_stream(dev).cuda_stream
                flag = _lib.err_flag(dev).data_ptr()
                for k in range(0, len(items), _lib.RK_ADAM_MAX_TENSORS):
                    chunk = items[k:k + _lib.RK_ADAM_MAX_TENSORS]
                    descs = (_lib.RkAdamTensor * len(chunk))()
                    for d, (group, p, touched, g, state) in zip(descs, chunk):
                        d.param, d.exp_avg, d.exp_avg_sq = (p.data_ptr(), state["exp_avg"].data_ptr(),
                                                            state["exp_avg_sq"].data_ptr())
                        d.step = state["step"].data_ptr()
                        if touched is None:
                            d.grad = g.data_ptr()
                            d.rows, d.dim = p.numel(), 1
                        else:
                            d.touched_rows = touched.rows.data_ptr()
                            d.touched_values = touched.values.data_ptr()
                            d.touched_count = touched.count.data_ptr()
                            d.capacity = touched.rows.numel()
                            d.rows, d.dim = p.shape
                        d.lr, d.eps = group["lr"], group["eps"]
                        d.beta1, d.beta2 = group["betas"]
                    _lib.check(lib.rk_adam_step(descs, len(chunk), flag, stream), "rk_adam_step")
        for _, p, touched in work:
            if touched is not None:
                p.touched_grad = None
        return loss
