"""Evaluation metrics on the device: exact ROC AUC, per-user AUC (uAUC), log loss and accuracy.

The reference ends every step with `loss.item(); label.cpu(); prob.cpu()` and every epoch with sklearn's
`roc_auc_score` / `accuracy_score` over host lists (DeepFM/deepfm.py:173-180, :184-208): one device->host
synchronisation per step and a host sort of the whole evaluation set.  `BinaryMetrics` keeps the scores
on the device instead.  `update` is one kernel launch (csrc/metrics.cu) with no synchronisation, so it can
sit inside a captured CUDA graph; `compute` sorts on the device and reads back one small result.

AUC is computed from integer counts (csrc/metrics.cu): it equals sklearn's tie-averaged `roc_auc_score`
to the last bit of the final division and does not depend on the order of the samples or on how they
were split into `update` calls.  uAUC is the challenge's metric: the AUC of every group (user) that has
both classes, averaged over those groups.

    metrics = BinaryMetrics(len(eval_set), device, num_groups=table_heights(vocab_dir, ["userid"])["userid"])
    for batch in loader:
        prob = model(...)[0]
        metrics.update(prob, batch["label"], batch["category"]["userid"])
    print(metrics.compute())     # {'n', 'auc', 'logloss', 'accuracy', 'uauc'}
    metrics.reset()

Under data parallelism each rank updates with its own shard, and `metrics.all_gather().compute()` gives every
rank the metrics of all ranks' samples together (one collective per buffer and one merge launch,
csrc/metrics.cu rk_metrics_merge).
"""
from __future__ import annotations

import torch

from . import _lib

_MAX_N = 1 << 31


class BinaryMetrics:
    """Accumulates up to `capacity` (score, label[, group]) samples on `device`.

    Scores are fp32 probabilities for `logloss` / `accuracy`; AUC and uAUC take any finite scores.
    Labels must be 0 or 1.  With `num_groups`, every `update` takes a group id in [0, num_groups) per
    sample (e.g. `category["userid"]`) and `compute` also returns `uauc`.
    """

    def __init__(self, capacity: int, device, num_groups: int | None = None):
        capacity = int(capacity)
        if not 1 <= capacity < _MAX_N:
            raise ValueError(f"capacity={capacity} outside [1, 2^31)")
        if num_groups is not None:
            num_groups = int(num_groups)
            if not 1 <= num_groups < _MAX_N:
                raise ValueError(f"num_groups={num_groups} outside [1, 2^31)")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.RankB200Error(f"BinaryMetrics: device {self.device}; the metrics run on CUDA only "
                                     "(no CPU fallback)")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.capacity = capacity
        self.num_groups = num_groups
        self.scores = torch.empty(capacity, dtype=torch.float32, device=self.device)
        self.labels = torch.empty(capacity, dtype=torch.float32, device=self.device)
        self.groups = None if num_groups is None else torch.empty(capacity, dtype=torch.int64, device=self.device)
        # [count, the append launch's arrival counter, status bits (low 32 bits)]: one read gives both
        self._state = torch.zeros(3, dtype=torch.int64, device=self.device)
        self._result = torch.zeros(_lib.C.sizeof(_lib.RkMetricsResult) // 8, dtype=torch.int64, device=self.device)
        self._ws = None
        self._gather = None     # (group, world, gather buffers, merged metrics) of all_gather, made on its first call

    def reset(self) -> None:
        """Forget every sample and every raised error (enqueued on the current stream)."""
        self._state.zero_()

    def update(self, prob: torch.Tensor, label: torch.Tensor, group: torch.Tensor | None = None) -> None:
        """Append a batch: `prob` [B] or [B, 1] fp32, `label` [B] (float32; other dtypes are cast),
        `group` [B] int64 when the metrics were built with `num_groups`.  One launch, no sync."""
        if (group is None) != (self.num_groups is None):
            raise ValueError("group ids are required exactly when BinaryMetrics has num_groups")
        prob = self._input(prob, "prob", torch.float32)
        if label.dtype != torch.float32:
            label = label.to(torch.float32)
        label = self._input(label, "label", torch.float32)
        B = prob.numel()
        if label.numel() != B:
            raise ValueError(f"label has {label.numel()} elements, prob has {B}")
        if group is not None:
            group = self._input(group, "group", torch.int64)
            if group.numel() != B:
                raise ValueError(f"group has {group.numel()} elements, prob has {B}")
        state = self._state.data_ptr()
        rc = _lib.load().rk_metrics_append(
            prob.data_ptr(), label.data_ptr(), _lib.ptr(group), B, self.scores.data_ptr(), self.labels.data_ptr(),
            _lib.ptr(self.groups), self.capacity, self.num_groups or 0, state, state + 16, _lib.stream_ptr())
        _lib.check(rc, "rk_metrics_append")

    def _input(self, t, name, dtype):
        t = _lib.require_cuda(t, name, dtype)
        if t.device != self.device:
            raise ValueError(f"{name} is on {t.device}, the metrics on {self.device}")
        if t.dim() == 2 and t.shape[1] == 1:
            t = t.reshape(-1)
        if t.dim() != 1:
            raise ValueError(f"{name}: expected shape [B] or [B, 1], got {tuple(t.shape)}")
        return t

    def compute(self) -> dict:
        """{'n', 'auc', 'logloss', 'accuracy'} and, with groups, 'uauc'.  Two device->host reads: the
        count and the result.  Raises ValueError where sklearn would (one class only, NaN, bad labels),
        for bad group ids, for samples dropped past capacity and for probabilities outside [0, 1]."""
        return self._compute(probabilities=True)

    def _compute(self, probabilities: bool) -> dict:
        state = self._state.cpu()
        n, status = int(state[0]), int(state[2]) & 0xFFFFFFFF
        if status & _lib.METRICS_OVERFLOW:
            raise ValueError(f"more than capacity={self.capacity} samples were appended; the rest were dropped")
        if status & _lib.METRICS_NONFINITE:
            raise ValueError("Input contains NaN or infinity.")
        if status & _lib.METRICS_BAD_LABEL:
            raise ValueError("y_true takes values other than 0 and 1")
        if status & _lib.METRICS_BAD_GROUP:
            raise ValueError(f"a group id is outside [0, {self.num_groups})")
        if probabilities and status & _lib.METRICS_NOT_PROB:
            raise ValueError("y_prob contains values outside [0, 1]: log loss and accuracy need probabilities")
        if n == 0:
            raise ValueError("no samples: the metrics are not defined")
        lib = _lib.load()
        groups = self.num_groups or 0
        need = lib.rk_metrics_workspace_bytes(n, groups)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        rc = lib.rk_metrics_compute(self.scores.data_ptr(), self.labels.data_ptr(), _lib.ptr(self.groups), n, groups,
                                    self._ws.data_ptr(), self._ws.numel(), self._result.data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "rk_metrics_compute")
        r = _lib.RkMetricsResult.from_buffer_copy(self._result.cpu().numpy().tobytes())
        if r.pos == 0 or r.neg == 0:
            raise ValueError("Only one class is present in y_true. ROC AUC score is not defined in that case.")
        out = {"n": n, "auc": r.u2 / (2 * r.pos * r.neg)}   # Python ints: a correctly rounded division
        if probabilities:
            out["logloss"] = r.logloss_sum / n
            out["accuracy"] = r.correct / n
        if self.num_groups is not None:
            if r.valid_groups == 0:
                raise ValueError("No group has both classes: uAUC is not defined.")
            out["uauc"] = r.uauc_sum / r.valid_groups
        return out

    def all_gather(self, group=None) -> "BinaryMetrics":
        """The samples of every rank of the process group `group` (default: the world) in one `BinaryMetrics`
        of capacity world * capacity, whose `compute()` gives the metrics of the whole evaluation set: the
        single-process result, since AUC and uAUC do not depend on the order of the samples.  The storage
        order is rank-major (rank 0's samples, then rank 1's, ...).  Every rank of the group must call it.

        The first call is eager: it exchanges (capacity, num_groups) on the host, raises the same ValueError
        on every rank if they differ, and allocates the gather buffers and the returned object.  Every later
        call returns that same object and enqueues device work only, on the current stream: one
        `all_gather_into_tensor` per buffer (scores, labels, groups, state) and one `rk_metrics_merge`
        launch.  It can be captured in a CUDA graph, e.g. with the last evaluation step.  An error raised on
        any rank (NaN, a bad label or group id, samples past capacity) travels in the merged status, so
        `compute()` on the result raises the same ValueError on every rank.

        Without an initialised process group the world is this process alone, and the result's `compute()`
        equals `self.compute()`."""
        import torch.distributed as dist
        lib = _lib.load()
        distributed = dist.is_available() and dist.is_initialized()
        if self._gather is None:
            self._gather = self._gather_setup(group if distributed else None, distributed)
        elif group is not self._gather[0]:
            raise ValueError("all_gather: a BinaryMetrics gathers over the group of its first all_gather call")
        group, world, bufs, merged = self._gather
        if distributed:
            for dst, src in zip(bufs, (self.scores, self.labels, self.groups, self._state)):
                if src is not None:
                    dist.all_gather_into_tensor(dst, src, group=group)
        score_g, label_g, group_g, state_g = bufs
        rc = lib.rk_metrics_merge(score_g.data_ptr(), label_g.data_ptr(), _lib.ptr(group_g), state_g.data_ptr(),
                                  world, self.capacity, merged.scores.data_ptr(), merged.labels.data_ptr(),
                                  _lib.ptr(merged.groups), merged._state.data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "rk_metrics_merge")
        return merged

    def _gather_setup(self, group, distributed):
        if not distributed:
            # world 1: the merge reads this object's own buffers
            bufs = (self.scores, self.labels, self.groups, self._state)
            return group, 1, bufs, BinaryMetrics(self.capacity, self.device, self.num_groups)
        import torch.distributed as dist
        world = dist.get_world_size(group)
        mine = torch.tensor([self.capacity, self.num_groups or 0], dtype=torch.int64, device=self.device)
        every = torch.empty(2 * world, dtype=torch.int64, device=self.device)
        dist.all_gather_into_tensor(every, mine, group=group)
        config = [tuple(c) for c in every.view(world, 2).tolist()]
        if any(c != config[0] for c in config):
            raise ValueError("all_gather: the ranks' BinaryMetrics differ in (capacity, num_groups or 0): "
                             + ", ".join(f"rank {r}: {c}" for r, c in enumerate(config)))
        merged = BinaryMetrics(world * self.capacity, self.device, self.num_groups)   # ValueError past 2^31
        n = world * self.capacity
        bufs = (torch.empty(n, dtype=torch.float32, device=self.device),
                torch.empty(n, dtype=torch.float32, device=self.device),
                None if self.groups is None else torch.empty(n, dtype=torch.int64, device=self.device),
                torch.empty(3 * world, dtype=torch.int64, device=self.device))
        return group, world, bufs, merged


def _one_shot(scores, labels, groups=None, num_groups=None) -> dict:
    scores = scores.reshape(-1) if scores.dim() == 2 and scores.shape[1] == 1 else scores
    m = BinaryMetrics(max(scores.numel(), 1), scores.device, num_groups)
    m.update(scores, labels, groups)
    return m._compute(probabilities=False)


def roc_auc(scores: torch.Tensor, labels: torch.Tensor) -> float:
    """sklearn.metrics.roc_auc_score(labels, scores) on the device; any finite fp32 scores (e.g. logits)."""
    return _one_shot(scores, labels)["auc"]


def group_auc(scores: torch.Tensor, labels: torch.Tensor, groups: torch.Tensor, num_groups: int) -> float:
    """The mean over groups with both classes of each group's ROC AUC (the challenge's uAUC)."""
    return _one_shot(scores, labels, groups, num_groups)["uauc"]
