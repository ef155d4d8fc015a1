"""rk_metrics_merge without a GPU: a numpy restatement of the merge (rank-major segments of the clamped counts,
the OR of the statuses) checked against concatenating every rank's prefix, and the entry point's argument
refusals (before any CUDA call).  tests/test_gpu_metrics_dp.py checks the kernel against `merge_reference`."""
import numpy as np
import pytest
import torch

from rank_b200 import _lib


def merge_reference(score_g, label_g, group_g, state_g, world, cap):
    """What rk_metrics_merge writes: (score, label, group or None) of length world * cap, of which the first
    n entries are defined, and the merged state {n, 0, OR of the statuses}.  Rank r's clamped count_r samples
    start at sum_{q<r} count_q; entries past n keep the fill value (NaN / -1) of the outputs."""
    state = np.asarray(state_g, np.int64).reshape(world, 3)
    counts = np.clip(state[:, 0], 0, cap)
    offsets = np.concatenate([[0], np.cumsum(counts)])
    n = int(offsets[-1])
    out = [np.full(world * cap, np.nan, np.float32), np.full(world * cap, np.nan, np.float32),
           None if group_g is None else np.full(world * cap, -1, np.int64)]
    for r in range(world):
        for dst, src in zip(out, (score_g, label_g, group_g)):
            if dst is not None:
                dst[offsets[r]:offsets[r + 1]] = np.asarray(src)[r * cap:r * cap + counts[r]]
    status = 0
    for s in state[:, 2]:
        status |= int(s) & 0xFFFFFFFF
    return out[0], out[1], out[2], np.array([n, 0, status], np.int64)


def _ranks(rng, world, cap, counts, statuses, groups=True):
    """The all-gathered layout of `world` ranks whose buffers hold random samples (every entry, also past the
    count: what an all-gather of a full buffer carries)."""
    score = rng.random(world * cap).astype(np.float32)
    label = (rng.random(world * cap) < 0.4).astype(np.float32)
    group = rng.integers(0, 50, world * cap).astype(np.int64) if groups else None
    state = np.zeros((world, 3), np.int64)
    state[:, 0] = counts
    state[:, 2] = statuses
    return score, label, group, state.reshape(-1)


@pytest.mark.parametrize("groups", [False, True])
@pytest.mark.parametrize("counts", [[5], [0], [7], [0, 7, 3], [7, 7], [2, 0, 9, 7, 0, 1, 7, 4], [-3, 4, 100]])
def test_reference_is_the_concatenation_of_the_rank_prefixes(counts, groups):
    world, cap = len(counts), 7
    rng = np.random.default_rng(len(counts) * 11 + sum(counts))
    statuses = [(1 << (r % 5)) if r % 3 == 1 else 0 for r in range(world)]
    score, label, group, state = _ranks(rng, world, cap, counts, statuses, groups)
    s, y, g, st = merge_reference(score, label, group, state, world, cap)
    clamped = [min(max(c, 0), cap) for c in counts]
    want = [np.concatenate([a[r * cap:r * cap + clamped[r]] for r in range(world)])
            for a in (score, label, group) if a is not None]
    n = sum(clamped)
    assert st[0] == n and st[1] == 0
    assert st[2] == np.bitwise_or.reduce(np.array(statuses, np.int64))
    assert np.array_equal(s[:n], want[0]) and np.array_equal(y[:n], want[1])
    assert (g is None) == (not groups)
    if groups:
        assert np.array_equal(g[:n], want[2])
        assert (g[n:] == -1).all()
    assert np.isnan(s[n:]).all() and np.isnan(y[n:]).all()       # nothing written past the merged count


def test_reference_keeps_only_the_low_32_status_bits():
    score, label, group, state = _ranks(np.random.default_rng(1), 2, 4, [1, 2], [0, 0])
    state[2] = (1 << 40) | _lib.METRICS_NONFINITE
    state[5] = _lib.METRICS_BAD_GROUP
    assert merge_reference(score, label, group, state, 2, 4)[3][2] == _lib.METRICS_NONFINITE | _lib.METRICS_BAD_GROUP


ADDR = 1 << 24          # placeholder device addresses: 16-byte aligned, distinct, never dereferenced


@pytest.mark.skipif(torch.cuda.is_available(),
                    reason="placeholder device addresses: only run where no kernel can launch")
@pytest.mark.parametrize("case", ["world", "capacity", "too_many", "null_score_g", "null_label_g", "null_state_g",
                                  "null_score_out", "null_label_out", "null_state_out", "group_out",
                                  "state_overlap"])
def test_entry_point_refuses_bad_arguments_before_the_device(case):
    lib = _lib.load()
    args = dict(score_g=ADDR * 1, label_g=ADDR * 2, group_g=ADDR * 3, state_g=ADDR * 4, world=4, capacity=100,
                score_out=ADDR * 5, label_out=ADDR * 6, group_out=ADDR * 7, state_out=ADDR * 8)
    if case == "world":
        args["world"] = 0
    elif case == "capacity":
        args["capacity"] = 0
    elif case == "too_many":
        args.update(world=8, capacity=1 << 28)                  # world * capacity = 2^31
    elif case.startswith("null_"):
        args[case[5:]] = None
    elif case == "group_out":
        args["group_out"] = None                                # groups in, nowhere to put them
    elif case == "state_overlap":
        args["state_out"] = args["state_g"] + 8 * 3 * 3         # rank 3's state triple
    rc = lib.rk_metrics_merge(*args.values(), None)
    assert rc < 0, (case, lib.rk_last_error())
    assert b"metrics_merge" in lib.rk_last_error(), case


@pytest.mark.skipif(torch.cuda.is_available(),
                    reason="placeholder device addresses: only run where no kernel can launch")
def test_largest_world_below_2_31_is_not_refused_for_its_size():
    """world * capacity = 2^31 - 1 passes the size check (it is refused here for the NULL output instead, so
    no kernel is launched)."""
    lib = _lib.load()
    rc = lib.rk_metrics_merge(ADDR, ADDR * 2, None, ADDR * 3, 1, (1 << 31) - 1, None, ADDR * 4, None, ADDR * 5, None)
    assert rc < 0 and b"NULL" in lib.rk_last_error()
