"""GPU parity of the index/integer machinery: gather (bit-exact), occurrence order (bit-exact),
segment reduction vs. the sequential oracle."""
import numpy as np
import pytest
import torch

import rank_b200
from rank_b200.sparse import GradSource, OccurrencePlan, gather_concat
from oracle import interactions as X

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _u32(t):
    return t.cpu().numpy().view(np.uint32)


@pytest.mark.parametrize("sizes,rows", [
    ([5], [3]),                                   # tiny, hot rows
    ([4097, 1, 300], [3, 70000, 17]),             # ragged, crosses a sort tile, 3 radix passes
    ([8192] * 6, [19627, 3, 18790, 25160, 17501, 351]),   # the DCN fields at batch 8192
    ([0, 50], [9, 9]),                            # an empty column
    ([409600, 8192], [106445, 106445]),           # DIN history + target at batch 8192
])
def test_plan_is_the_stable_order(sizes, rows):
    gen = torch.Generator().manual_seed(1)
    cols = [torch.randint(0, r, (n,), generator=gen, dtype=torch.int64) for n, r in zip(sizes, rows)]
    plan = OccurrencePlan([c.to(DEV) for c in cols], rows, direct=False)
    torch.cuda.synchronize()
    keys, perm = X.stable_occurrence_order([c.numpy() for c in cols], rows)
    n = sum(sizes)
    assert np.array_equal(_u32(plan.sorted_keys)[:n], keys)
    assert np.array_equal(_u32(plan.perm)[:n], perm)
    rank_b200.check_index_errors()


def test_plan_flags_out_of_range_index():
    idx = torch.tensor([0, 5, 2], dtype=torch.int64, device=DEV)
    OccurrencePlan([idx], [4], direct=False)
    with pytest.raises(IndexError):
        rank_b200.check_index_errors()
    rank_b200.check_index_errors()    # the flag is cleared by the raise
    # the one-launch reduction reports it too (and counts the occurrence as row 0, like the forward)
    g = torch.ones(3, 2, device=DEV)
    (dw,) = OccurrencePlan([idx], [4]).reduce_to_dense([GradSource(g, 0, 2, 2, 4, 0)])
    assert dw.cpu().tolist() == [[2.0, 2.0], [0.0, 0.0], [1.0, 1.0], [0.0, 0.0]]
    with pytest.raises(IndexError):
        rank_b200.check_index_errors()


@pytest.mark.parametrize("direct", [True, False], ids=["direct", "sorted"])
@pytest.mark.parametrize("n,rows,dim", [(1, 1, 1), (100, 3, 2), (5000, 3, 16), (8192, 351, 4),
                                         (8192, 19627, 16), (3000, 40, 32), (777, 11, 5), (8192, 1, 4),
                                         (8192, 257, 1), (33, 256, 8), (8191, 106445, 16),
                                         (65536, 106445, 1)])
def test_segment_reduce_matches_sequential_sum(n, rows, dim, direct):
    """Both reductions — the one-launch output-partitioned kernel for per-sample columns (n <= 8192) and
    the sorted segment reduction — against the sequential CPU sum."""
    gen = torch.Generator().manual_seed(n + dim)
    idx = torch.randint(0, rows, (n,), generator=gen, dtype=torch.int64)
    if n >= 1000:
        idx[: n // 3] = idx[0]                      # one hot row: a run longer than a warp's share
    ld = dim + 3
    g = torch.randn(n, ld, generator=gen)
    plan = OccurrencePlan([idx.to(DEV)], [rows], direct=direct)
    assert plan.direct == [direct and n <= 8192]
    gd = g.to(DEV)
    (dw,) = plan.reduce_to_dense([GradSource(gd, 1, ld, dim, rows, 0)])
    want = X.dense_embedding_grad(idx.numpy(), g[:, 1:1 + dim].numpy(), rows)
    got = dw.cpu().numpy()
    # rows met once or within one 16-occurrence chunk are summed in exactly the oracle's order
    assert np.allclose(got, want, rtol=1e-5, atol=1e-5 * max(1.0, np.abs(want).max()))
    untouched = np.setdiff1d(np.arange(rows), idx.numpy())
    assert not got[untouched].any()


@pytest.mark.parametrize("direct", [True, False], ids=["direct", "sorted"])
@pytest.mark.parametrize("n,rows,dim", [(8192, 23, 128), (5000, 3, 64), (3000, 40, 36), (8192, 2, 100),
                                         (4000, 5, 50)])
def test_reduce_wide_rows_hit_hundreds_of_times(n, rows, dim, direct):
    """Rows wider than 32 floats (2 or 4 per lane) whose runs are longer than a warp's share, so that every
    warp of the CTA sums a slice of the same row (a DeepFM embedding of 64 or 128 and its `device` field)."""
    gen = torch.Generator().manual_seed(n + dim)
    idx = torch.randint(0, rows, (n,), generator=gen, dtype=torch.int64)
    off = 4 if dim % 4 == 0 else 2
    ld = dim + off
    g = torch.randn(n, ld, generator=gen)
    plan = OccurrencePlan([idx.to(DEV)], [rows], direct=direct)
    (dw,) = plan.reduce_to_dense([GradSource(g.to(DEV), off, ld, dim, rows, 0)])
    want = X.dense_embedding_grad(idx.numpy(), g[:, off:off + dim].numpy(), rows)
    assert np.allclose(dw.cpu().numpy(), want, rtol=1e-5, atol=1e-5 * np.abs(want).max())


@pytest.mark.parametrize("direct", [True, False], ids=["direct", "sorted"])
def test_segment_reduce_is_deterministic_and_shares_a_plan(direct):
    gen = torch.Generator().manual_seed(5)
    idx = [torch.randint(0, r, (4096,), generator=gen, dtype=torch.int64).to(DEV) for r in (3, 1000)]
    plan = OccurrencePlan(idx, [3, 1000], direct=direct)
    g16 = torch.randn(4096, 32, generator=gen).to(DEV)
    g1 = torch.randn(4096, 1, generator=gen).to(DEV)
    src = [GradSource(g16, 0, 32, 16, 3, 0), GradSource(g16, 16, 32, 16, 1000, 1),
           GradSource(g1, 0, 1, 1, 3, 0), GradSource(g1, 0, 1, 1, 1000, 1)]
    a = [t.clone() for t in plan.reduce_to_dense(src)]
    b = plan.reduce_to_dense(src)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    want = X.dense_embedding_grad(idx[1].cpu().numpy(), g16[:, 16:].cpu().numpy(), 1000)
    assert np.allclose(a[1].cpu().numpy(), want, rtol=1e-5, atol=1e-5)
    want1 = X.dense_embedding_grad(idx[0].cpu().numpy(), g1.cpu().numpy(), 3)
    assert np.allclose(a[2].cpu().numpy(), want1, rtol=1e-5, atol=1e-4)


def test_mixed_direct_and_sorted_fields_in_one_plan():
    """A per-sample column (direct) and a padded history (sorted, dead positions dropped) in one plan,
    sources given in an order that interleaves the two kinds."""
    from rank_b200 import _lib
    gen = torch.Generator().manual_seed(12)
    B, T, rows = 700, 9, 500
    cat = torch.randint(0, 40, (B,), generator=gen, dtype=torch.int64)
    hist = torch.randint(0, rows, (B, T), generator=gen, dtype=torch.int64)
    length = torch.randint(0, T + 1, (B,), generator=gen, dtype=torch.int64)
    live = torch.arange(T).expand(B, T) < length.unsqueeze(1)
    plan = OccurrencePlan([cat.to(DEV), hist.view(-1).to(DEV)], [40, rows], seq_len=[None, length.to(DEV)],
                          live_mode=[_lib.LIVE_ALL, _lib.LIVE_PREFIX])
    assert plan.direct == [True, False]
    g_cat = torch.randn(B, 4, generator=gen)
    g_hist = torch.randn(B * T, 16, generator=gen) * live.view(-1, 1)
    d_hist, d_cat = plan.reduce_to_dense([GradSource(g_hist.to(DEV), 0, 16, 16, rows, 1),
                                          GradSource(g_cat.to(DEV), 0, 4, 4, 40, 0)])
    assert np.allclose(d_cat.cpu().numpy(), X.dense_embedding_grad(cat.numpy(), g_cat.numpy(), 40), rtol=1e-5, atol=1e-5)
    assert np.allclose(d_hist.cpu().numpy(), X.dense_embedding_grad(hist.view(-1).numpy(), g_hist.numpy(), rows),
                       rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("dims,n_dense", [([16, 2, 4, 4, 4, 4], 16), ([16] * 6, 0), ([32] * 10, 16),
                                           ([1, 3, 5], 2)])
def test_gather_concat_is_bit_exact(dims, n_dense):
    gen = torch.Generator().manual_seed(9)
    B = 1000
    tables = [torch.randn(50 + 7 * k, d, generator=gen) for k, d in enumerate(dims)]
    idx = [torch.randint(0, t.shape[0], (B,), generator=gen, dtype=torch.int64) for t in tables]
    dense = torch.randn(B, n_dense, generator=gen) if n_dense else None
    offs, off = [], n_dense
    for d in dims:
        offs.append(off)
        off += d
    out = gather_concat([t.to(DEV) for t in tables], [i.to(DEV) for i in idx], offs,
                        None if dense is None else dense.to(DEV))
    want = X.concat_features(dense if dense is not None else torch.zeros(B, 0), tables, idx)
    assert torch.equal(out.cpu(), want)
