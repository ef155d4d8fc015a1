"""Host restatement of the integer AUC scheme of csrc/metrics.cu (CPU; no extension needed), checked
against sklearn: the order-preserving score key, the per-element form of the tie-run numerator the
kernels compute, and its grouped version against the challenge's per-user AUC."""
import numpy as np
import pytest
from sklearn.metrics import roc_auc_score

from metrics_oracle import (auc_from_counts, element_counts, host_auc, host_uauc, run_counts, score_keys,
                            sklearn_uauc, zipf_users)


def float_sweep():
    f = np.float32
    tiny, big = np.finfo(f).tiny, np.finfo(f).max
    sub_min = np.nextafter(f(0), f(1))
    base = np.array([0.0, sub_min, 2 * sub_min, tiny / 2, np.nextafter(tiny, f(0)), tiny, np.nextafter(tiny, f(1)),
                     1e-30, 1e-3, 0.5, np.nextafter(f(0.5), f(0)), np.nextafter(f(0.5), f(1)), 1.0,
                     np.nextafter(f(1), f(2)), 3.0, 1e30, np.nextafter(big, f(0)), big], dtype=f)
    rng = np.random.default_rng(0)
    rand = (rng.standard_normal(4000) * 10.0 ** rng.integers(-40, 38, 4000)).astype(f)
    vals = np.concatenate([base, -base, rand, np.array([-0.0], f)])
    return vals[np.isfinite(vals)]


def test_score_key_is_monotone_and_ties_signed_zeros():
    v = float_sweep()
    v = v[np.argsort(v.astype(np.float64), kind="stable")]
    k = score_keys(v).astype(np.int64)
    d = np.diff(v.astype(np.float64))
    dk = np.diff(k)
    assert np.all(dk[d > 0] > 0)
    assert np.all(dk[d == 0] == 0)
    assert score_keys(np.array([-0.0], np.float32))[0] == score_keys(np.array([0.0], np.float32))[0]
    # neighbouring floats get neighbouring keys (nothing is skipped or folded)
    x = np.float32(1.5)
    assert int(score_keys(np.array([np.nextafter(x, np.float32(2))]))[0]) - int(score_keys(np.array([x]))[0]) == 1
    y = np.float32(-1.5)
    assert int(score_keys(np.array([y]))[0]) - int(score_keys(np.array([np.nextafter(y, np.float32(-2))]))[0]) == 1


def cases():
    rng = np.random.default_rng(1)
    out = []
    for n, rate in ((2, 0.5), (50, 0.3), (1000, 0.1), (20000, 0.0356)):
        y = (rng.random(n) < rate).astype(np.float32)
        y[0], y[-1] = 1.0, 0.0
        s = rng.random(n).astype(np.float32)
        out.append(("random", s, y))
        out.append(("tied_1e-3", np.round(s, 3).astype(np.float32), y))
        out.append(("logits_signed_zero", np.where(rng.random(n) < 0.1, np.float32(0.0) * rng.choice([-1, 1], n),
                                                  rng.standard_normal(n)).astype(np.float32), y))
    return out


@pytest.mark.parametrize("name,s,y", cases(), ids=lambda v: v if isinstance(v, str) else "")
def test_tie_run_numerator_matches_sklearn(name, s, y):
    u2, p, n = element_counts(s, y)
    assert abs(auc_from_counts(u2[0], p[0], n[0]) - roc_auc_score(y, s)) <= 1e-12
    if len(s) <= 1000:
        ru2, rp, rn = run_counts(s, y)
        assert (int(u2[0]), int(p[0]), int(n[0])) == (ru2[0], rp[0], rn[0])


def test_degenerate_orders():
    rng = np.random.default_rng(2)
    y = (rng.random(5000) < 0.2).astype(np.float32)
    y[:2] = [0, 1]
    assert host_auc(np.full(5000, 0.25, np.float32), y) == 0.5
    s = np.sort(rng.random(5000).astype(np.float32))
    order = np.argsort(y, kind="stable")             # negatives first
    assert host_auc(s, y[order]) == 1.0
    assert host_auc(s[::-1].copy(), y[order]) == 0.0
    # order of the input does not matter: the counts are integers
    perm = rng.permutation(5000)
    t = np.round(rng.random(5000), 2).astype(np.float32)
    assert host_auc(t, y) == host_auc(t[perm], y[perm])


def test_grouped_counts_match_challenge_uauc():
    rng = np.random.default_rng(3)
    num_users, n = 19627, 60000
    users = zipf_users(rng, n, num_users)
    y = (rng.random(n) < 0.0356).astype(np.float32)
    s = np.round(rng.random(n), 3).astype(np.float32)
    u2, p, q = element_counts(s, y, users, num_users)
    single = ((p > 0) ^ (q > 0)).sum()
    assert single > 1000 and ((p > 0) & (q > 0)).sum() > 50    # many one-class users, enough valid ones
    assert abs(host_uauc(s, y, users, num_users) - sklearn_uauc(s, y, users)) <= 1e-12
    small = users[:800] % 37
    ru2, rp, rq = run_counts(s[:800], y[:800], small, 37)
    eu2, ep, eq = element_counts(s[:800], y[:800], small, 37)
    assert (list(eu2), list(ep), list(eq)) == (ru2, rp, rq)
