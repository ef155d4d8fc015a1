"""numpy restatement of the integer AUC scheme of csrc/metrics.cu (used by test_metrics.py and
test_gpu_metrics.py), and the sklearn definitions it must agree with."""
import numpy as np
from sklearn.metrics import roc_auc_score


def score_keys(scores):
    """metrics.cu::score_key: -0.0 -> +0.0, then flip every bit of negatives, only the sign bit of positives."""
    u = np.ascontiguousarray(scores, dtype=np.float32).view(np.uint32).copy()
    u[u == 0x80000000] = 0
    return np.where(u & 0x80000000, ~u, u | np.uint32(0x80000000)).astype(np.uint32)


def _sorted(scores, labels, groups):
    key = score_keys(scores)
    g = np.zeros(len(key), np.int64) if groups is None else np.asarray(groups, np.int64)
    order = np.lexsort((key, g))              # by group, then score key; stable
    return key[order], g[order], np.asarray(labels)[order] > 0.5


def element_counts(scores, labels, groups=None, num_groups=1):
    """The kernel's per-element form: (2U, P, N) of every group as int64 arrays of num_groups entries.
    positive: 2 (NRS - NGS) + (NC - NRS);  negative: (j - RS) - (NC - NRS)."""
    k, g, y = _sorted(scores, labels, groups)
    n = len(k)
    u2, pos, neg = (np.zeros(num_groups, np.int64) for _ in range(3))
    if n == 0:
        return u2, pos, neg
    j = np.arange(n, dtype=np.int64)
    is_gs = np.ones(n, bool)
    is_gs[1:] = g[1:] != g[:-1]
    is_rs = is_gs.copy()
    is_rs[1:] |= k[1:] != k[:-1]
    isneg = (~y).astype(np.int64)
    NC = np.cumsum(isneg) - isneg
    RS = np.maximum.accumulate(np.where(is_rs, j, -1))
    GS = np.maximum.accumulate(np.where(is_gs, j, -1))
    NRS, NGS = NC[RS], NC[GS]
    c = np.where(y, 2 * (NRS - NGS) + (NC - NRS), (j - RS) - (NC - NRS))
    starts = np.flatnonzero(is_gs)
    ids = g[starts]
    u2[ids] = np.add.reduceat(c, starts)
    neg[ids] = np.add.reduceat(isneg, starts)
    pos[ids] = np.add.reduceat(1 - isneg, starts)
    return u2, pos, neg


def run_counts(scores, labels, groups=None, num_groups=1):
    """The run form of the scheme: every run r of equal (group, key) adds
    pos_r * (2 neg_before_r + neg_r) to its group's 2U (plain Python loop; small inputs)."""
    k, g, y = _sorted(scores, labels, groups)
    u2, pos, neg = [0] * num_groups, [0] * num_groups, [0] * num_groups
    i = 0
    while i < len(k):
        e = i
        while e < len(k) and k[e] == k[i] and g[e] == g[i]:
            e += 1
        p_r = int(y[i:e].sum())
        n_r = (e - i) - p_r
        gi = int(g[i])
        u2[gi] += p_r * (2 * neg[gi] + n_r)    # neg[gi] so far = negatives below the run in its group
        pos[gi] += p_r
        neg[gi] += n_r
        i = e
    return u2, pos, neg


def auc_from_counts(u2, pos, neg):
    return int(u2) / (2 * int(pos) * int(neg))


def host_auc(scores, labels):
    u2, p, n = element_counts(scores, labels)
    return auc_from_counts(u2[0], p[0], n[0])


def host_uauc(scores, labels, groups, num_groups):
    u2, p, n = element_counts(scores, labels, groups, num_groups)
    valid = (p > 0) & (n > 0)
    aucs = [auc_from_counts(a, b, c) for a, b, c in zip(u2[valid], p[valid], n[valid])]
    return sum(aucs) / len(aucs)


def sklearn_uauc(scores, labels, groups):
    """The challenge's uAUC: roc_auc_score per user whose labels are not all equal, then the plain mean."""
    labels, scores, groups = np.asarray(labels), np.asarray(scores), np.asarray(groups)
    order = np.argsort(groups, kind="stable")
    g = groups[order]
    cuts = np.flatnonzero(np.diff(g)) + 1
    total, count = 0.0, 0
    for idx in np.split(order, cuts):
        y = labels[idx]
        if y.min() == y.max():
            continue
        total += roc_auc_score(y, scores[idx])
        count += 1
    return total / count


def zipf_users(rng, n, num_users, alpha=1.05):
    """Users drawn with a Zipf law over ranks, as the WeChat interaction logs are."""
    w = np.arange(1, num_users + 1, dtype=np.float64) ** -alpha
    return rng.permutation(num_users)[rng.choice(num_users, size=n, p=w / w.sum())].astype(np.int64)
