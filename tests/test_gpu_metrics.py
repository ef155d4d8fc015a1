"""BinaryMetrics / roc_auc / group_auc on the device (csrc/metrics.cu) against the host integer oracle
(tests/metrics_oracle.py), sklearn and float64 torch."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from sklearn.metrics import accuracy_score, roc_auc_score

import rank_b200
from rank_b200 import _lib, synthetic
from rank_b200.metrics import BinaryMetrics, group_auc, roc_auc
from metrics_oracle import host_auc, host_uauc, sklearn_uauc, zipf_users

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
USERS = 19627          # the userid table of the WeChat vocabulary (19 626 lines + row 0)


def dataset(n, kind, rate, seed):
    rng = np.random.default_rng(seed)
    y = (rng.random(n) < rate).astype(np.float32)
    y[0], y[-1] = 1.0, 0.0                       # both classes at every n
    if kind == "prob":
        s = rng.random(n).astype(np.float32)
        s[rng.random(n) < 0.01] = 0.0
        s[rng.random(n) < 0.01] = 1.0
    elif kind == "tied":
        s = np.round(rng.random(n), 3).astype(np.float32)
    else:                                        # logits with a share of +0.0 / -0.0
        s = (rng.standard_normal(n) * 3).astype(np.float32)
        z = rng.random(n) < 0.05
        s[z] = np.where(rng.random(z.sum()) < 0.5, np.float32(0.0), np.float32(-0.0))
    return s, y


def run(s, y, g=None, num_groups=None, splits=(1,)):
    """Accumulate in chunks of the given relative sizes, then compute."""
    m = BinaryMetrics(len(s), DEV, num_groups)
    st, yt = torch.from_numpy(s).to(DEV), torch.from_numpy(y).to(DEV)
    gt = None if g is None else torch.from_numpy(g).to(DEV)
    cuts = np.cumsum(np.array(splits, np.float64) / sum(splits) * len(s)).astype(np.int64)
    lo = 0
    for hi in cuts:
        if hi > lo:
            m.update(st[lo:hi], yt[lo:hi], None if gt is None else gt[lo:hi])
        lo = hi
    return m.compute()


@pytest.mark.parametrize("n", [2, 1000, 8192, 2 ** 20 + 17, 4 * 2 ** 20])
@pytest.mark.parametrize("kind,rate", [("prob", 0.3), ("tied", 0.0356), ("logits", 0.0356)])
def test_auc_is_exact(n, kind, rate):
    s, y = dataset(n, kind, rate, seed=n)
    ref = host_auc(s, y)
    auc = roc_auc(torch.from_numpy(s).to(DEV), torch.from_numpy(y).to(DEV))
    assert auc == ref                                        # bit-equal to the integer oracle
    assert abs(auc - roc_auc_score(y, s)) <= 1e-12
    if kind != "logits":
        out = run(s, y)
        assert out["auc"] == ref and out["n"] == n
        expect = F.binary_cross_entropy(torch.from_numpy(s).double(), torch.from_numpy(y).double()).item()
        assert abs(out["logloss"] - expect) <= 1e-12 * expect
        assert out["accuracy"] == accuracy_score(y, s > 0.5)


def grouped(n=300_000, seed=5):
    rng = np.random.default_rng(seed)
    g = zipf_users(rng, n, USERS - 700)             # the last 700 ids get no sample at all
    y = (rng.random(n) < 0.0356).astype(np.float32)
    s = np.round(rng.random(n), 3).astype(np.float32)
    return s, y, g


def test_uauc_matches_per_user_sklearn():
    s, y, g = grouped()
    out = run(s, y, g, USERS)
    assert abs(out["uauc"] - sklearn_uauc(s, y, g)) <= 1e-12
    assert abs(out["uauc"] - host_uauc(s, y, g, USERS)) <= 1e-12
    assert out["auc"] == host_auc(s, y)
    assert abs(group_auc(torch.from_numpy(s).to(DEV), torch.from_numpy(y).to(DEV), torch.from_numpy(g).to(DEV),
                         USERS) - out["uauc"]) == 0.0


def test_results_do_not_depend_on_order_or_split():
    s, y, g = grouped(seed=6)
    a = run(s, y, g, USERS)
    b = run(s, y, g, USERS)
    assert a == b                                            # two runs, every field bit-identical
    c = run(s, y, g, USERS, splits=(3, 1, 7, 2, 5, 1, 1))
    assert c == a                                            # same storage order: log loss too
    perm = np.random.default_rng(7).permutation(len(s))
    d = run(s[perm], y[perm], g[perm], USERS, splits=(2, 9, 4))
    assert (d["auc"], d["uauc"]) == (a["auc"], a["uauc"])
    assert abs(d["logloss"] - a["logloss"]) <= 1e-12 * a["logloss"] and d["accuracy"] == a["accuracy"]


def test_update_captured_in_a_graph_equals_eager():
    B, k = 4096, 6
    rng = np.random.default_rng(8)
    batches = [(rng.random(B).astype(np.float32), (rng.random(B) < 0.1).astype(np.float32),
                rng.integers(0, USERS, B).astype(np.int64)) for _ in range(k)]
    eager = BinaryMetrics(B * k, DEV, USERS)
    for s, y, g in batches:
        eager.update(torch.from_numpy(s).to(DEV), torch.from_numpy(y).to(DEV), torch.from_numpy(g).to(DEV))
    graphed = BinaryMetrics(B * k, DEV, USERS)
    st = torch.zeros(B, 1, device=DEV)
    yt = torch.zeros(B, device=DEV)
    gt = torch.zeros(B, dtype=torch.int64, device=DEV)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                            # warm-up on a side stream, then reset
        graphed.update(st, yt, gt)
    torch.cuda.current_stream().wait_stream(side)
    graphed.reset()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        graphed.update(st, yt, gt)
    for s, y, g in batches:
        st.copy_(torch.from_numpy(s).view(B, 1))
        yt.copy_(torch.from_numpy(y))
        gt.copy_(torch.from_numpy(g))
        graph.replay()
    assert graphed.compute() == eager.compute()


def test_errors_raise_value_error():
    def fresh(groups=False):
        return BinaryMetrics(64, DEV, USERS if groups else None)
    ones = torch.ones(8, device=DEV)
    p = torch.linspace(0.1, 0.9, 8, device=DEV)
    g = torch.arange(8, device=DEV)
    m = fresh()
    m.update(p, ones)
    with pytest.raises(ValueError, match="Only one class"):
        m.compute()
    y = (torch.arange(8, device=DEV) % 2).float()
    m = fresh()
    m.update(torch.where(y > 0, p, torch.full_like(p, float("nan"))), y)
    with pytest.raises(ValueError, match="NaN"):
        m.compute()
    m = fresh()
    m.update(p, y * 2)
    with pytest.raises(ValueError, match="other than 0 and 1"):
        m.compute()
    m = fresh(groups=True)
    m.update(p, y, g + USERS - 4)
    with pytest.raises(ValueError, match="group id"):
        m.compute()
    m = fresh(groups=True)
    m.update(p, y, g * 0)                                   # group 0 has both classes
    m.update(p, y * 0, g + 1)                               # groups 1..8 negatives only: skipped
    assert abs(m.compute()["uauc"] - roc_auc_score(y.cpu().numpy(), p.cpu().numpy())) <= 1e-12
    m = fresh(groups=True)
    m.update(p, (g == 0).float(), g)                        # every group has one class
    with pytest.raises(ValueError, match="No group"):
        m.compute()
    m = fresh()
    m.update(p * 4 - 2, y)                                  # logits: AUC fine, log loss undefined
    with pytest.raises(ValueError, match="outside \\[0, 1\\]"):
        m.compute()
    assert abs(roc_auc(p * 4 - 2, y) - roc_auc_score(y.cpu().numpy(), p.cpu().numpy())) <= 1e-12
    m = BinaryMetrics(10, DEV)
    m.update(p, y)
    m.update(p, y)
    with pytest.raises(ValueError, match="capacity"):
        m.compute()
    m.reset()
    m.update(p, y)
    assert m.compute()["n"] == 8


def test_overflow_writes_nothing_past_capacity():
    lib = _lib.load()
    cap, B = 10, 16
    buf_s = torch.full((2 * cap,), -7.0, device=DEV)
    buf_y = torch.full((2 * cap,), -7.0, device=DEV)
    buf_g = torch.full((2 * cap,), -7, dtype=torch.int64, device=DEV)
    state = torch.zeros(3, dtype=torch.int64, device=DEV)
    s = torch.rand(B, device=DEV)
    y = (torch.arange(B, device=DEV) % 2).float()
    g = torch.arange(B, device=DEV)
    for _ in range(2):
        _lib.check(lib.rk_metrics_append(s.data_ptr(), y.data_ptr(), g.data_ptr(), B, buf_s.data_ptr(),
                                         buf_y.data_ptr(), buf_g.data_ptr(), cap, 100, state.data_ptr(),
                                         state.data_ptr() + 16, _lib.stream_ptr()), "rk_metrics_append")
    st = state.cpu()
    assert int(st[0]) == cap and int(st[1]) == 0 and int(st[2]) & _lib.METRICS_OVERFLOW
    assert torch.equal(buf_s[:cap], s[:cap]) and torch.equal(buf_g[:cap], g[:cap])
    assert bool((buf_s[cap:] == -7.0).all()) and bool((buf_y[cap:] == -7.0).all()) and bool((buf_g[cap:] == -7).all())
    assert ctypes.sizeof(_lib.RkMetricsResult) == 56


def test_dcn_evaluation_end_to_end(wechat_vocab_dir):
    torch.manual_seed(0)
    model = rank_b200.DCNModel(wechat_vocab_dir, hidden_units=[64, 32], num_cross_layer=3).to(DEV).eval()
    users = rank_b200.table_heights(wechat_vocab_dir, ["userid"])["userid"]
    B, steps = 4096, 5
    metrics = BinaryMetrics(B * steps, DEV, num_groups=users)
    probs, labels, uids = [], [], []
    with torch.no_grad():
        for step in range(steps):
            batch = synthetic.to_device(synthetic.side_batch(B, seed=100 + step), DEV)
            batch["label"] = (torch.rand(B, device=DEV) < 0.3).float()   # enough positives per user to matter
            prob = model(batch["dense"], batch["category"])[0]
            metrics.update(prob, batch["label"], batch["category"]["userid"])
            probs.append(prob.squeeze(1).cpu())
            labels.append(batch["label"].cpu())
            uids.append(batch["category"]["userid"].cpu())
    out = metrics.compute()
    p, y, u = torch.cat(probs).numpy(), torch.cat(labels).numpy(), torch.cat(uids).numpy()
    assert out["n"] == B * steps
    assert abs(out["auc"] - roc_auc_score(y, p)) <= 1e-12
    assert abs(out["uauc"] - sklearn_uauc(p, y, u)) <= 1e-12
    expect = F.binary_cross_entropy(torch.from_numpy(p).double(), torch.from_numpy(y).double()).item()
    assert abs(out["logloss"] - expect) <= 1e-12 * expect
    assert out["accuracy"] == accuracy_score(y, p > 0.5)
