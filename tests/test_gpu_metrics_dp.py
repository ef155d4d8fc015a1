"""BinaryMetrics.all_gather / rk_metrics_merge on the GPU: simulated worlds of 1..8 ranks on one device against
the numpy restatement (tests/test_metrics_dp.py), against one BinaryMetrics fed every rank's batches and against
sklearn; every rank's errors reach the merged compute(); a world-1 NCCL group, eager and graph-captured; and
two NCCL ranks evaluating a DCN model on their DeviceWechat shards (where two GPUs are present)."""
import os
import queue
import socket
import traceback

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
from sklearn.metrics import roc_auc_score

import rank_b200
from rank_b200 import _lib
from rank_b200.metrics import BinaryMetrics
from metrics_oracle import host_auc, sklearn_uauc, zipf_users
from test_metrics_dp import merge_reference

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
USERS = 19627          # the userid table of the WeChat vocabulary (19 626 lines + row 0)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _rank_batches(rng, world, cap, users, num_users):
    """Per rank, a list of (score, label, group) batches: random batch counts and sizes, rank 0 empty when there
    are several, the last rank filled to exactly `cap`.  Users are drawn from `users` ids for every rank alike,
    so each user's rows are spread over the ranks."""
    out = []
    for r in range(world):
        if world > 1 and r == 0:
            out.append([])
            continue
        total = cap if r == world - 1 else int(rng.integers(1, cap + 1))
        cuts = np.sort(rng.choice(np.arange(1, total), size=min(int(rng.integers(0, 6)), total - 1), replace=False))
        sizes = np.diff(np.concatenate([[0], cuts, [total]]))
        batches = []
        for b in sizes:
            g = zipf_users(rng, b, users) if users < num_users else rng.integers(0, num_users, b)
            batches.append((np.round(rng.random(b), 3).astype(np.float32),
                            (rng.random(b) < 0.3).astype(np.float32), g.astype(np.int64)))
        out.append(batches)
    return out


def _fed(batches, cap, num_groups):
    m = BinaryMetrics(cap, DEV, num_groups)
    for s, y, g in batches:
        m.update(torch.from_numpy(s).to(DEV), torch.from_numpy(y).to(DEV),
                 None if num_groups is None else torch.from_numpy(g).to(DEV))
    return m


def _merge(ranks, cap):
    """Stack the ranks' buffers as an all-gather lays them out and merge them with the entry point directly;
    the merged buffers are pre-filled with what merge_reference leaves past the count."""
    world, groups = len(ranks), ranks[0].groups is not None
    num_groups = ranks[0].num_groups
    merged = BinaryMetrics(world * cap, DEV, num_groups)
    merged.scores.fill_(float("nan"))
    merged.labels.fill_(float("nan"))
    if groups:
        merged.groups.fill_(-1)
    merged._state.fill_(-5)
    score_g = torch.cat([m.scores for m in ranks])
    label_g = torch.cat([m.labels for m in ranks])
    group_g = torch.cat([m.groups for m in ranks]) if groups else None
    state_g = torch.cat([m._state for m in ranks])
    _lib.check(_lib.load().rk_metrics_merge(
        score_g.data_ptr(), label_g.data_ptr(), _lib.ptr(group_g), state_g.data_ptr(), world, cap,
        merged.scores.data_ptr(), merged.labels.data_ptr(), _lib.ptr(merged.groups), merged._state.data_ptr(),
        _lib.stream_ptr()), "rk_metrics_merge")
    host = [t.cpu().numpy() if t is not None else None for t in (score_g, label_g, group_g, state_g)]
    return merged, merge_reference(*host, world, cap)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint8)


@pytest.mark.parametrize("world", [1, 2, 3, 8])
@pytest.mark.parametrize("users", [200, USERS])
def test_simulated_world_equals_one_rank_fed_every_batch(world, users):
    cap = 3000
    rng = np.random.default_rng(world * 100 + users)
    per_rank = _rank_batches(rng, world, cap, users, USERS)
    ranks = [_fed(b, cap, USERS) for b in per_rank]
    merged, (s, y, g, st) = _merge(ranks, cap)
    assert np.array_equal(merged._state.cpu().numpy(), st)
    assert _bits(merged.scores.cpu().numpy()).tobytes() == _bits(s).tobytes()
    assert _bits(merged.labels.cpu().numpy()).tobytes() == _bits(y).tobytes()
    assert np.array_equal(merged.groups.cpu().numpy(), g)

    every = [b for batches in per_rank for b in batches]                  # rank-major
    one = _fed(every, world * cap, USERS)
    out = merged.compute()
    assert out == one.compute()                                           # every field, bit for bit
    assert out["n"] == sum(len(b[0]) for b in every)
    ss, yy, gg = (np.concatenate([b[i] for b in every]) for i in range(3))
    assert out["auc"] == host_auc(ss, yy)
    assert abs(out["auc"] - roc_auc_score(yy, ss)) <= 1e-12
    assert abs(out["uauc"] - sklearn_uauc(ss, yy, gg)) <= 1e-12
    if world > 1 and users == 200:                                        # users really are split over ranks
        seen = [set(np.concatenate([b[2] for b in batches])) for batches in per_rank if batches]
        assert len(set.intersection(*seen)) > 50


def test_without_groups_and_without_a_process_group():
    assert not dist.is_initialized()
    rng = np.random.default_rng(3)
    per_rank = _rank_batches(rng, 3, 500, USERS, USERS)
    ranks = [_fed(b, 500, None) for b in per_rank]
    merged, (s, y, g, st) = _merge(ranks, 500)
    assert g is None and merged.groups is None
    assert np.array_equal(merged._state.cpu().numpy(), st)
    assert _bits(merged.scores.cpu().numpy()).tobytes() == _bits(s).tobytes()
    assert merged.compute() == _fed([b for x in per_rank for b in x], 1500, None).compute()
    m = ranks[-1]
    alone = m.all_gather()                                                # world 1: this process only
    assert alone.capacity == m.capacity and alone.compute() == m.compute()
    assert m.all_gather() is alone


def _messages(m):
    with pytest.raises(ValueError) as e:
        m.compute()
    return str(e.value)


@pytest.mark.parametrize("fault", ["nan", "label", "group", "overflow"])
def test_an_error_on_one_rank_reaches_the_merged_compute(fault):
    cap, world = 400, 3
    rng = np.random.default_rng(9)
    per_rank = _rank_batches(rng, world, cap, USERS, USERS)
    ranks = [_fed(b, cap, USERS) for b in per_rank]
    m = ranks[1] = BinaryMetrics(cap, DEV, USERS)                         # the faulty rank, between the others
    p = torch.linspace(0.1, 0.9, 8, device=DEV)
    y = (torch.arange(8, device=DEV) % 2).float()
    g = torch.arange(8, device=DEV)
    if fault == "nan":
        m.update(torch.where(y > 0, p, torch.full_like(p, float("nan"))), y, g)
    elif fault == "label":
        m.update(p, y * 2, g)
    elif fault == "group":
        m.update(p, y, g + USERS - 4)
    else:
        m.update(torch.rand(cap, device=DEV), (torch.rand(cap, device=DEV) < 0.5).float(),
                 torch.zeros(cap, dtype=torch.int64, device=DEV))
        m.update(p, y, g)                                                 # 8 rows past capacity
    want = _messages(m)
    merged, _ = _merge(ranks, cap)
    got = _messages(merged)
    if fault == "overflow":                                               # the message names each one's capacity
        assert want.startswith("more than capacity") and got.startswith("more than capacity")
    else:
        assert got == want
    healthy, _ = _merge([ranks[0], ranks[2]], cap)
    healthy.compute()                                                     # the other ranks alone are fine


@pytest.fixture
def single_rank_nccl():
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{_free_port()}", rank=0, world_size=1,
                            device_id=DEV)
    yield
    dist.destroy_process_group()


def test_all_gather_over_a_world1_nccl_group_eager_and_captured(single_rank_nccl):
    B, cap = 4096, 4096 * 8
    rng = np.random.default_rng(12)
    batches = [(rng.random(B).astype(np.float32), (rng.random(B) < 0.1).astype(np.float32),
                rng.integers(0, USERS, B).astype(np.int64)) for _ in range(6)]
    m = BinaryMetrics(cap, DEV, USERS)
    st = torch.zeros(B, 1, device=DEV)
    yt = torch.zeros(B, device=DEV)
    gt = torch.zeros(B, dtype=torch.int64, device=DEV)

    def load(k):
        s, y, g = batches[k]
        st.copy_(torch.from_numpy(s).view(B, 1))
        yt.copy_(torch.from_numpy(y))
        gt.copy_(torch.from_numpy(g))

    for k in range(2):
        load(k)
        m.update(st, yt, gt)
    merged = m.all_gather()                                               # eager first call
    assert merged.capacity == cap and merged.compute() == m.compute()

    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):                                         # the last evaluation step + the gather
        m.update(st, yt, gt)
        m.all_gather()
    for k in range(2, 6):
        load(k)
        graph.replay()
        captured = merged.compute()
        assert captured["n"] == (k + 1) * B
        assert captured == m.compute()
    assert m.all_gather() is merged and merged.compute() == captured      # eager again: the same result
    ref = BinaryMetrics(cap, DEV, USERS)
    for s, y, g in batches:
        ref.update(torch.from_numpy(s).to(DEV), torch.from_numpy(y).to(DEV), torch.from_numpy(g).to(DEV))
    assert captured == ref.compute()


def _dp_worker(rank, world, port, vocab_dir, out):
    """One data-parallel rank: a DCN model evaluated on this rank's shard of every batch of a 3000-row frame
    (5 full batches of 512 and a 440-row tail), then all_gather().compute(); then a mismatched capacity."""
    try:
        from rank_b200.loader import EncodedWechat
        from test_gpu_device_data import _random_frame
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        torch.cuda.set_device(rank)
        dev = torch.device("cuda", rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        torch.manual_seed(0)
        model = rank_b200.DCNModel(vocab_dir, hidden_units=[64, 32], num_cross_layer=3).to(dev).eval()
        users = rank_b200.table_heights(vocab_dir, ["userid"])["userid"]
        data = EncodedWechat(_random_frame(3000, 11), vocab_dir, "dcn").to_device(dev)
        B = 512
        feed = data.feed(B, rank=rank, world=world)
        metrics = BinaryMetrics(len(data) // world, dev, num_groups=users)
        kept = []

        def evaluate(b):
            prob = model(b["dense"], b["category"])[0]
            metrics.update(prob, b["label"], b["category"]["userid"])
            kept.append((prob.reshape(-1).cpu().numpy(), b["label"].cpu().numpy(),
                         b["category"]["userid"].cpu().numpy()))

        with torch.no_grad():
            feed.start_epoch(shuffle=True, generator=torch.Generator().manual_seed(3))
            for _ in range(len(feed)):
                evaluate(feed.next())
            evaluate(feed.tail())
        feed.check()
        result = metrics.all_gather().compute()
        try:
            BinaryMetrics(100 + rank, dev, users).all_gather()
            mismatch = None
        except ValueError as e:
            mismatch = str(e)
        out.put((rank, result, mismatch, [np.concatenate([k[i] for k in kept]) for i in range(3)]))
        dist.barrier()
        dist.destroy_process_group()
    except BaseException:
        out.put((rank, "error", traceback.format_exc(), None))
        raise


def test_two_ranks_over_nccl_equal_one_process(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from test_gpu_device_data import LINES, _random_frame
    from rank_b200.loader import EncodedWechat
    vocab_dir = rank_b200.write_vocab_dir(str(tmp_path / "vocab"), LINES) + "/"
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, vocab_dir, out)) for r in range(2)]
    try:
        for p in procs:
            p.start()
        results = {}
        while len(results) < 2:
            try:
                rank, result, mismatch, rows = out.get(timeout=10)
            except queue.Empty:
                assert all(p.exitcode in (None, 0) for p in procs), [p.exitcode for p in procs]
                continue
            assert result != "error", mismatch
            results[rank] = (result, mismatch, rows)
        for p in procs:
            p.join(120)
            assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
                p.join(30)
    (r0, m0, rows0), (r1, m1, rows1) = results[0], results[1]
    assert r0 == r1                                                       # identical on both ranks
    assert m0 is not None and m0 == m1 and "differ" in m0                 # the same error on both ranks
    p, y, u = (np.concatenate([rows0[i], rows1[i]]) for i in range(3))
    enc = EncodedWechat(_random_frame(3000, 11), vocab_dir, "dcn")
    assert r0["n"] == len(enc) == len(p)                                  # every row of the frame, once
    assert np.array_equal(np.sort(u), np.sort(enc.category["userid"]))
    assert np.array_equal(np.sort(y), np.sort(enc.label))
    users = rank_b200.table_heights(vocab_dir, ["userid"])["userid"]
    one = BinaryMetrics(len(p), DEV, users)                               # one process, rank-major order
    one.update(torch.from_numpy(p).to(DEV), torch.from_numpy(y).to(DEV), torch.from_numpy(u).to(DEV))
    assert one.compute() == r0
    perm = np.random.default_rng(0).permutation(len(p))                   # one process, any order
    shuffled = BinaryMetrics(len(p), DEV, users)
    shuffled.update(*(torch.from_numpy(a[perm]).to(DEV) for a in (p, y, u)))
    s = shuffled.compute()
    assert (s["n"], s["auc"], s["uauc"], s["accuracy"]) == (r0["n"], r0["auc"], r0["uauc"], r0["accuracy"])
    assert abs(s["logloss"] - r0["logloss"]) <= 1e-12 * r0["logloss"]
    assert abs(r0["auc"] - roc_auc_score(y, p)) <= 1e-12
    assert abs(r0["uauc"] - sklearn_uauc(p, y, u)) <= 1e-12
