"""rank_b200.DeviceWechat / BatchFeed on the GPU: every batch gathered by rk_batch_gather equals the host
loader's batch (EncodedWechat.batch + parallel.shard_batch) bit for bit; the feed equals PackedBatch.fill of
the host batch padded to seq_width, also when replayed from a CUDA graph; the status bits; and DIN training
fed from the device is bit-identical to training fed from the host."""
import numpy as np
import pandas as pd
import pytest
import torch
import torch.nn.functional as F

import rank_b200
from rank_b200.loader import DIN_SEQ, KINDS, EncodedWechat
from rank_b200.parallel import shard_batch
from rank_b200.staging import PackedBatch, _leaves
import loader_cases
from test_loader import _same

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
LINES = {"userid": 300, "feedid": 500, "device": 2, "authorid": 120, "bgm_song_id": 90, "bgm_singer_id": 70,
         "manual_tag_list": 30}
SPLITS = [(False, 0, 1), (True, 0, 1), (False, 1, 2), (True, 2, 3)]      # (drop_last, rank, world)


def _cpu(b):
    return {k: _cpu(v) for k, v in b.items()} if isinstance(b, dict) else b.cpu()


def _pad(batch, width):
    """The host batch with DIN's history zero-padded to `width` (what the feed writes)."""
    if "sequence" not in batch:
        return batch
    out = dict(batch)
    seq = batch["sequence"][DIN_SEQ]
    out["sequence"] = {DIN_SEQ: F.pad(seq, (0, width - seq.shape[1])),
                       DIN_SEQ + "_length": batch["sequence"][DIN_SEQ + "_length"]}
    return out


def _random_frame(n, seed):
    """WeChat-shaped frame over the LINES vocabularies: 30 % empty histories, lengths 1..50, some unknown ids."""
    rng = np.random.default_rng(seed)

    def ids(col, k=n):
        return [f"{col}_{v}" for v in rng.integers(1, LINES[col] + 20, k)]

    df = pd.DataFrame({c: ids(c) for c in ("userid", "feedid", "authorid", "bgm_song_id", "bgm_singer_id",
                                            "manual_tag_list")})
    df["device"] = [f"device_{v}" for v in rng.integers(1, 3, n)]
    df["read_comment"] = (rng.random(n) < 0.3).astype(np.int64)
    for c in loader_cases.DENSE:
        df[c] = np.log1p(rng.poisson(3.0, n)).astype(np.float64)
    lens = rng.integers(1, 51, n) * (rng.random(n) >= 0.3)
    df[DIN_SEQ] = [ids("feedid", k) for k in lens]
    return df


@pytest.fixture(scope="module")
def vocab(tmp_path_factory):
    return {"cases": loader_cases.write_vocab(str(tmp_path_factory.mktemp("vocab_cases"))) + "/",
            "random": rank_b200.write_vocab_dir(str(tmp_path_factory.mktemp("vocab_random")), LINES) + "/"}


def _encoded(kind, frame, vocab):
    if frame == "random":
        return EncodedWechat(_random_frame(3000, 11), vocab["random"], kind, max_seq_length=20)
    return EncodedWechat(loader_cases.make_frame(frame), vocab["cases"], kind, max_seq_length=5)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("frame", ["string", "list"])
@pytest.mark.parametrize("shuffle", [False, True])
@pytest.mark.parametrize("size", ["1", "7", "n-1", "n", "n+5"])
def test_batches_equal_the_host_loader(kind, frame, shuffle, size, vocab):
    enc = _encoded(kind, frame, vocab)
    data = enc.to_device(DEV)
    n = len(enc)
    B = {"1": 1, "7": 7, "n-1": n - 1, "n": n, "n+5": n + 5}[size]
    for drop_last, rank, world in SPLITS:
        gen = lambda: torch.Generator().manual_seed(19)
        want = list(enc.batches(B, shuffle=shuffle, generator=gen(), drop_last=drop_last))
        got = list(data.batches(B, shuffle=shuffle, generator=gen(), drop_last=drop_last, rank=rank, world=world))
        assert len(got) == len(want)
        for i, (g, w) in enumerate(zip(got, want)):
            _same(_cpu(g), shard_batch(w, rank, world), f"{kind}[{i}] rank {rank}/{world}")


@pytest.mark.parametrize("kind", KINDS)
def test_batches_of_a_large_frame(kind, vocab):
    enc = _encoded(kind, "random", vocab)
    data = enc.to_device(DEV)
    for B, rank, world in ((256, 0, 1), (500, 1, 4)):
        order = torch.randperm(len(enc), generator=torch.Generator().manual_seed(4)).numpy()
        got = data.batches(B, shuffle=True, generator=torch.Generator().manual_seed(4), rank=rank, world=world)
        for i, g in enumerate(got):
            _same(_cpu(g), shard_batch(enc.batch(order[i * B:(i + 1) * B]), rank, world), f"{kind}[{i}]")


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("rank,world", [(0, 1), (1, 2)])
def test_feed_equals_packed_fill_of_the_padded_host_batch(kind, rank, world, vocab):
    enc = _encoded(kind, "random", vocab)
    data = enc.to_device(DEV, seq_width=60 if kind == "din" else None)
    B = 256
    order = torch.randperm(len(enc), generator=torch.Generator().manual_seed(8)).numpy()
    first = _pad(shard_batch(enc.batch(order[:B]), rank, world), data.seq_width)
    packed = PackedBatch.like(first, DEV)
    feed = data.feed(B, rank=rank, world=world, packed=packed)
    plain = data.feed(B, rank=rank, world=world)
    assert len(feed) == len(enc) // B
    ref = PackedBatch.like(first, DEV)
    for f in (feed, plain):
        f.start_epoch(shuffle=True, generator=torch.Generator().manual_seed(8))
    for i in range(len(feed)):
        ref.fill(_pad(shard_batch(enc.batch(order[i * B:(i + 1) * B]), rank, world), data.seq_width))
        views = feed.next()
        assert views is packed.device_views
        _same(_cpu(plain.next()), _cpu(views))
        for (path, want), (_, have) in zip(_leaves(ref.host_views), _leaves(packed.device_views)):
            assert torch.equal(have.cpu().reshape(-1).view(torch.uint8), want.reshape(-1).view(torch.uint8)), path
    tail = feed.tail()
    _same(_cpu(tail), shard_batch(enc.batch(order[len(feed) * B:]), rank, world))
    feed.check()
    plain.check()


def test_feed_replayed_from_a_cuda_graph_over_two_epochs(vocab):
    enc = _encoded("din", "random", vocab)
    data = enc.to_device(DEV)
    B = 512
    graph_feed, eager_feed = data.feed(B), data.feed(B)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        views = graph_feed.next()
    gen_g, gen_e = torch.Generator().manual_seed(2), torch.Generator().manual_seed(2)
    for epoch in range(2):
        graph_feed.start_epoch(shuffle=True, generator=gen_g)
        eager_feed.start_epoch(shuffle=True, generator=gen_e)
        order = graph_feed._order_host.clone().numpy()
        for i in range(len(graph_feed)):
            g.replay()
            got = _cpu(views)
            _same(got, _cpu(eager_feed.next()), f"epoch {epoch} batch {i}")
            _same(got, _pad(enc.batch(order[i * B:(i + 1) * B]), data.seq_width), f"epoch {epoch} batch {i}")
        graph_feed.check()
        eager_feed.check()


def test_status_bits_are_raised_without_a_fault(vocab):
    enc = _encoded("din", "random", vocab)
    data = enc.to_device(DEV)
    B = 1024
    feed = data.feed(B)
    for _ in range(len(feed)):
        feed.next()
    before = _cpu(feed.views)
    feed.next()                                          # past the last full batch: writes nothing
    torch.cuda.synchronize()
    _same(_cpu(feed.views), before)
    with pytest.raises(IndexError, match="len"):
        feed.check()
    feed.check()                                         # the bits were cleared

    feed.start_epoch()
    feed.order[3] = len(enc) + 7                         # an order entry past the frame
    feed.order[4] = -1
    batch = _cpu(feed.next())
    with pytest.raises(IndexError, match="outside"):
        feed.check()
    for path, t in _leaves(batch):
        assert not t[3:5].any(), path                    # those rows are written as zeros

    feed.start_epoch()
    lens = np.diff(enc.seq_offsets)
    width = 3
    outs = data._outputs(B, width)                       # a width below the longest history, on the ABI directly
    data._gather(outs, feed.order, len(enc), feed.cursor, 0, B, width, feed.status)
    with pytest.raises(ValueError, match="longer"):
        feed.check()
    got = dict(outs)
    rows = np.arange(B)
    assert torch.equal(got[("sequence", DIN_SEQ + "_length")].cpu(), torch.from_numpy(np.minimum(lens[rows], width)))
    want = enc.batch(rows)["sequence"][DIN_SEQ]
    kept = min(width, want.shape[1])
    assert torch.equal(got[("sequence", DIN_SEQ)].cpu()[:, :kept], want[:, :kept])

    feed.start_epoch()                                   # and the feed still works
    _same(_cpu(feed.next()), _pad(enc.batch(np.arange(B)), data.seq_width))
    feed.check()
    torch.cuda.synchronize()


def _train(model, opt, batches, steps):
    losses = []
    for step in range(steps):
        b = batches(step)
        torch.manual_seed(1000 + step)                   # the per-call attention MLP draw (DIN/din.py:61-67)
        model.zero_grad(set_to_none=True)
        prob, _, l2 = model(b["dense"], b["category"], b["sequence"], b["target"])
        loss = F.binary_cross_entropy(prob.squeeze(1), b["label"]) + l2
        loss.backward()
        opt.step()
        losses.append(loss.detach().clone())
    return torch.stack(losses).cpu()


def test_din_training_fed_from_the_device_matches_the_host_path(vocab):
    enc = _encoded("din", "random", vocab)
    data = enc.to_device(DEV)
    B, steps = 128, 20
    models = []
    for _ in range(2):
        torch.manual_seed(0)
        m = rank_b200.DIN(vocab["random"], hidden_units=[64, 32], dropout_rate=0.0, use_softmax=False).to(DEV)
        m.activation_unit_precision = "bf16"
        m.train()
        models.append((m, rank_b200.Adam(m.parameters(), lr=1e-3)))
    assert len(enc) // B >= steps
    order = torch.randperm(len(enc), generator=torch.Generator().manual_seed(6)).numpy()

    def host(step):
        rows = order[step * B:(step + 1) * B]
        return {k: (v.to(DEV) if torch.is_tensor(v) else {c: t.to(DEV) for c, t in v.items()})
                for k, v in _pad(enc.batch(rows), data.seq_width).items()}

    feed = data.feed(B)
    feed.start_epoch(shuffle=True, generator=torch.Generator().manual_seed(6))
    l_host = _train(*models[0], host, steps)
    l_dev = _train(*models[1], lambda step: feed.next(), steps)
    feed.check()
    rank_b200.check_index_errors()
    assert torch.equal(l_host, l_dev), (l_host, l_dev)
    for (k, p), (_, q) in zip(models[0][0].named_parameters(), models[1][0].named_parameters()):
        assert torch.equal(p, q), k
