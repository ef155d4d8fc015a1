"""DeviceWechat.from_frame on the GPU: every device array equals that of EncodedWechat(...).to_device(...) bit for
bit, on the loader's synthetic frames and on a 10^6-row frame with edge-case histories, non-ASCII ids, a
10^6-line vocabulary and one exactly at the slot bound; and its batches and graph-captured feed equal those of
the host-encoded frame."""
import os

import numpy as np
import pytest
import torch

import rank_b200
from rank_b200.loader import DIN_SEQ, KINDS, EncodedWechat
import loader_cases
from test_gpu_device_data import LINES, _cpu, _random_frame
from test_loader import _same

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def _arrays(data):
    out = {path: src for path, src in data._leaves if src is not None}
    if data.kind == "din":
        out["seq_flat"], out["seq_offsets"] = data.seq_flat, data.seq_offsets
    return out


def assert_same_arrays(got, want):
    assert got.kind == want.kind and got.n == want.n and got.seq_width == want.seq_width
    assert [p for p, _ in got._leaves] == [p for p, _ in want._leaves]
    g, w = _arrays(got), _arrays(want)
    assert g.keys() == w.keys()
    for k in w:
        assert g[k].device == w[k].device and g[k].dtype == w[k].dtype and g[k].shape == w[k].shape, k
        assert torch.equal(g[k].reshape(-1).view(torch.uint8), w[k].reshape(-1).view(torch.uint8)), k
    if want.kind == "din":
        assert np.array_equal(got._seq_len, want._seq_len)


@pytest.fixture(scope="module")
def cases_vocab(tmp_path_factory):
    return loader_cases.write_vocab(str(tmp_path_factory.mktemp("vocab_cases"))) + "/"


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("history", ["string", "list"])
@pytest.mark.parametrize("max_seq_length", [0, 5, 50])
def test_from_frame_equals_the_host_encoding(kind, history, max_seq_length, cases_vocab):
    frame = loader_cases.make_frame(history)
    got = rank_b200.DeviceWechat.from_frame(frame, cases_vocab, kind, DEV, max_seq_length=max_seq_length)
    if kind == "bst" and max_seq_length == 0:
        # the host encoder indexes seq[:, 0] of a width-0 sequence and raises; the device path gives the empty
        # sequences and the zero lengths (min(1, 0)) that the reference's cut / pad produces
        with pytest.raises(IndexError):
            EncodedWechat(frame, cases_vocab, kind, max_seq_length=0)
        arrays = _arrays(got)
        assert arrays[("seq_feedid",)].shape == (len(frame), 0)
        assert not arrays[("seq_length",)].any()
        return
    want = EncodedWechat(frame, cases_vocab, kind, max_seq_length=max_seq_length).to_device(DEV)
    assert_same_arrays(got, want)
    assert got.encode_paths["device"] == "zeros" and got.encode_paths["userid"] == "strings"
    if kind == "din":
        assert got.encode_paths[DIN_SEQ] == ("split" if history == "string" else "lists")


def test_from_a_parquet_file(cases_vocab, tmp_path):
    path = str(tmp_path / "frame.parquet")
    loader_cases.make_frame("list").to_parquet(path)                  # histories come back as arrays
    for kind in ("din", "bst"):
        want = EncodedWechat(path, cases_vocab, kind, max_seq_length=5).to_device(DEV)
        got = rank_b200.DeviceWechat.from_frame(path, cases_vocab, kind, DEV, max_seq_length=5)
        assert_same_arrays(got, want)
    assert got.encode_paths["feedid"] == "strings"


BIG = 10 ** 6
AT_BOUND = 1 << 16          # userid keys: exactly n_slots / 2


def _big_vocab(path):
    """feedid: 10^6 lines, some non-ASCII, one empty line (the key '') and one duplicated line; userid: exactly
    at the slot bound; the rest as write_vocab_dir writes them."""
    lines = dict(LINES, feedid=BIG, userid=AT_BOUND)
    rank_b200.write_vocab_dir(path, lines)
    feed = [f"feedid_{i}" if i % 11 else f"фид_{i}_飞" for i in range(1, BIG + 1)]
    feed[500] = ""
    feed.append("feedid_7")                           # duplicated: keeps this last position
    with open(os.path.join(path, "feedid.txt"), "w", encoding="utf-8") as f:
        f.write("".join(x + "\n" for x in feed))
    return path + "/"


def _big_frame(seed=3):
    lines = dict(LINES, feedid=BIG, userid=AT_BOUND)
    df = _random_frame(BIG, seed)
    rng = np.random.default_rng(seed + 1)

    def fid(v):
        return f"фид_{v}_飞" if v % 11 == 0 else f"feedid_{v}"

    df["userid"] = [f"userid_{v}" for v in rng.integers(1, lines["userid"] + 20, BIG)]
    feeds = rng.integers(1, BIG + 20, BIG)
    df["feedid"] = [fid(v) for v in feeds]
    lens = rng.integers(1, 51, BIG) * (rng.random(BIG) >= 0.3)
    items = rng.integers(1, BIG + 20, int(lens.sum()))
    hist, at = [], 0
    for k in lens:
        hist.append(",".join(fid(v) for v in items[at:at + k]))
        at += k
    for i, h in zip(range(0, BIG, 9973), ["", "a,", ",,", ",feedid_3", "feedid_7,,фид_22_飞,"] * 200):
        hist[i] = h
    df[DIN_SEQ] = hist
    return df


@pytest.fixture(scope="module")
def big(tmp_path_factory):
    return _big_frame(), _big_vocab(str(tmp_path_factory.mktemp("vocab_big")))


@pytest.mark.parametrize("kind", ["din", "bst", "deepfm"])
def test_a_million_rows_with_edge_cases(kind, big):
    frame, vocab = big
    want = EncodedWechat(frame, vocab, kind, max_seq_length=20).to_device(DEV)
    got = rank_b200.DeviceWechat.from_frame(frame, vocab, kind, DEV, max_seq_length=20)
    assert_same_arrays(got, want)
    if kind == "din":
        assert got.encode_paths[DIN_SEQ] == "split"
        lens = got._seq_len[0:BIG:9973][:5]
        assert lens.tolist() == [1, 2, 3, 2, 4]       # '', 'a,', ',,', ',feedid_3', 'feedid_7,,фид_22_飞,'
        hits = got.seq_flat.cpu().numpy()
        assert (hits > 0).mean() > 0.9                # the probes found the keys, not only misses


def test_batches_and_a_graph_captured_feed_equal_the_host_encoded_frame(tmp_path):
    vocab = rank_b200.write_vocab_dir(str(tmp_path / "vocab"), LINES) + "/"
    frame = _random_frame(3000, 11)
    frame[DIN_SEQ] = [",".join(h) for h in frame[DIN_SEQ]]
    host = EncodedWechat(frame, vocab, "din").to_device(DEV)
    dev = rank_b200.DeviceWechat.from_frame(frame, vocab, "din", DEV)
    assert dev.encode_paths[DIN_SEQ] == "split"
    for B, rank, world in ((256, 0, 1), (500, 1, 2)):
        got = dev.batches(B, shuffle=True, generator=torch.Generator().manual_seed(5), rank=rank, world=world)
        want = host.batches(B, shuffle=True, generator=torch.Generator().manual_seed(5), rank=rank, world=world)
        for i, (g, w) in enumerate(zip(got, want)):
            _same(_cpu(g), _cpu(w), f"batch {i} rank {rank}/{world}")
    B = 512
    feeds = (dev.feed(B), host.feed(B))
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        views = feeds[0].next()
    gens = (torch.Generator().manual_seed(2), torch.Generator().manual_seed(2))
    for epoch in range(2):
        for f, gen in zip(feeds, gens):
            f.start_epoch(shuffle=True, generator=gen)
        for i in range(len(feeds[0])):
            g.replay()
            _same(_cpu(views), _cpu(feeds[1].next()), f"epoch {epoch} batch {i}")
        _same(_cpu(feeds[0].tail()), _cpu(feeds[1].tail()), f"epoch {epoch} tail")
        for f in feeds:
            f.check()
