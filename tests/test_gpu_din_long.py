"""DIN on histories wider than one 128-row tile (fp32 activation unit), and on batches with no history.

Against the oracle at the 1e-5 fp32 bar with the float64 arbiter of test_gpu_models.py; invariance of the fp32
kernels to padding a 128-wide batch past one tile; width 0; the index check past position 128; graph capture
and determinism; the device input path at width 300; and the tensor-core unit's refusal above 128."""
import numpy as np
import pandas as pd
import pytest
import torch
import torch.nn.functional as F

import rank_b200
from rank_b200 import _lib, synthetic
from rank_b200.loader import DIN_SEQ, EncodedWechat
from conftest import rel_err
from test_gpu_models import FP32_TOL, _pair, _run_both, compare
from test_gpu_device_data import LINES, _pad, _train
import loader_cases

pytestmark = pytest.mark.gpu
DEV = "cuda"
SEQ, SEQ_LEN = "his_read_comment_7d_seq", "his_read_comment_7d_seq_length"


def _with_lengths(batch, length):
    """The batch with new history lengths; positions past a length hold the padding id 0."""
    seq = batch["sequence"][SEQ]
    T = seq.shape[1]
    gen = torch.Generator().manual_seed(17)
    full = torch.where(seq > 0, seq, torch.randint(1, 1000, seq.shape, generator=gen))
    out = dict(batch)
    out["sequence"] = {SEQ: full * (torch.arange(T).expand_as(full) < length.unsqueeze(1)), SEQ_LEN: length}
    return out


def _padded(batch, T):
    out = dict(batch)
    seq = batch["sequence"][SEQ]
    out["sequence"] = {SEQ: F.pad(seq, (0, T - seq.shape[1])), SEQ_LEN: batch["sequence"][SEQ_LEN]}
    return out


@pytest.mark.parametrize("soft", [False, True])
@pytest.mark.parametrize("B,T", [(2048, 129), (1024, 200), (512, 1000), (64, 4096)])
def test_din_long_histories_vs_oracle(wechat_vocab_dir, B, T, soft):
    ours, ref = _pair("DIN", "OracleDIN", wechat_vocab_dir, dropout_rate=0.0, use_softmax=soft)
    compare(*_run_both(ours, ref, "DIN", synthetic.din_batch(B, T)))


@pytest.mark.parametrize("soft", [False, True])
def test_din_lengths_straddling_the_tile_edge(wechat_vocab_dir, soft):
    T = 300
    pattern = torch.tensor([0, 1, 127, 128, 129, 255, 256, 257, T])
    gen = torch.Generator().manual_seed(4)
    length = pattern.repeat(100)[torch.randperm(900, generator=gen)]
    ours, ref = _pair("DIN", "OracleDIN", wechat_vocab_dir, dropout_rate=0.0, use_softmax=soft)
    compare(*_run_both(ours, ref, "DIN", _with_lengths(synthetic.din_batch(900, T), length)))


@pytest.mark.parametrize("soft", [False, True])
def test_din_every_history_full(wechat_vocab_dir, soft):
    B, T = 256, 256
    ours, ref = _pair("DIN", "OracleDIN", wechat_vocab_dir, dropout_rate=0.0, use_softmax=soft)
    batch = _with_lengths(synthetic.din_batch(B, T), torch.full((B,), T, dtype=torch.int64))
    compare(*_run_both(ours, ref, "DIN", batch))


@pytest.mark.parametrize("soft", [False, True])
def test_din_width_zero_vs_oracle(wechat_vocab_dir, soft):
    B = 512
    batch = synthetic.din_batch(B, 1)
    batch["sequence"] = {SEQ: batch["sequence"][SEQ][:, :0].contiguous(), SEQ_LEN: torch.zeros(B, dtype=torch.int64)}
    ours, ref = _pair("DIN", "OracleDIN", wechat_vocab_dir, dropout_rate=0.0, use_softmax=soft)
    compare(*_run_both(ours, ref, "DIN", batch))


def test_din_attention_long_history():
    from oracle import interactions as X
    gen = torch.Generator().manual_seed(3)
    B, T, D = 200, 300, 16
    q = torch.randn(B, D, generator=gen, requires_grad=True)
    k = torch.randn(B, T, D, generator=gen, requires_grad=True)
    n = torch.randint(0, T + 1, (B,), generator=gen)
    n[:4] = torch.tensor([0, 128, 129, T])
    cot = torch.randn(B, D, generator=gen)
    for soft in (False, True):
        torch.manual_seed(5)
        net = torch.nn.Sequential(torch.nn.Linear(4 * D, 64), torch.nn.ReLU(), torch.nn.Linear(64, 32),
                                  torch.nn.ReLU(), torch.nn.Linear(32, 1))
        want = X.din_local_activation(q, k, n, tuple(p.detach() for p in net.parameters()), soft)
        q.grad = k.grad = None
        (want * cot).sum().backward()
        qa, ka = q.detach().to(DEV).requires_grad_(), k.detach().to(DEV).requires_grad_()
        torch.manual_seed(5)
        got = rank_b200.din_attention(qa, ka, n.to(DEV), soft)
        (got * cot.to(DEV)).sum().backward()
        assert rel_err(got, want) <= FP32_TOL, soft
        assert rel_err(qa.grad, q.grad) <= FP32_TOL and rel_err(ka.grad, k.grad) <= FP32_TOL, soft


def _step(model, batch, cot, seed=5):
    """Forward + backward of one batch: (logit, l2, {parameter: gradient})."""
    model.zero_grad(set_to_none=True)
    torch.manual_seed(seed)                  # the per-call attention MLP draw
    _, logit, l2 = model(batch["dense"], batch["category"], batch["sequence"], batch["target"])
    ((logit * cot).sum() + l2).backward()
    return logit.detach().clone(), l2.detach().clone(), {k: p.grad.clone() for k, p in model.named_parameters()
                                                         if p.grad is not None}


@pytest.mark.parametrize("soft", [False, True])
def test_padding_past_128_changes_nothing(wechat_vocab_dir, soft):
    ours, _ = _pair("DIN", "OracleDIN", wechat_vocab_dir, dropout_rate=0.0, use_softmax=soft)
    batch = synthetic.din_batch(1024, 128)
    cot = torch.randn(1024, 1, generator=torch.Generator().manual_seed(2), device="cpu").to(DEV) / 1024
    base = _step(ours, synthetic.to_device(batch, DEV), cot)
    for T in (129, 300):
        got = _step(ours, synthetic.to_device(_padded(batch, T), DEV), cot)
        assert rel_err(got[0], base[0]) <= FP32_TOL and rel_err(got[1], base[1]) <= FP32_TOL, T
        assert set(got[2]) == set(base[2])
        for k in base[2]:
            assert rel_err(got[2][k], base[2][k]) <= FP32_TOL, (T, k)
    rank_b200.check_index_errors()


def test_out_of_range_history_id_past_128_is_reported(wechat_vocab_dir):
    ours, _ = _pair("DIN", "OracleDIN", wechat_vocab_dir, dropout_rate=0.0)
    batch = synthetic.din_batch(64, 300)
    length = batch["sequence"][SEQ_LEN].clone()
    length[3] = 280
    batch = _with_lengths(batch, length)
    batch["sequence"][SEQ][3, 200] = 10 ** 9
    batch = synthetic.to_device(batch, DEV)
    rank_b200.check_index_errors()
    with torch.no_grad():                    # the forward kernel alone (no gradient plan)
        ours(batch["dense"], batch["category"], batch["sequence"], batch["target"])
    with pytest.raises(IndexError):
        rank_b200.check_index_errors()
    rank_b200.check_index_errors()           # the flag was cleared


def test_training_step_at_300_from_a_cuda_graph(wechat_vocab_dir):
    B, T = 512, 300
    ours, _ = _pair("DIN", "OracleDIN", wechat_vocab_dir, hidden_units=[64, 32], dropout_rate=0.0,
                    use_softmax=True)
    ours.train()
    ours.draw_ephemeral()
    ours.ephemeral_frozen = True            # one fixed draw: a graph cannot hold the CPU-generator draws
    batch = synthetic.to_device(synthetic.din_batch(B, T), DEV)
    cot = torch.randn(B, 1, generator=torch.Generator().manual_seed(2)).to(DEV) / B
    params = [p for p in ours.parameters()]
    state = [p.detach().clone() for p in params]

    def body():
        _, logit, l2 = ours(batch["dense"], batch["category"], batch["sequence"], batch["target"])
        loss = (logit * cot).sum() + l2
        loss.backward()
        return loss

    ours.zero_grad(set_to_none=True)
    eager_loss = body().detach().clone()
    eager = [p.grad.clone() for p in params]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            ours.zero_grad(set_to_none=True)
            body()
    torch.cuda.current_stream().wait_stream(side)
    ours.zero_grad(set_to_none=True)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        loss = body()
    replays = []
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        replays.append((loss.clone(), [p.grad.clone() for p in params]))
    rank_b200.check_index_errors()
    for p, s in zip(params, state):
        assert torch.equal(p.detach(), s)
    assert torch.equal(replays[0][0], replays[1][0])
    for a, b in zip(replays[0][1], replays[1][1]):
        assert torch.equal(a, b)
    assert rel_err(replays[0][0], eager_loss) <= FP32_TOL
    for k, (a, b) in enumerate(zip(replays[0][1], eager)):
        assert rel_err(a, b) <= FP32_TOL, k


def _long_frame(n, seed, longest):
    """WeChat-shaped frame over the LINES vocabularies with histories of 0..`longest` ids."""
    rng = np.random.default_rng(seed)

    def ids(col, k=n):
        return [f"{col}_{v}" for v in rng.integers(1, LINES[col] + 20, k)]

    df = pd.DataFrame({c: ids(c) for c in ("userid", "feedid", "authorid", "bgm_song_id", "bgm_singer_id",
                                            "manual_tag_list")})
    df["device"] = [f"device_{v}" for v in rng.integers(1, 3, n)]
    df["read_comment"] = (rng.random(n) < 0.3).astype(np.int64)
    for c in loader_cases.DENSE:
        df[c] = np.log1p(rng.poisson(3.0, n)).astype(np.float64)
    lens = rng.integers(1, longest + 1, n) * (rng.random(n) >= 0.3) if longest else np.zeros(n, np.int64)
    if longest:
        lens[0] = longest
    df[DIN_SEQ] = [ids("feedid", k) for k in lens]
    return df


@pytest.fixture(scope="module")
def vocab(tmp_path_factory):
    return rank_b200.write_vocab_dir(str(tmp_path_factory.mktemp("vocab_long")), LINES) + "/"


def _models(vocab, n=2):
    out = []
    for _ in range(n):
        torch.manual_seed(0)
        m = rank_b200.DIN(vocab, hidden_units=[64, 32], dropout_rate=0.0, use_softmax=True).to(DEV)
        m.train()
        out.append((m, rank_b200.Adam(m.parameters(), lr=1e-3)))
    return out


def test_feed_at_width_300_trains_as_the_host_path(vocab):
    enc = EncodedWechat(_long_frame(3000, 12, 300), vocab, "din")
    data = enc.to_device(DEV, seq_width=300)
    B, steps = 128, 20
    models = _models(vocab)
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
    assert torch.isfinite(l_host).all()
    assert torch.equal(l_host, l_dev), (l_host, l_dev)
    for (k, p), (_, q) in zip(models[0][0].named_parameters(), models[1][0].named_parameters()):
        assert torch.equal(p, q), k


def test_batches_with_no_history_train(vocab):
    enc = EncodedWechat(_long_frame(600, 13, 0), vocab, "din")
    data = enc.to_device(DEV)
    B = 128
    dev_batches = list(data.batches(B))
    assert dev_batches[0]["sequence"][DIN_SEQ].shape == (B, 0)
    models = _models(vocab)

    def host(step):
        rows = np.arange(step * B, (step + 1) * B)
        return {k: (v.to(DEV) if torch.is_tensor(v) else {c: t.to(DEV) for c, t in v.items()})
                for k, v in enc.batch(rows).items()}

    l_host = _train(*models[0], host, 3)
    l_dev = _train(*models[1], lambda step: dev_batches[step], 3)
    rank_b200.check_index_errors()
    assert torch.isfinite(l_dev).all()
    assert torch.equal(l_host, l_dev), (l_host, l_dev)
    before = {k: p.detach().clone() for k, p in models[1][0].named_parameters()}
    _train(*models[1], lambda step: dev_batches[step], 1)
    assert any(not torch.equal(before[k], p) for k, p in models[1][0].named_parameters())


def test_tensor_core_unit_refuses_129_positions_before_any_launch(wechat_vocab_dir):
    ours, _ = _pair("DIN", "OracleDIN", wechat_vocab_dir, dropout_rate=0.0)
    ours.activation_unit_precision = "bf16"
    batch = synthetic.to_device(synthetic.din_batch(256, 129), DEV)
    lib = _lib.load()
    torch.cuda.synchronize()
    launches = lib.rk_launch_count()
    with pytest.raises(_lib.RankB200Error, match="fp32"):
        ours(batch["dense"], batch["category"], batch["sequence"], batch["target"])
    assert lib.rk_launch_count() == launches
    ours.activation_unit_precision = "fp32"
    ours(batch["dense"], batch["category"], batch["sequence"], batch["target"])
    assert lib.rk_launch_count() > launches
