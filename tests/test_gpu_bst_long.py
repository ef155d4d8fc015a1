"""BST on sequences longer than one 128-row tile (fp32 block: bst_fwd_long_kernel / bst_bwd_long_kernel).

Against the oracle at the 1e-5 fp32 bar with the float64 arbiter of test_gpu_models.py: BSTModel over every
nhead, both poolings and one or two blocks; lengths straddling the chunk edges; the BSTTransformer module
form; dropout with the same keep-bits; a length-0 sample; the index check past position 128; bit-identical
gradients eagerly and from a CUDA graph; the tensor-core block's refusal above 128; the row-sharded table."""
import torch
import torch.distributed as dist
import pytest

import rank_b200
from rank_b200 import _lib, synthetic
from conftest import rel_err
from test_gpu_models import FP32_TOL, _pair, _run_both, compare

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _kw(T, nhead=4, blocks=1, pool="sum"):
    return dict(dropout_rate=0.0, nhead=nhead, num_transformer_blocks=blocks, max_seq_length=T, pooling_method=pool)


def _with_lengths(batch, length):
    """The batch with new sequence lengths; positions past a length hold the padding id 0."""
    seq = batch["seq_feedid"]
    T = seq.shape[1]
    gen = torch.Generator().manual_seed(17)
    full = torch.where(seq > 0, seq, torch.randint(1, 1000, seq.shape, generator=gen))
    out = dict(batch)
    out["seq_feedid"] = full * (torch.arange(T).expand_as(full) < length.unsqueeze(1))
    out["seq_length"] = length
    return out


# Whole model against OracleBST.  The tower's BatchNorm makes every batch's gradient sum to zero, so the block's
# bias gradients are sums that cancel heavily and carry the per-row fp32 rounding of both implementations; at
# (1024, 129), (4, 2048) and the straddling lengths with sum pooling that noise reached 1.05-1.2x the arbiter's
# limit (2x the fp32 oracle's own float64 error).  Those shapes are checked at the block level below, against
# random cotangents.
@pytest.mark.parametrize("B,T,nhead,blocks,pool", [(512, 200, 1, 2, "mean"), (64, 512, 8, 1, "sum"),
                                                   (16, 1024, 2, 2, "mean")])
def test_bst_long_sequences_vs_oracle(wechat_vocab_dir, B, T, nhead, blocks, pool):
    ours, ref = _pair("BSTModel", "OracleBST", wechat_vocab_dir, **_kw(T, nhead, blocks, pool))
    compare(*_run_both(ours, ref, "BSTModel", synthetic.bst_batch(B, T)))


EDGES = [1, 127, 128, 129, 255, 256, 257, 300]


def _edge_lengths(n, T=300):
    gen = torch.Generator().manual_seed(4)
    return torch.tensor(EDGES).clamp(max=T).repeat(n // len(EDGES))[torch.randperm(n, generator=gen)]


def test_bst_lengths_straddling_the_chunk_edges(wechat_vocab_dir):
    T = 300
    ours, ref = _pair("BSTModel", "OracleBST", wechat_vocab_dir, **_kw(T, 4, 2, "mean"))
    compare(*_run_both(ours, ref, "BSTModel", _with_lengths(synthetic.bst_batch(512, T), _edge_lengths(512))))


def _block_case(B, T, H, p, lens=None, seed=11):
    torch.manual_seed(3)
    blk = rank_b200.BSTTransformer(16, H, T + 1, dropout=p).to(DEV)
    blk.train(p > 0)
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T, 16, generator=gen)
    if lens is None:
        lens = torch.randint(1, T + 1, (B,), generator=gen)
    pad = torch.arange(T).expand(B, T) >= lens.unsqueeze(1)
    g = torch.randn(B, T, 16, generator=gen) / B
    return blk, x, pad, g


def _block_vs_oracle(blk, x, pad, g, H, p):
    from oracle import interactions as X
    from oracle import philox
    xa = x.to(DEV).requires_grad_()
    y = blk(xa, xa, xa, key_padding_mask=pad.to(DEV))
    keep = None
    if p > 0:
        seed, offset = (int(v) for v in blk._last_rng.tolist())
        B, T = x.shape[:2]
        keep = torch.from_numpy(philox.bst_keep_masks(seed, offset, B * T, p).reshape(3, B, T, 16))
    y.backward(g.to(DEV))
    rank_b200.check_index_errors()
    params = {k: v.detach().cpu().clone().requires_grad_() for k, v in blk.named_parameters()}
    xr = x.clone().requires_grad_()
    yr = X.bst_transformer_block(xr, pad, params, H, dropout_p=p, keep=keep)
    yr.backward(g)
    ref_grads = {k: v.grad for k, v in params.items()}
    ref_grads["x"] = xr.grad
    grads = {k: v.grad for k, v in blk.named_parameters()}
    grads["x"] = xa.grad
    p64 = {k: v.detach().double().requires_grad_() for k, v in params.items()}
    x64 = x.double().requires_grad_()
    X.bst_transformer_block(x64, pad, p64, H, dropout_p=p, keep=keep).backward(g.double())
    grads64 = {k: v.grad for k, v in p64.items()}
    grads64["x"] = x64.grad
    compare([y], grads, [yr.detach()], ref_grads, FP32_TOL, grads64)


@pytest.mark.parametrize("B,T,H", [(256, 300, 2), (256, 300, 8), (1024, 129, 4), (4, 2048, 16)])
def test_bst_transformer_module(B, T, H):
    blk, x, pad, g = _block_case(B, T, H, 0.0)
    _block_vs_oracle(blk, x, pad, g, H, 0.0)


def test_bst_transformer_module_lengths_straddling_the_chunk_edges():
    blk, x, pad, g = _block_case(512, 300, 4, 0.0, lens=_edge_lengths(512))
    _block_vs_oracle(blk, x, pad, g, 4, 0.0)


def test_bst_dropout_at_300_with_the_same_masks():
    blk, x, pad, g = _block_case(256, 300, 4, 0.1)
    _block_vs_oracle(blk, x, pad, g, 4, 0.1)


def test_length_zero_sample_is_nan_where_the_oracle_is():
    from oracle import interactions as X
    B, T, H = 64, 300, 4
    lens = torch.randint(1, T + 1, (B,), generator=torch.Generator().manual_seed(2))
    lens[5] = 0
    blk, x, pad, _ = _block_case(B, T, H, 0.0, lens=lens)
    with torch.no_grad():
        xd = x.to(DEV)
        y = blk(xd, xd, xd, key_padding_mask=pad.to(DEV)).cpu()
        params = {k: v.detach().cpu() for k, v in blk.named_parameters()}
        yr = X.bst_transformer_block(x, pad, params, H)
    assert torch.equal(torch.isnan(y), torch.isnan(yr))
    assert torch.isnan(yr[5]).all()
    keep = torch.arange(B) != 5
    assert rel_err(y[keep], yr[keep]) <= FP32_TOL


def test_out_of_range_id_past_128_is_reported(wechat_vocab_dir):
    ours, _ = _pair("BSTModel", "OracleBST", wechat_vocab_dir, **_kw(300))
    batch = synthetic.bst_batch(64, 300)
    length = batch["seq_length"].clone()
    length[3] = 280
    batch = _with_lengths(batch, length)
    batch["seq_feedid"][3, 200] = 10 ** 9
    batch = synthetic.to_device(batch, DEV)
    rank_b200.check_index_errors()
    with torch.no_grad():
        ours(batch["dense"], batch["category"], batch["seq_feedid"], batch["seq_length"])
    with pytest.raises(IndexError):
        rank_b200.check_index_errors()
    rank_b200.check_index_errors()           # the flag was cleared


def _step(model, batch, cot):
    model.zero_grad(set_to_none=True)
    _, logit = model(batch["dense"], batch["category"], batch["seq_feedid"], batch["seq_length"])
    (logit * cot).sum().backward()
    return logit.detach().clone(), {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}


def test_two_eager_backward_passes_are_bit_identical(wechat_vocab_dir):
    ours, _ = _pair("BSTModel", "OracleBST", wechat_vocab_dir, **_kw(600, 4, 2, "mean"))
    batch = synthetic.to_device(synthetic.bst_batch(700, 600), DEV)
    cot = torch.randn(700, 1, generator=torch.Generator().manual_seed(2)).to(DEV) / 700
    a, b = _step(ours, batch, cot), _step(ours, batch, cot)
    assert torch.equal(a[0], b[0])
    assert set(a[1]) == set(b[1])
    for k in a[1]:
        assert torch.equal(a[1][k], b[1][k]), k


def test_training_step_at_300_from_a_cuda_graph(wechat_vocab_dir):
    B, T = 512, 300
    ours, _ = _pair("BSTModel", "OracleBST", wechat_vocab_dir, hidden_units=[64, 32], **_kw(T, 4, 2))
    ours.train()
    batch = synthetic.to_device(synthetic.bst_batch(B, T), DEV)
    cot = torch.randn(B, 1, generator=torch.Generator().manual_seed(2)).to(DEV) / B
    params = list(ours.parameters())
    state = [p.detach().clone() for p in params]

    def body():
        _, logit = ours(batch["dense"], batch["category"], batch["seq_feedid"], batch["seq_length"])
        loss = (logit * cot).sum()
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
        assert rel_err(a, b, 1e-3 * float(b.abs().max()) + 1e-30) <= FP32_TOL, k


def test_tensor_core_block_refuses_129_positions_before_any_launch(wechat_vocab_dir):
    ours, _ = _pair("BSTModel", "OracleBST", wechat_vocab_dir, **_kw(129))
    ours.block_precision = "bf16"
    batch = synthetic.to_device(synthetic.bst_batch(256, 129), DEV)
    args = (batch["dense"], batch["category"], batch["seq_feedid"], batch["seq_length"])
    lib = _lib.load()
    torch.cuda.synchronize()
    launches = lib.rk_launch_count()
    with pytest.raises(_lib.RankB200Error, match="fp32"):
        ours(*args)
    assert lib.rk_launch_count() == launches
    blk = ours.transformer_blocks[0]
    x = torch.randn(4, 129, 16, device=DEV)
    with pytest.raises(_lib.RankB200Error, match="fp32"):
        blk.run(x, torch.full((4,), 129, device=DEV), precision="bf16")
    assert lib.rk_launch_count() == launches
    ours.block_precision = "fp32"
    ours(*args)
    assert lib.rk_launch_count() > launches


@pytest.mark.skipif(not dist.is_nccl_available(), reason="no NCCL")
def test_row_sharded_table_at_200_matches_replicated(wechat_vocab_dir):
    from test_sharded import _free_port
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{_free_port()}", rank=0, world_size=1,
                            device_id=torch.device("cuda", 0))
    try:
        torch.manual_seed(0)
        kw = _kw(200)
        a = rank_b200.BSTModel(wechat_vocab_dir, **kw).cuda()
        b = rank_b200.BSTModel(wechat_vocab_dir, **kw)
        b.load_state_dict(a.state_dict())
        b = rank_b200.shard_bst_feedid_table(b.cuda(), sparse_grad=False)
        batch = synthetic.to_device(synthetic.bst_batch(512, 200), DEV)
        outs = []
        for m in (a, b):
            m.train()
            logit = m(batch["dense"], batch["category"], batch["seq_feedid"], batch["seq_length"])[1]
            torch.nn.functional.binary_cross_entropy_with_logits(logit.squeeze(), batch["label"]).backward()
            outs.append(logit)
        assert rel_err(outs[1], outs[0]) <= 1e-6
        assert rel_err(b.embeddings["feedid"].weight.grad, a.embeddings["feedid"].weight.grad) <= 1e-5
        for (na, pa), (_, pb) in zip(a.named_parameters(), b.named_parameters()):
            if "feedid" not in na:
                assert rel_err(pb.grad, pa.grad, 1e-3 * float(pa.grad.abs().max()) + 1e-30) <= 1e-5, na
    finally:
        dist.destroy_process_group()
