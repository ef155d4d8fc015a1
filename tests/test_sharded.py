"""Row-sharded table: the exchange logic on CPU (gloo, world size 2, device steps injected from the
oracle side) and the CUDA path on one GPU (world size 1) / two GPUs when present."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import rank_b200
from rank_b200.sharded import RowShardedEmbedding
from oracle import interactions as X


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


class OracleShardOps:
    """CPU stand-in for CudaShardOps (test infrastructure): same contracts, numpy/torch."""

    def route(self, idx, rows_total, rows_per_rank, world):
        idx = idx.reshape(-1)
        if idx.numel() and (int(idx.min()) < 0 or int(idx.max()) >= rows_total):
            raise IndexError("index out of range in self")
        owner = idx // rows_per_rank
        order = torch.from_numpy(np.argsort(owner.numpy(), kind="stable"))
        inv = torch.empty_like(order)
        inv[order] = torch.arange(order.numel())
        send_local = idx[order] - owner[order] * rows_per_rank
        return send_local, inv, torch.bincount(owner, minlength=world).to(torch.int64)

    def gather(self, table, rows_idx):
        return X.gather_rows(table, rows_idx)

    def owner_plan(self, recv_key, rows_plus):
        return recv_key

    def reduce(self, plan, g_rows, rows_local, dim, sparse, any_dead):
        dense = torch.from_numpy(X.dense_embedding_grad(plan.numpy(), g_rows.detach().numpy(), rows_local + 1))
        dense = dense[:rows_local]
        if not sparse:
            return dense
        from rank_b200.sparse import TouchedRows
        uniq = torch.unique(plan[plan < rows_local])
        return TouchedRows(uniq, dense[uniq], torch.tensor([uniq.numel()]), (rows_local, dim))


def _gloo_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    gen = torch.Generator().manual_seed(7)
    V, D, n = 37, 4, 50
    full = torch.randn(V, D, generator=gen)
    idx_all = torch.randint(0, V, (world, n), generator=gen)
    cot_all = torch.randn(world, n, D, generator=gen)
    for sparse in (False, True):
        emb = RowShardedEmbedding.from_full(full, sparse_grad=sparse, _ops=OracleShardOps())
        emb.grad_scale = 1.0
        got = emb(idx_all[rank])
        (got * cot_all[rank]).sum().backward()
        ok_fwd = torch.equal(got.detach(), full[idx_all[rank]])
        # reference: the replicated table sees the occurrences of every rank
        ref = full.clone().requires_grad_()
        sum((ref[idx_all[r]] * cot_all[r]).sum() for r in range(world)).backward()
        lo, hi = emb.row_range
        g = emb.weight.touched_grad.to_dense() if sparse else emb.weight.grad
        assert not sparse or emb.weight.grad is None
        err = float((g[:hi - lo] - ref.grad[lo:hi]).abs().max())
        out.put((rank, sparse, ok_fwd, err))
    dist.barrier()
    dist.destroy_process_group()


def test_exchange_logic_world2_gloo():
    ctx = mp.get_context("spawn")
    out = ctx.SimpleQueue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(180)
        assert p.exitcode == 0
    results = [out.get() for _ in range(4)]
    assert len(results) == 4
    for rank, sparse, ok_fwd, err in results:
        assert ok_fwd, (rank, sparse)
        assert err < 1e-5, (rank, sparse, err)


@pytest.fixture
def single_rank_nccl():
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{_free_port()}", rank=0, world_size=1,
                            device_id=torch.device("cuda", 0))
    yield
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("sparse", [False, True])
def test_sharded_embedding_cuda_world1(single_rank_nccl, sparse):
    gen = torch.Generator().manual_seed(3)
    V, D = 5000, 16
    full = torch.randn(V, D, generator=gen)
    idx = torch.randint(0, V, (300, 20), generator=gen)
    idx[0, :5] = 7                                    # duplicates
    cot = torch.randn(300, 20, D, generator=gen)
    emb = RowShardedEmbedding.from_full(full.cuda(), sparse_grad=sparse)
    got = emb(idx.cuda())
    assert torch.equal(got.cpu(), full[idx])           # gathered rows are bit-exact
    (got * cot.cuda()).sum().backward()
    ref = full.clone().requires_grad_()
    (ref[idx] * cot).sum().backward()
    g = emb.weight.grad
    if sparse:
        t = emb.weight.touched_grad          # distinct rows + summed rows, count on the device (no host sync)
        assert g is None and int(t.count) == int(torch.unique(idx).numel())
        assert torch.equal(t.rows[:int(t.count)].cpu(), torch.unique(idx))
        g = t.to_dense()
    assert float((g.cpu() - ref.grad).abs().max()) <= 1e-5 * float(ref.grad.abs().max())
    rank_b200.check_index_errors()


@pytest.mark.gpu
def test_bst_with_sharded_feedid_table_matches_replicated(single_rank_nccl, wechat_vocab_dir):
    from rank_b200 import synthetic
    from conftest import to_device, rel_err
    torch.manual_seed(0)
    kw = dict(dropout_rate=0.0, nhead=4, num_transformer_blocks=1, max_seq_length=20)
    a = rank_b200.BSTModel(wechat_vocab_dir, **kw).cuda()
    b = rank_b200.BSTModel(wechat_vocab_dir, **kw)
    b.load_state_dict(a.state_dict())
    b = rank_b200.shard_bst_feedid_table(b.cuda(), sparse_grad=False)
    batch = to_device(synthetic.bst_batch(512, 20), "cuda")
    outs = []
    for m in (a, b):
        m.train()
        logit = m(batch["dense"], batch["category"], batch["seq_feedid"], batch["seq_length"])[1]
        torch.nn.functional.binary_cross_entropy_with_logits(logit.squeeze(), batch["label"]).backward()
        outs.append(logit)
    assert rel_err(outs[1], outs[0]) <= 1e-6
    ga = a.embeddings["feedid"].weight.grad
    gb = b.embeddings["feedid"].weight.grad
    assert rel_err(gb, ga) <= 1e-5
    for (na, pa), (nb, pb) in zip(a.named_parameters(), b.named_parameters()):
        if "feedid" not in na:
            assert rel_err(pb.grad, pa.grad, 1e-3 * float(pa.grad.abs().max()) + 1e-30) <= 1e-5, na


def _nccl_worker(rank, world, port, vocab_dir, out):
    """Two ranks, each with its own batch: the sharded model against a replicated model fed every
    rank's batch (what scripts/sharded_bst.py checks at 8 GPUs), dense and touched-rows gradients."""
    import torch.nn.functional as F
    from rank_b200 import synthetic
    from rank_b200.parallel import GradientAllReducer
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    kw = dict(dropout_rate=0.0, nhead=4, num_transformer_blocks=1, max_seq_length=20)

    def rel(a, b):
        return float((a.double() - b.double()).abs().max() / max(float(b.abs().max()), 1e-30))

    def loss_of(model, b):
        logit = model(b["dense"], b["category"], b["seq_feedid"], b["seq_length"])[1]
        return F.binary_cross_entropy_with_logits(logit.squeeze(), b["label"]), logit

    res = {}
    for sparse in (False, True):
        torch.manual_seed(0)
        full = rank_b200.BSTModel(vocab_dir, **kw).to(dev)
        torch.manual_seed(0)
        shard = rank_b200.shard_bst_feedid_table(rank_b200.BSTModel(vocab_dir, **kw).to(dev), sparse_grad=sparse)
        reducer = GradientAllReducer(shard)
        batches = [synthetic.to_device(synthetic.bst_batch(256, 20, seed=100 + r), dev) for r in range(world)]
        shard.train(); full.train()
        l_s, logit_s = loss_of(shard, batches[rank])
        l_s.backward()
        reducer.allreduce()
        for r in range(world):
            l_r, logit_r = loss_of(full, batches[r])
            (l_r / world).backward()
            if r == rank:
                e_logit = rel(logit_s, logit_r)
        feed = shard.embeddings["feedid"]
        lo, hi = feed.row_range
        g = feed.weight.touched_grad.to_dense() if sparse else feed.weight.grad
        e_shard = rel(g[:hi - lo], full.embeddings["feedid"].weight.grad[lo:hi])
        e_rest = max(rel(ps.grad, pf.grad) for (ns, ps), (nf, pf) in
                     zip(shard.named_parameters(), full.named_parameters())
                     if "feedid" not in ns and float(pf.grad.abs().max()) > 1e-6)
        res[sparse] = (e_logit, e_shard, e_rest)
    rank_b200.check_index_errors()
    out.put((rank, res))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_sharded_bst_two_ranks_nccl(wechat_vocab_dir):
    """The all-to-all path proper (needs two GPUs; the one-GPU box runs the world-1 tests above)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ctx = mp.get_context("spawn")
    out = ctx.SimpleQueue()
    port = _free_port()
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, wechat_vocab_dir, out)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
        assert p.exitcode == 0
    for _ in range(2):
        rank, res = out.get()
        for sparse, (e_logit, e_shard, e_rest) in res.items():
            assert e_logit <= 1e-5 and e_shard <= 1e-5 and e_rest <= 1e-4, (rank, sparse, e_logit, e_shard, e_rest)
