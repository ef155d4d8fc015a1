"""rank_b200.Adam (rk_adam_step, csrc/optim.cu) against torch.optim.Adam(fused=True), bit for bit: dense
gradients, touched-rows gradients, whole models, a CUDA graph of the whole training step, state_dict
interchange, and the refusals."""
import pytest
import torch

import rank_b200
from rank_b200 import _lib
from rank_b200.optim import RowwiseAdam
from rank_b200.sparse import TouchedRows

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _assert_same(ours, ref, ps_o, ps_r, where):
    for po, pr in zip(ps_o, ps_r):
        assert torch.equal(po, pr), where
        so, sr = ours.state[po], ref.state[pr]
        for k in ("step", "exp_avg", "exp_avg_sq"):
            assert torch.equal(so[k], sr[k]), (where, k)


def _twins(shapes, seed=0):
    gen = torch.Generator().manual_seed(seed)
    base = [torch.randn(s, generator=gen) for s in shapes]
    return ([torch.nn.Parameter(b.to(DEV)) for b in base], [torch.nn.Parameter(b.to(DEV)) for b in base])


DENSE_SHAPES = [(1, 1), (3, 2), (100_000, 1), (7, 4), (12_345, 5), (50_000, 16), (333, 32), (100_000, 32),
                (513,), (1,), ()]


def test_dense_gradients_bitwise_two_groups():
    """Tables of every width the models use (and 5), biases, a 0-d tensor, a parameter whose storage is not
    16-byte aligned, and 70 small tensors (more than one launch), in two groups with different lr and betas."""
    shapes_a = DENSE_SHAPES
    shapes_b = [(4, 16), (9,)] + [(3 + k % 5,) for k in range(70)]
    a_o, a_r = _twins(shapes_a, 1)
    b_o, b_r = _twins(shapes_b, 2)
    store = torch.randn(97 * 4 + 1, device=DEV)              # a view at offset 1: vector width falls back to 1
    mis_o = torch.nn.Parameter(store[1:].view(97, 4))
    mis_r = torch.nn.Parameter(mis_o.detach().clone())
    assert mis_o.data_ptr() % 16 != 0
    groups_o = [dict(params=a_o + [mis_o]), dict(params=b_o, lr=3e-2, betas=(0.8, 0.95), eps=1e-6)]
    groups_r = [dict(params=a_r + [mis_r]), dict(params=b_r, lr=3e-2, betas=(0.8, 0.95), eps=1e-6)]
    ours = rank_b200.Adam(groups_o, lr=1e-3)
    ref = torch.optim.Adam(groups_r, lr=1e-3, fused=True)
    ps_o, ps_r = a_o + [mis_o] + b_o, a_r + [mis_r] + b_r
    gen = torch.Generator(device=DEV).manual_seed(5)
    n0 = _lib.load().rk_launch_count()
    for step in range(5):
        for po, pr in zip(ps_o, ps_r):
            g = torch.randn(po.shape, generator=gen, device=DEV) * 10 ** (step - 3)
            po.grad, pr.grad = g.clone(), g.clone()
        ours.step()
        ref.step()
        _assert_same(ours, ref, ps_o, ps_r, step)
    assert _lib.load().rk_launch_count() - n0 == 5 * 2             # 84 tensors: two launches per step


def _touched(V, D, rows, gen, capacity=None, garbage_rows=False):
    """A TouchedRows of the given distinct rows (sorted here), with `capacity` slots; values are zero past the
    count, as the backward leaves them."""
    rows = torch.as_tensor(sorted(set(int(r) for r in rows)), dtype=torch.int64)
    n = rows.numel()
    cap = max(n, capacity or n)
    r = torch.zeros(cap, dtype=torch.int64)
    if garbage_rows:
        r[n:] = torch.arange(cap - n) % V
    r[:n] = rows
    vals = torch.zeros(cap, D)
    vals[:n] = torch.randn(n, D, generator=gen)
    return TouchedRows(r.to(DEV), vals.to(DEV), torch.tensor([n], device=DEV), (V, D))


@pytest.mark.parametrize("V,D", [(1, 1), (7, 2), (5000, 1), (5000, 4), (12_345, 5), (100_000, 16), (333, 32),
                                 (4099, 32)])
def test_touched_gradients_bitwise(V, D):
    """Touched sets with a count of 0, a count below capacity, every row, and rows 0 and V-1, against fused Adam
    fed the dense gradient they stand for; the untouched rows' moments decay (RowwiseAdam leaves them alone)."""
    gen = torch.Generator().manual_seed(V * 100 + D)
    (po,), (pr,) = _twins([(V, D)], V + D)
    (pl,), _ = _twins([(V, D)], V + D)
    ours = rank_b200.Adam([po], lr=1e-2)
    ref = torch.optim.Adam([pr], lr=1e-2, fused=True)
    lazy = RowwiseAdam([pl], lr=1e-2)
    sets = [
        (torch.randint(0, V, (max(1, V // 3),), generator=gen).tolist(), V),             # count < capacity
        ([], 4),                                                                          # count 0
        (list(range(V)), None),                                                           # every row
        ([0, V - 1], 2 * V),                                                              # the first and last row
        (torch.randint(0, V, (max(1, V // 50),), generator=gen).tolist(), None),
    ]
    for step, (rows, cap) in enumerate(sets):
        t = _touched(V, D, rows, gen, cap, garbage_rows=step == 0)
        m_before = ours.state[po]["exp_avg"].clone() if ours.state else None
        pr.grad = t.to_dense()
        pl.touched_grad = t
        po.touched_grad = t
        ours.step()
        ref.step()
        assert po.touched_grad is None
        _assert_same(ours, ref, [po], [pr], step)
        untouched = torch.ones(V, dtype=torch.bool, device=DEV)
        untouched[t.rows[:int(t.count)]] = False
        m_lazy = lazy.state[pl]["exp_avg"].clone() if lazy.state else None
        lazy.step()
        if m_before is not None:
            moved = (m_before != 0) & untouched[:, None]
            if bool(moved.any()):
                assert bool((ours.state[po]["exp_avg"][moved] != m_before[moved]).all())      # decayed
                assert torch.equal(lazy.state[pl]["exp_avg"][moved], m_lazy[moved])          # left alone
    rank_b200.check_index_errors()


# ---- whole models ----------------------------------------------------------------------------------
def _workload(key):
    import bench
    return bench.WORKLOADS[key]()


MODELS = ["deepfm", "dcn", "din", "din_tc", "bst"]       # DIN with the fp32 and the bf16 activation unit
LR = 1e-3


def _train(key, vocab, mode, opt_kind, steps=3, B=None):
    """`steps` training steps; returns the model, its optimizer, the initial weights and the first step's dense
    gradients."""
    from rank_b200 import sparse, synthetic
    wl = _workload(key)
    torch.manual_seed(0)
    model = wl.model(rank_b200, False, vocab).to(DEV)
    model.train()
    opt = rank_b200.Adam(model.parameters(), lr=LR) if opt_kind == "ours" else \
        torch.optim.Adam(model.parameters(), lr=LR, fused=True)
    init = {k: p.detach().clone() for k, p in model.named_parameters()}
    first = {}
    sparse.set_table_gradients(mode)
    try:
        for step in range(steps):
            batch = synthetic.to_device(wl.make_batch(B or min(wl.batch, 4096), 100 + step), DEV)
            opt.zero_grad(set_to_none=True)
            torch.manual_seed(step)
            wl.loss(model, batch).backward()
            if step == 0:
                first = {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}
            opt.step()
    finally:
        sparse.set_table_gradients("dense")
    return model, opt, init, first


@pytest.mark.parametrize("key", MODELS)
def test_models_default_mode_bitwise_and_touched_mode_close(wechat_vocab_dir, key):
    from conftest import grad_floor
    ref_model, ref_opt, init, grads = _train(key, wechat_vocab_dir, "dense", "torch_fused")
    ours_model, ours_opt, _, _ = _train(key, wechat_vocab_dir, "dense", "ours")
    ps_o, ps_r = list(ours_model.parameters()), list(ref_model.parameters())
    _assert_same(ours_opt, ref_opt, ps_o, ps_r, key)
    touched_model, _, _, _ = _train(key, wechat_vocab_dir, "touched", "ours")
    # Touched-mode table gradients equal the dense ones within 1e-6 (test_gpu_optim.py), and the trajectories stay
    # that close: the difference of the two runs is at most 1e-2 of how far the parameters moved (L2 over each
    # tensor).  Parameters whose gradient is mathematically zero (a bias that a Linear + BatchNorm cancels, e.g.
    # DeepFM's deep_layers.0.bias, BST's norm2.bias) hold only rounding noise, below the gradient floor of
    # conftest.grad_floor; Adam divides by sqrt(v), so noise moves them by up to ~lr per step in either run, and they
    # are held to Adam's step size only.
    floor = grad_floor(grads)
    ref_p = dict(ref_model.named_parameters())
    for k, p in touched_model.named_parameters():
        diff = p.detach() - ref_p[k].detach()
        assert float(diff.abs().max()) <= 2 * LR * 3, k
        if k in grads and float(grads[k].abs().max()) > floor:
            moved = float((ref_p[k].detach() - init[k]).norm())
            assert float(diff.norm()) <= 1e-2 * moved, (k, float(diff.norm()), moved)
    rank_b200.check_index_errors()


def test_captured_touched_step_equals_eager_steps(wechat_vocab_dir):
    """zero_grad + forward + loss + backward + Adam.step of DeepFM in touched mode, captured in one CUDA graph and
    replayed k times, equals k eager steps bit for bit; an eager step() does not synchronise with the host."""
    from rank_b200 import sparse, synthetic
    wl = _workload("deepfm")
    torch.manual_seed(0)
    eager = wl.model(rank_b200, False, wechat_vocab_dir).to(DEV)
    graphed = wl.model(rank_b200, False, wechat_vocab_dir).to(DEV)
    graphed.load_state_dict(eager.state_dict())
    opt_e = rank_b200.Adam(eager.parameters(), lr=LR)
    opt_g = rank_b200.Adam(graphed.parameters(), lr=LR)
    batches = [synthetic.to_device(wl.make_batch(1024, 200 + i), DEV) for i in range(6)]
    static = synthetic.to_device(wl.make_batch(1024, 200), DEV)

    def copy_in(dst, src):
        for k in dst:
            if torch.is_tensor(dst[k]):
                dst[k].copy_(src[k])
            else:
                copy_in(dst[k], src[k])

    def body(model, opt, batch):
        opt.zero_grad(set_to_none=True)
        wl.loss(model, batch).backward()
        opt.step()

    sparse.set_table_gradients("touched")
    try:
        for i in range(2):                                # warm-up, the same steps on both
            body(eager, opt_e, batches[i])
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for i in range(2):
                body(graphed, opt_g, batches[i])
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            body(graphed, opt_g, static)
        for i in range(2, 6):
            copy_in(static, batches[i])
            graph.replay()
            opt_e.zero_grad(set_to_none=True)
            wl.loss(eager, batches[i]).backward()
            torch.cuda.synchronize()
            torch.cuda.set_sync_debug_mode("error")
            try:
                opt_e.step()
            finally:
                torch.cuda.set_sync_debug_mode(0)
        torch.cuda.synchronize()
    finally:
        sparse.set_table_gradients("dense")
    ps_e, ps_g = list(eager.parameters()), list(graphed.parameters())
    _assert_same(opt_g, opt_e, ps_g, ps_e, "graph")
    assert float(opt_g.state[ps_g[0]]["step"]) == 6.0
    rank_b200.check_index_errors()


# ---- state_dict interchange -------------------------------------------------------------------------
STATE_SHAPES = [(1000, 16), (50, 5), (64,), ()]


def _grads(shapes, steps):
    gen = torch.Generator(device=DEV).manual_seed(11)
    return [[torch.randn(s, generator=gen, device=DEV) for s in shapes] for _ in range(steps)]


def _run(opt, ps, grads):
    for gs in grads:
        for p, g in zip(ps, gs):
            p.grad = g.clone()
        opt.step()


@pytest.mark.parametrize("first", ["torch_fused", "ours", "torch_foreach"])
def test_state_dict_round_trip(first):
    """Two steps with one optimizer, its state loaded into the other, two more steps: equal to four steps of the
    continuing optimizer alone (fused Adam and rank_b200.Adam are the same arithmetic)."""
    grads = _grads(STATE_SHAPES, 4)
    ps_a, ps_b = _twins(STATE_SHAPES, 3)
    make = {"torch_fused": lambda ps: torch.optim.Adam(ps, lr=1e-2, betas=(0.85, 0.99), fused=True),
            "torch_foreach": lambda ps: torch.optim.Adam(ps, lr=1e-2, betas=(0.85, 0.99), foreach=True),
            "ours": lambda ps: rank_b200.Adam(ps, lr=1e-2, betas=(0.85, 0.99))}
    a = make[first](ps_a)
    _run(a, ps_a, grads[:2])
    then = rank_b200.Adam if first != "ours" else (lambda ps: torch.optim.Adam(ps, lr=0.5, fused=True))
    b = then(ps_a)
    b.load_state_dict(a.state_dict())
    _run(b, ps_a, grads[2:])
    # the reference: two steps of `first`, then two of fused-Adam arithmetic on the same state
    ref = make[first](ps_b)
    _run(ref, ps_b, grads[:2])
    ref2 = make["torch_fused"](ps_b)
    ref2.load_state_dict(ref.state_dict())
    ref2.param_groups[0]["fused"], ref2.param_groups[0]["foreach"] = True, None
    for st in ref2.state.values():                        # foreach keeps the step on the host; fused wants it here
        st["step"] = st["step"].to(DEV)
    _run(ref2, ps_b, grads[2:])
    _assert_same(b, ref2, ps_a, ps_b, first)


# ---- refusals ---------------------------------------------------------------------------------------
def _refused(opt, ps, exc, match=None):
    lib = _lib.load()
    n0 = lib.rk_launch_count()
    before = [p.detach().clone() for p in ps]
    steps = {id(p): opt.state[p]["step"].clone() for p in ps if opt.state.get(p)}
    with pytest.raises(exc, match=match):
        opt.step()
    torch.cuda.synchronize()
    assert lib.rk_launch_count() == n0
    assert all(torch.equal(p, b) for p, b in zip(ps, before))
    assert all(torch.equal(opt.state[p]["step"], steps[id(p)]) for p in ps if id(p) in steps)


def _with(bad):
    """An optimizer over a valid parameter that has state already (its step must not move on a refusal) and `bad`."""
    good = torch.nn.Parameter(torch.randn(10, 4, device=DEV))
    good.grad = torch.ones_like(good)
    opt = rank_b200.Adam([good])
    opt.step()
    good.grad = torch.ones_like(good)
    opt.add_param_group(dict(params=[bad]))
    return opt, [good, bad]


def test_every_refusal_comes_before_a_launch():

    half = torch.nn.Parameter(torch.randn(10, 4, device=DEV, dtype=torch.float16))
    half.grad = torch.ones_like(half)
    _refused(*_with(half), TypeError)

    strided = torch.nn.Parameter(torch.randn(4, 10, device=DEV).t())
    strided.grad = torch.ones_like(strided)
    _refused(*_with(strided), RuntimeError, "contiguous")

    cpu = torch.nn.Parameter(torch.randn(3))
    cpu.grad = torch.ones_like(cpu)
    _refused(*_with(cpu), rank_b200.RankB200Error)

    emb = torch.nn.Embedding(10, 4, sparse=True).to(DEV)
    emb(torch.tensor([1, 2], device=DEV)).sum().backward()
    _refused(*_with(emb.weight), RuntimeError, "sparse")

    gen = torch.Generator().manual_seed(0)
    both = torch.nn.Parameter(torch.randn(10, 4, device=DEV))
    both.grad = torch.ones_like(both)
    both.touched_grad = _touched(10, 4, [1, 3], gen)
    _refused(*_with(both), RuntimeError, "both")

    wrong = torch.nn.Parameter(torch.randn(10, 4, device=DEV))
    wrong.touched_grad = _touched(11, 4, [1, 3], gen)
    _refused(*_with(wrong), RuntimeError, "does not match")


def test_touched_row_out_of_range_sets_the_index_flag():
    gen = torch.Generator().manual_seed(1)
    V, D = 300, 4
    for bad in ([-3, 5, 17], [0, 5, V + 2]):
        (po,), (pr,) = _twins([(V, D)], 9)
        t = _touched(V, D, bad, gen)
        ok = t.rows[:3].clone()
        valid = (ok >= 0) & (ok < V)
        dense = torch.zeros(V, D, device=DEV)
        dense[ok[valid]] = t.values[:3][valid]
        po.touched_grad = t
        pr.grad = dense
        ours, ref = rank_b200.Adam([po]), torch.optim.Adam([pr], fused=True)
        ours.step()
        ref.step()
        _assert_same(ours, ref, [po], [pr], bad)          # the valid rows are updated, the others skipped
        with pytest.raises(IndexError):
            rank_b200.check_index_errors()
    rank_b200.check_index_errors()
