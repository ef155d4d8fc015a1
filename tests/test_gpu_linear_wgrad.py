"""rk_linear_wgrad (csrc/linear.cu) against float64 G^T X and G.sum(0), its determinism under CUDA graphs, and
run_tower's nn.Linear routing against the plain modules."""
import copy

import pytest
import torch
import torch.nn as nn

import rank_b200
from rank_b200 import _lib, tower
from conftest import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5
# (B, in, out) of every Linear that run_tower meets in bench.py's workloads: DIN, BST, DCN, DeepFM
BENCH_SHAPES = [(8192, 82, 512), (8192, 512, 256), (8192, 256, 128), (8192, 66, 512), (8192, 128, 1),
                (8192, 50, 512), (1024, 96, 512), (1024, 512, 256), (1024, 256, 128)]


def wgrad(x, g, bias=True):
    lib = _lib.load()
    B, K = x.shape
    N = g.shape[1]
    dW = torch.empty(N, K, device=DEV)
    db = torch.empty(N, device=DEV) if bias else None
    partials = torch.empty(lib.rk_linear_wgrad_scratch_floats(B, K, N), device=DEV)
    _lib.check(lib.rk_linear_wgrad(x.data_ptr(), x.stride(0), g.data_ptr(), g.stride(0), B, K, N, dW.data_ptr(),
                                   _lib.ptr(db), partials.data_ptr() if partials.numel() else None,
                                   _lib.stream_ptr()), "rk_linear_wgrad")
    return dW, db


def check_against_float64(x, g):
    dW, db = wgrad(x, g)
    x64, g64 = x.double(), g.double()
    # the error bar of an fp32 sum of B products is relative to sum |g x|, not to the (cancelling) result
    scale_w = float((g64.abs().t() @ x64.abs()).max())
    scale_b = float(g64.abs().sum(0).max())
    assert float((dW.double() - g64.t() @ x64).abs().max()) <= TOL * scale_w
    assert float((db.double() - g64.sum(0)).abs().max()) <= TOL * scale_b


@pytest.mark.parametrize("B,K,N", BENCH_SHAPES)
def test_bench_shapes_match_float64(B, K, N):
    gen = torch.Generator(device=DEV).manual_seed(B + K + N)
    x = torch.randn(B, K, device=DEV, generator=gen)
    g = torch.randn(B, N, device=DEV, generator=gen) / B
    check_against_float64(x, g)


@pytest.mark.parametrize("B", [1, 2, 333, 1024, 8192, 16384])
@pytest.mark.parametrize("K", [1, 82, 200])
@pytest.mark.parametrize("N", [1, 3, 512])
def test_shapes_match_float64(B, K, N):
    gen = torch.Generator(device=DEV).manual_seed(7 * B + K + N)
    x = torch.randn(B, K, device=DEV, generator=gen) + 0.5
    g = torch.randn(B, N, device=DEV, generator=gen)
    check_against_float64(x, g)


@pytest.mark.parametrize("B,K,N,pad_x,pad_g", [(8192, 82, 512, 1, 3), (1000, 128, 256, 4, 0), (333, 5, 7, 2, 1),
                                               (8192, 256, 128, 0, 4)])
def test_strided_rows(B, K, N, pad_x, pad_g):
    gen = torch.Generator(device=DEV).manual_seed(B + pad_x)
    xs = torch.randn(B, K + pad_x, device=DEV, generator=gen)
    gs = torch.randn(B, N + pad_g, device=DEV, generator=gen)
    x, g = xs[:, pad_x:], gs[:, :N]                 # row pitch K + pad_x / N + pad_g, x offset by pad_x floats
    check_against_float64(x, g)
    dW, db = wgrad(x, g)
    dW_c, db_c = wgrad(x.contiguous(), g.contiguous())
    assert torch.equal(dW, dW_c) and torch.equal(db, db_c)


def test_no_bias():
    x = torch.randn(4096, 82, device=DEV)
    g = torch.randn(4096, 512, device=DEV)
    dW, db = wgrad(x, g, bias=False)
    assert db is None
    assert torch.equal(dW, wgrad(x, g)[0])


@pytest.mark.parametrize("B,K,N", [(8192, 256, 128), (333, 82, 3)])
def test_bit_identical_runs_and_graph_replays(B, K, N):
    x = torch.randn(B, K, device=DEV)
    g = torch.randn(B, N, device=DEV)
    dW1, db1 = wgrad(x, g)
    dW2, db2 = wgrad(x, g)
    assert torch.equal(dW1, dW2) and torch.equal(db1, db2)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        wgrad(x, g)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        dW3, db3 = wgrad(x, g)
    for _ in range(3):
        dW3.zero_(), db3.zero_()
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(dW1, dW3) and torch.equal(db1, db3)


def _tower(kind):
    torch.manual_seed(3)
    if kind == "din":
        mods = []
        for k, n in ((82, 512), (512, 256), (256, 128)):
            mods += [nn.Linear(k, n), rank_b200.Dice(n), nn.BatchNorm1d(n)]
    elif kind == "bst":
        mods = []
        for k, n in ((66, 512), (512, 256), (256, 128)):
            mods += [nn.Linear(k, n), nn.BatchNorm1d(n), nn.LeakyReLU(0.01)]
        mods.append(nn.Linear(128, 1))
    else:
        mods = [nn.Linear(50, 512), nn.ReLU(), nn.Linear(512, 256), nn.ReLU(), nn.Linear(256, 128), nn.ReLU()]
    return nn.ModuleList(mods).to(DEV).train(), mods[0].in_features


def _run(mods, x0, cot, fused):
    tower.FUSED = fused
    try:
        x = x0.clone().requires_grad_()
        out = tower.run_tower(mods, x)
        mods.zero_grad()
        (out * cot).sum().backward()
    finally:
        tower.FUSED = True
    return out.detach(), x.grad, [p.grad for p in mods.parameters()]


def _inputs(kind, width):
    gen = torch.Generator().manual_seed(11)
    x0 = torch.randn(8192, width, generator=gen).to(DEV)
    return x0, torch.randn(8192, 1 if kind == "bst" else 128, generator=gen).to(DEV) / 8192


def _grads64(mods, x0, cot):
    """The parameter gradients of the same tower run by torch in float64: the arbiter of sums over the batch."""
    m64 = copy.deepcopy(mods).double()
    return _run(m64, x0.double(), cot.double(), False)[2]


def _linear_grads_close(mods, ours, ref, ref64):
    """Within 1e-5 of torch's fp32 gradients (those that are zero up to cancellation against the tower's
    gradient scale).  Where a batch-long fp32 sum misses that, as test_gpu_models does: ours within 1e-5 of the
    float64 run, or no further from it than twice torch's fp32 result."""
    gmax = max(float(g.abs().max()) for g in ref)
    names = [k for k, _ in mods.named_parameters()]
    for k, a, b, t in zip(names, ours, ref, ref64):
        zero = float(b.abs().max()) < 1e-4 * gmax
        scale = gmax if zero else float(b.abs().max())
        if float((a - b).abs().max()) > TOL * scale:
            scale = gmax if zero else float(t.abs().max())
            e_ours = float((a.double() - t).abs().max()) / scale
            e_ref = float((b.double() - t).abs().max()) / scale
            assert e_ours <= max(TOL, 2.0 * e_ref), (k, e_ours, e_ref)


@pytest.mark.parametrize("kind", ["din", "bst", "dcn"])
def test_run_tower_matches_modules(kind):
    """FUSED on against FUSED off: outputs and the input gradient within 1e-5, every parameter gradient as
    _linear_grads_close judges it."""
    fused, width = _tower(kind)
    plain = copy.deepcopy(fused)
    x0, cot = _inputs(kind, width)
    gp64 = _grads64(fused, x0, cot)
    o1, gx1, gp1 = _run(fused, x0, cot, True)
    o2, gx2, gp2 = _run(plain, x0, cot, False)
    assert rel_err(o1, o2) <= TOL and rel_err(gx1, gx2) <= TOL
    _linear_grads_close(plain, gp1, gp2, gp64)


@pytest.mark.parametrize("kind", ["din", "bst", "dcn"])
def test_only_linear_weight_gradients_change(kind):
    """The same fused tower with each nn.Linear hidden in an nn.Sequential (so torch computes its weight
    gradients): outputs, the input gradient and every non-Linear gradient are bit-identical."""
    fused, width = _tower(kind)
    plain = nn.ModuleList([nn.Sequential(m) if type(m) is nn.Linear else m for m in copy.deepcopy(fused)])
    x0, cot = _inputs(kind, width)
    gp64 = _grads64(fused, x0, cot)
    o1, gx1, gp1 = _run(fused, x0, cot, True)
    o2, gx2, gp2 = _run(plain, x0, cot, True)
    assert torch.equal(o1, o2) and torch.equal(gx1, gx2)
    linear_params = {id(p) for m in fused if type(m) is nn.Linear for p in m.parameters()}
    for p, a, b in zip(fused.parameters(), gp1, gp2):
        if id(p) not in linear_params:
            assert torch.equal(a, b)
    _linear_grads_close(fused, gp1, gp2, gp64)


def test_linear_layers_route_through_the_kernel():
    mods, width = _tower("dcn")
    x = torch.randn(512, width, device=DEV, requires_grad=True)
    before = _lib.load().rk_launch_count()
    tower.run_tower(mods, x).sum().backward()
    torch.cuda.synchronize()
    assert _lib.load().rk_launch_count() - before >= 3


def test_narrow_linear_keeps_torchs_weight_gradient():
    """Fewer outputs than one dW tile (BST's final Linear(128, 1)): torch is faster there and runs it."""
    mods = nn.ModuleList([nn.Linear(128, tower.LINEAR_MIN_OUT - 1)]).to(DEV)
    x = torch.randn(8192, 128, device=DEV, requires_grad=True)
    before = _lib.load().rk_launch_count()
    tower.run_tower(mods, x).sum().backward()
    torch.cuda.synchronize()
    assert _lib.load().rk_launch_count() == before
