"""rk_linear_wgrad (csrc/linear.cu) at the edges of its tensor-core tiling, against float64: output tiles of 128
n (one TMEM lane each), input tiles of up to 128 k padded to a multiple of 32 (the MMA's N), batch stages of
16 rows and slabs of the plan, with batches that are not a multiple of 8 or 32 rows.  Every shape here has a
grid large enough for the tensor-core kernel (test_linear_wgrad_tc.py checks that); smaller ones run the SIMT
kernel, which test_gpu_linear_wgrad.py covers."""
import pytest
import torch

from test_gpu_linear_wgrad import check_against_float64, wgrad

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.mark.parametrize("N", [127, 128, 129, 257])
@pytest.mark.parametrize("K", [8, 95, 96, 97, 129])
@pytest.mark.parametrize("B", [4099, 8197])
def test_tile_edges_match_float64(B, K, N):
    gen = torch.Generator(device=DEV).manual_seed(B * 1000 + K * 10 + N)
    x = torch.randn(B, K, device=DEV, generator=gen) + 0.25
    g = torch.randn(B, N, device=DEV, generator=gen)
    check_against_float64(x, g)


@pytest.mark.parametrize("B,K,N", [(8192 + 5, 82, 512), (4099, 512, 256), (8191, 256, 129), (4097, 96, 128)])
def test_slab_boundaries_match_float64(B, K, N):
    """Last slabs that end 1-31 rows into a 32-row group, and a last 16-row stage with fewer than 8 rows."""
    gen = torch.Generator(device=DEV).manual_seed(B + K + N)
    x = torch.randn(B, K, device=DEV, generator=gen)
    g = torch.randn(B, N, device=DEV, generator=gen) / B
    check_against_float64(x, g)


def test_magnitudes_far_from_one_match_float64():
    """The lo terms carry the bits below tf32 at any exponent."""
    gen = torch.Generator(device=DEV).manual_seed(5)
    x = torch.randn(2049, 97, device=DEV, generator=gen) * 1e-20
    g = torch.randn(2049, 129, device=DEV, generator=gen) * 1e15
    check_against_float64(x, g)


def test_bit_identical_runs_and_graph_replays_at_tile_edges():
    B, K, N = 1003, 97, 257
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
