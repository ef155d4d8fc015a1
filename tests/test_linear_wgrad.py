"""rk_linear_wgrad without a GPU: argument refusals, the scratch query, and the slab / tile partition of
csrc/linear.cu restated in numpy (every batch row meets every output exactly once)."""
import math

import numpy as np
import pytest

from rank_b200 import _lib

TILE, ROWS, TARGET_CTAS = 64, 32, 148 * 4       # csrc/linear.cu: kLinTile, kLinRows, kLinTargetCtas
BENCH_SHAPES = [(82, 512), (512, 256), (256, 128), (128, 1), (66, 512), (82, 200), (200, 80), (80, 1), (1, 1)]


def plan(B, K, N):
    """linear_plan: (slabs, rows per slab)."""
    tiles = math.ceil(K / TILE) * math.ceil(N / TILE)
    want = math.ceil(TARGET_CTAS / tiles)
    rows = math.ceil(math.ceil(B / want) / ROWS) * ROWS
    return math.ceil(B / rows), rows


@pytest.mark.parametrize("B,K,N", [(0, 8, 8), (8, 0, 8), (8, 8, 0), (-1, 8, 8)])
def test_bad_shapes_are_refused(B, K, N):
    lib = _lib.load()
    assert lib.rk_linear_wgrad_scratch_floats(B, K, N) == -1
    assert lib.rk_linear_wgrad(16, K, 16, N, B, K, N, 16, 16, 16, None) < 0


def test_bad_pointers_and_pitches_are_refused():
    lib = _lib.load()
    assert lib.rk_linear_wgrad(None, 8, 16, 8, 4, 8, 8, 16, None, 16, None) < 0           # x
    assert lib.rk_linear_wgrad(16, 8, None, 8, 4, 8, 8, 16, None, 16, None) < 0           # g
    assert lib.rk_linear_wgrad(16, 8, 16, 8, 4, 8, 8, None, None, 16, None) < 0           # dW
    assert lib.rk_linear_wgrad(16, 7, 16, 8, 4, 8, 8, 16, None, 16, None) < 0             # ldx < K
    assert lib.rk_linear_wgrad(16, 8, 16, 7, 4, 8, 8, 16, None, 16, None) < 0             # ldg < N
    assert lib.rk_linear_wgrad(16, 8, 16, 65535 * 64 + 1, 4, 8, 65535 * 64 + 1, 16, None, 16, None) < 0
    B, K, N = 8192, 256, 128                                                                # needs partials
    assert lib.rk_linear_wgrad_scratch_floats(B, K, N) > 0
    assert lib.rk_linear_wgrad(16, K, 16, N, B, K, N, 16, 16, None, None) < 0
    assert b"partials" in lib.rk_last_error()


@pytest.mark.parametrize("B", [1, 2, 31, 333, 1024, 8192, 16384, 1 << 20])
@pytest.mark.parametrize("K,N", BENCH_SHAPES)
def test_scratch_query_matches_the_plan(B, K, N):
    S, rows = plan(B, K, N)
    assert rows % ROWS == 0 and (S - 1) * rows < B <= S * rows        # no empty slab
    want = S * (N * K + N) if S > 1 else 0
    assert _lib.load().rk_linear_wgrad_scratch_floats(B, K, N) == want


@pytest.mark.parametrize("B,K,N", [(1, 1, 1), (2, 82, 3), (333, 82, 512), (8192, 256, 128), (1000, 200, 80),
                                   (8192, 512, 256), (97, 65, 129)])
def test_partition_covers_every_row_and_output_once(B, K, N):
    """Every CTA (k tile, n tile, slab) and every staged step within it, as the kernel walks them.  A step
    visits (its rows) x (its tile's n) x (its tile's k), so each (row, n, k) is visited once exactly when
    the steps cover each row once and the tiles cover each (n, k) once; the db CTAs (first k tile) then
    cover each (row, n) once."""
    S, rows = plan(B, K, N)
    seen_rows = np.zeros(B, dtype=np.int32)
    for s in range(S):
        row0, row_end = s * rows, min(B, (s + 1) * rows)
        for step in range(math.ceil((row_end - row0) / ROWS)):
            r = np.arange(row0 + step * ROWS, row0 + (step + 1) * ROWS)
            seen_rows[r[r < row_end]] += 1                         # zero-filled beyond the slab
    seen_out = np.zeros((N, K), dtype=np.int32)
    seen_db = np.zeros(N, dtype=np.int32)
    for kt in range(math.ceil(K / TILE)):
        for nt in range(math.ceil(N / TILE)):
            seen_out[nt * TILE:(nt + 1) * TILE, kt * TILE:(kt + 1) * TILE] += 1
            if kt == 0:
                seen_db[nt * TILE:(nt + 1) * TILE] += 1
    assert (seen_rows == 1).all()
    assert (seen_out == 1).all()
    assert (seen_db == 1).all()
