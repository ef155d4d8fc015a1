"""csrc/linear.cu's tensor-core scheme restated on the host (CPU; no extension needed):
  * the MN-major tf32 staging: where each (batch row, column) of a 16-row stage is stored, and that the
    shared-memory descriptors the MMAs read with walk exactly those slots, each once;
  * the kind::tf32 instruction descriptor and the shared-memory descriptor, packed from the documented fields;
  * the 3xTF32 split x = hi + lo;
  * the CTA tiling: every (n, k) of dW in one tile, every batch row of a slab in one stage.
"""
import math

import numpy as np
import pytest

# csrc/linear.cu
TC_N, TC_K, TC_ROWS, TC_STAGES, TC_THREADS = 128, 128, 16, 3, 256
LINE = 128                       # bytes: one staged row of 32 fp32 columns
BLOCK = TC_ROWS * LINE           # 32-column block of a stage: the leading byte offset
TILE = 4 * BLOCK                 # 128 columns x 16 rows
STAGE = 4 * TILE                 # G hi, G lo, X hi, X lo
SMEM = 1024 + TC_STAGES * STAGE + 64
TMEM_COLS = 128


def chunk_offset(r, c):
    """linear.cu::tc_chunk_offset: 16-byte chunk of columns 4c..4c+3 of stage row r."""
    return (c >> 3) * BLOCK + r * LINE + ((((c & 7) >> 1) ^ (r & 3)) << 5) + ((c & 1) << 4)


def staged_address(r, col):
    return chunk_offset(r, col // 4) + 4 * (col % 4)


def mma_read_address(start, lbo, mn, line, sbo=512):
    """What an MN-major SWIZZLE_128B_BASE32B operand descriptor (the only layout MN-major tf32 takes) addresses
    for element (mn, K line) of one MMA (K = 8 lines): blocks of 32 tf32 MN elements `lbo` apart, 128-byte lines,
    4-line groups `sbo` apart, then the swizzle on the absolute address (bits [5,7) ^= bits [7,9), CUTLASS's
    Swizzle<2,5,2> of Layout_MN_SW128_32B_Atom)."""
    a = start + (mn // 32) * lbo + (line // 4) * sbo + (line % 4) * LINE + (mn % 32) * 4
    return a ^ (((a >> 7) & 3) << 5)


def test_staging_fills_every_slot_of_a_tile_once():
    slots = np.array([staged_address(r, c) for r in range(TC_ROWS) for c in range(TC_N)])
    assert (slots % 4 == 0).all()
    assert sorted(slots // 4) == list(range(TILE // 4))


@pytest.mark.parametrize("tile_base", [0, 1024 * 7, 1024 * 40])      # 1024-aligned, as the kernel rounds its base
def test_descriptors_walk_the_staged_rows(tile_base):
    """MMA kk of a stage reads rows 8kk..8kk+7: descriptor start +1024 bytes per 8 rows (two 4-line atoms),
    32-column blocks BLOCK apart.  Each (row, column) of the stage is read exactly once, from where it was staged."""
    seen = np.zeros(TILE // 4, dtype=np.int32)
    for kk in range(TC_ROWS // 8):
        start = tile_base + 1024 * kk
        for line in range(8):
            for mn in range(TC_N):
                a = mma_read_address(start, BLOCK, mn, line)
                assert a == tile_base + staged_address(8 * kk + line, mn)
                seen[(a - tile_base) // 4] += 1
    assert (seen == 1).all()


def test_unaligned_base_breaks_the_swizzle():
    """Why the kernel rounds the dynamic shared-memory base up to 1024 bytes."""
    base = 128
    bad = [mma_read_address(base, BLOCK, mn, line) != base + staged_address(line, mn)
           for line in range(8) for mn in range(TC_N)]
    assert any(bad)


def smem_desc_shipped(addr, lbo):
    """umma.cuh::umma_desc_mn_tf32, restated by hand (the GPU tests check the encoding itself)."""
    d = (addr & 0x3FFFF) >> 4
    d |= ((lbo >> 4) & 0x3FFF) << 16
    d |= (512 >> 4) << 32
    d |= 1 << 46
    d |= 1 << 61
    return d


def smem_desc_fields(addr, lbo, sbo=512):
    """The documented tcgen05 shared-memory descriptor: start >> 4 [0,14), leading byte offset >> 4 [16,30),
    stride byte offset >> 4 [32,46), version 1 [46,48), base offset 0 [49,52), lbo mode 0 [52],
    layout 1 = SWIZZLE_128B_BASE32B [61,64)."""
    fields = [(0, 14, addr >> 4), (16, 14, lbo >> 4), (32, 14, sbo >> 4), (46, 2, 1), (49, 3, 0), (52, 1, 0),
              (61, 3, 1)]
    d = 0
    for lo, width, v in fields:
        assert 0 <= v < (1 << width)
        d |= v << lo
    return d


@pytest.mark.parametrize("addr", [0, 1024, 97 * 1024, 200 * 1024 + 3 * TILE])
def test_smem_descriptor_bits(addr):
    assert smem_desc_shipped(addr, BLOCK) == smem_desc_fields(addr, BLOCK)


def idesc_tf32_shipped(n):
    """umma.cuh::umma_idesc_tf32(n) | kUmmaAMn | kUmmaBMn, restated by hand (the GPU tests check the encoding)."""
    return (1 << 4) | (2 << 7) | (2 << 10) | ((n >> 3) << 17) | ((128 >> 4) << 24) | (1 << 15) | (1 << 16)


def idesc_fields(n, m=128):
    """The documented instruction descriptor of kind::tf32: D format F32 = 1 [4,6), A and B format TF32 = 2
    [7,10) and [10,13), no negation [13], [14], A and B MN-major = 1 [15], [16], N >> 3 [17,23), M >> 4 [24,29)."""
    fields = [(4, 2, 1), (7, 3, 2), (10, 3, 2), (13, 1, 0), (14, 1, 0), (15, 1, 1), (16, 1, 1), (17, 6, n >> 3),
              (24, 5, m >> 4)]
    d = 0
    for lo, width, v in fields:
        assert 0 <= v < (1 << width)
        d |= v << lo
    return d


@pytest.mark.parametrize("n", [32, 64, 96, 128])
def test_instruction_descriptor_bits(n):
    assert n % 16 == 0 and 16 <= n <= 256                # valid N for M = 128
    assert idesc_tf32_shipped(n) == idesc_fields(n)


def split_tf32(x):
    """umma.cuh::split_tf32: hi = cvt.rna.tf32.f32(x) (round the magnitude to 10 mantissa bits, ties away
    from zero), lo = x - hi in fp32."""
    x = np.asarray(x, dtype=np.float32)
    bits = x.view(np.uint32)
    hi = ((bits + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)
    return hi, (x - hi).astype(np.float32)


def _values():
    rng = np.random.default_rng(0)
    normal = rng.standard_normal(20000).astype(np.float32) * np.float32(10.0) ** rng.integers(-30, 30, 20000)
    sub = (rng.integers(1, 1 << 23, 5000, dtype=np.int64).astype(np.uint32)).view(np.float32)
    large = rng.uniform(1e37, 3.0e38, 5000).astype(np.float32)       # below FLT_MAX's tf32 rounding to inf
    edge = np.array([0.0, -0.0, 1.0, -1.0, 1 + 2.0 ** -11, 1 + 2.0 ** -10, 1 - 2.0 ** -12, 1.5 * 2.0 ** -126],
                    dtype=np.float32)
    vals = np.concatenate([normal, sub, large, edge]).astype(np.float32)
    return np.concatenate([vals, -vals])


def test_split_is_exact():
    x = _values()
    hi, lo = split_tf32(x)
    assert np.isfinite(hi).all()
    assert (hi.view(np.uint32) & np.uint32(0x1FFF) == 0).all()
    assert np.array_equal(hi + lo, x)
    assert np.array_equal(hi.astype(np.float64) + lo.astype(np.float64), x.astype(np.float64))
    normal = np.abs(x) >= np.float32(2.0 ** -126)
    assert (np.abs(lo[normal]) <= np.abs(x[normal]) * 2.0 ** -11).all()


def test_split_keeps_22_bits_when_the_tensor_core_reads_lo_as_tf32():
    x = _values()
    x = x[np.abs(x) >= 2.0 ** -100]                      # lo stays a normal number
    hi, lo = split_tf32(x)
    lo_read = (lo.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)   # the top 19 bits
    err = np.abs(hi.astype(np.float64) + lo_read.astype(np.float64) - x.astype(np.float64))
    assert (err <= np.abs(x.astype(np.float64)) * 2.0 ** -21).all()


def test_shared_memory_and_tmem_allow_two_ctas_per_sm():
    """B200: 228 KB of shared memory per SM with 1 KB reserved per CTA, 512 TMEM columns, 64 K registers."""
    assert TC_N * (TC_K + 1) * 4 + 8 * TC_N * 8 <= TC_STAGES * STAGE      # epilogue tiles reuse the stages
    assert 2 * (SMEM + 1024) <= 228 * 1024 < 3 * (SMEM + 1024)
    assert 2 * TMEM_COLS <= 512
    assert 2 * TC_THREADS * 128 <= 64 * 1024                 # __launch_bounds__(256, 2): at most 128 registers


def plan(B, K, N, tile=64, rows=32, target=148 * 4):
    """linear.cu::linear_plan (unchanged: it also sizes the scratch)."""
    tiles = math.ceil(K / tile) * math.ceil(N / tile)
    want = math.ceil(target / tiles)
    r = math.ceil(math.ceil(B / want) / rows) * rows
    return math.ceil(B / r), r


def tc_ctas(B, K, N):
    S, _ = plan(B, K, N)
    return S * math.ceil(K / TC_K) * math.ceil(N / TC_N)


def runs_on_tensor_cores(B, K, N, min_ctas=148 // 2):
    """rk_linear_wgrad's choice: the tensor-core kernel unless its grid holds fewer than min_ctas CTAs."""
    return tc_ctas(B, K, N) >= min_ctas


@pytest.mark.parametrize("B,K,N,ctas", [(8192, 82, 512, 148), (8192, 512, 256, 152), (8192, 256, 128, 128)])
def test_din_layers_fill_the_gpu(B, K, N, ctas):
    assert tc_ctas(B, K, N) == ctas and runs_on_tensor_cores(B, K, N)


@pytest.mark.parametrize("B,K,N,tc", [(8192, 66, 512, True), (8192, 128, 1, True), (8192, 50, 512, True),
                                      (1024, 96, 512, True), (1024, 512, 256, True), (1024, 256, 128, False)])
def test_bench_shapes_kernel_choice(B, K, N, tc):
    """Of bench.py's Linear shapes only DeepFM's 256 -> 128 at B = 1024 (64 CTAs) runs the SIMT kernel."""
    assert runs_on_tensor_cores(B, K, N) == tc


@pytest.mark.parametrize("B,K,N", [(B, K, N) for B in (4099, 8197) for K in (8, 95, 96, 97, 129)
                                   for N in (127, 128, 129, 257)] +
                         [(8197, 82, 512), (4099, 512, 256), (8191, 256, 129), (4097, 96, 128), (2049, 97, 129),
                          (1003, 97, 257)])
def test_gpu_tile_edge_shapes_run_on_tensor_cores(B, K, N):
    """The shapes of test_gpu_linear_wgrad_tc.py exercise the tensor-core kernel, not the SIMT one."""
    assert runs_on_tensor_cores(B, K, N)


@pytest.mark.parametrize("B,K,N", [(1, 1, 1), (37, 8, 127), (37, 129, 257), (1003, 97, 257), (8192, 82, 512),
                                   (4099, 512, 256), (65, 129, 129), (8191, 256, 129), (4097, 96, 128)])
def test_tiles_and_stages_cover_everything_once(B, K, N):
    S, rows = plan(B, K, N)
    seen_rows = np.zeros(B, dtype=np.int32)
    for s in range(S):
        row0, row_end = s * rows, min(B, (s + 1) * rows)
        for st in range(math.ceil((row_end - row0) / TC_ROWS)):
            r0 = row0 + st * TC_ROWS
            left = row_end - r0
            kmma = TC_ROWS // 8 if left >= TC_ROWS else math.ceil(left / 8)      # MMAs issued
            r = np.arange(r0, r0 + 8 * kmma)
            assert (r < row_end).sum() == min(left, TC_ROWS)                     # no live row is skipped
            seen_rows[r[r < row_end]] += 1
    assert (seen_rows == 1).all()
    seen = np.zeros((N, K), dtype=np.int32)
    for kt in range(math.ceil(K / TC_K)):
        k0 = kt * TC_K
        nk = min(TC_K, (K - k0 + 31) & ~31)                                      # the MMA's N
        assert nk % 32 == 0 and nk >= min(TC_K, K - k0)
        assert TC_ROWS * (nk // 4) <= 2 * TC_THREADS                             # X chunks: two per thread
        for nt in range(math.ceil(N / TC_N)):
            seen[nt * TC_N:(nt + 1) * TC_N, k0:k0 + nk] += 1
    assert (seen == 1).all()
