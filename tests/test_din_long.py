"""DIN's fp32 activation unit at every history width, and batches with no history at all (CPU only).

* The C ABI's argument checks for the history width: a negative width and the tensor-core unit above 128
  positions are refused before any CUDA call; width 0 and widths above 128 pass the checks (with B = 0 the
  entry points return before any launch).  Placeholder device addresses, never dereferenced, as in
  test_abi_tiles.py; skipped where a GPU is present.
* A numpy restatement of the fp32 kernels' tile planner (plan_tile in csrc/din.cu): every live (b, t) row is
  covered exactly once, in tiles of at most 128 rows, and samples of at most 128 positions are packed whole,
  as many to a tile as fit (so at T <= 128 a tile holds whole samples only).
"""
import ctypes as C

import numpy as np
import pytest
import torch

from rank_b200 import _lib

K_ROWS, K_SAMPLES = 128, 8
ADDR = 1 << 24
D = 16
no_gpu = pytest.mark.skipif(torch.cuda.is_available(),
                            reason="placeholder device addresses: only run where no kernel can launch")


def _addr(k):
    return ADDR * (k + 1)


def _args(T, B, precision=0, history=True):
    a = _lib.RkDinArgs()
    a.cat, a.n_cat, a.n_dense = None, 0, 0
    a.target = _lib.RkField(_addr(0), _addr(1), 10, D, 0)
    a.history = _lib.RkField(_addr(2), _addr(3), 10, D, 0) if history else _lib.RkField(None, None, 0, D, 0)
    a.hist_len = _addr(4)
    a.T = T
    a.att_off, a.width, a.l2_from, a.use_softmax = D, 2 * D, 0, 1
    a.precision = precision
    a.mlp = _addr(5)
    a.B = B
    a.mlp_tiles = _addr(11) if precision == 1 else None
    return a


def _fwd(a):
    return _lib.load().rk_din_fwd(C.byref(a), _addr(6), _addr(7), _addr(8), _addr(9), _addr(10), None)


def _bwd(a):
    return _lib.load().rk_din_bwd(C.byref(a), _addr(6), _addr(7), _addr(8), _addr(9), _addr(12), _addr(13),
                                  _addr(14), _addr(15), _addr(10), None)


def _refused(rc, *words):
    msg = _lib.load().rk_last_error().decode()
    assert rc < 0, (rc, msg)
    for w in words:
        assert w in msg, msg


@no_gpu
@pytest.mark.parametrize("call", [_fwd, _bwd])
def test_negative_width_is_refused(call):
    _refused(call(_args(-1, 4)), "negative")


@no_gpu
@pytest.mark.parametrize("call", [_fwd, _bwd])
@pytest.mark.parametrize("T", [129, 300, 5000])
def test_tensor_core_unit_above_128_positions_is_refused(call, T):
    _refused(call(_args(T, 4, precision=1)), "RK_DIN_FP32", str(T))


@no_gpu
@pytest.mark.parametrize("call", [_fwd, _bwd])
@pytest.mark.parametrize("T", [0, 129, 1000, 4096, 100000])
def test_fp32_accepts_any_width(call, T):
    assert call(_args(T, 0)) == 0, _lib.load().rk_last_error().decode()


@no_gpu
@pytest.mark.parametrize("call", [_fwd, _bwd])
@pytest.mark.parametrize("precision", [0, 1])
def test_width_zero_needs_no_history_pointers(call, precision):
    assert call(_args(0, 0, precision, history=False)) == 0, _lib.load().rk_last_error().decode()
    _refused(call(_args(1, 0, precision, history=False)), "NULL")


# ---- the tile planner ---------------------------------------------------------------------------
def plan_tile(lens, s_begin, t_begin):
    """plan_tile (csrc/din.cu): segments [(sample, t0, n)] of the tile and the next cursor."""
    rows, s, t0, segs = 0, s_begin, t_begin, []
    while s < len(lens):
        rem = lens[s] - t0
        if rem <= K_ROWS - rows:
            segs.append((s, t0, rem))
            rows += rem
            s, t0 = s + 1, 0
            continue
        if lens[s] <= K_ROWS or rows == K_ROWS:
            break
        segs.append((s, t0, K_ROWS - rows))
        t0 += K_ROWS - rows
        rows = K_ROWS
        break
    return segs, rows, s, t0


def plan_cta(lens):
    tiles, s, t = [], 0, 0
    while s < len(lens):
        segs, rows, s, t = plan_tile(lens, s, t)
        tiles.append((segs, rows))
    return tiles


def plan_short(lens):
    """Whole samples while they fit: how samples of at most 128 positions must be packed."""
    tiles, s = [], 0
    while s < len(lens):
        rows, e = 0, s
        while e < len(lens) and rows + lens[e] <= K_ROWS:
            rows += lens[e]
            e += 1
        tiles.append((list(range(s, e)), rows))
        s = e
    return tiles


def _row_map(segs):
    """row_map: tile row -> (sample, t)."""
    r0 = np.cumsum([0] + [n for _, _, n in segs])
    out = []
    for m in range(r0[-1]):
        j = 0
        while j + 1 < len(segs) and m >= r0[j + 1]:
            j += 1
        out.append((segs[j][0], segs[j][1] + m - r0[j]))
    return out


def _length_cases():
    rng = np.random.default_rng(5)
    yield [0] * K_SAMPLES
    yield [0, 1, 127, 128, 129, 255, 256, 257]
    yield [4096] * K_SAMPLES
    yield [128] * K_SAMPLES
    yield [129, 0, 0, 129, 1, 300, 0, 5]
    for T in (50, 128, 129, 200, 256, 1000, 4096):
        for n in (1, 3, K_SAMPLES):
            for _ in range(40):
                lens = rng.integers(1, T + 1, n) * (rng.random(n) >= 0.3)
                yield [int(v) for v in lens]


def test_every_live_row_is_covered_once_in_tiles_of_at_most_128():
    for lens in _length_cases():
        tiles = plan_cta(lens)
        seen = []
        for segs, rows in tiles:
            assert 0 <= rows <= K_ROWS
            assert rows == sum(n for _, _, n in segs)
            assert len(segs) <= K_SAMPLES
            assert [s for s, _, _ in segs] == list(range(segs[0][0], segs[0][0] + len(segs)))
            for s, t0, n in segs:
                if lens[s] <= K_ROWS:
                    assert (t0, n) == (0, lens[s]), "a short sample was split"
            rm = _row_map(segs)
            assert len(rm) == rows
            seen += rm
        want = [(s, t) for s in range(len(lens)) for t in range(lens[s])]
        assert seen == want, lens
        # every sample appears, and its last segment ends at its length (where the pooling finishes it)
        last = {}
        for segs, _ in tiles:
            for s, t0, n in segs:
                last[s] = t0 + n
        assert last == {s: lens[s] for s in range(len(lens))}
        # a tile is full unless the next sample (short) does not fit or the CTA's samples ran out
        for (segs, rows), (nxt, _) in zip(tiles, tiles[1:]):
            s, t0, _ = nxt[0]
            if t0 == 0:
                assert lens[s] <= K_ROWS and rows + lens[s] > K_ROWS or rows == K_ROWS


def test_short_samples_are_packed_as_the_existing_planner_packs_them():
    rng = np.random.default_rng(9)
    for _ in range(500):
        n = int(rng.integers(1, K_SAMPLES + 1))
        lens = [int(v) for v in rng.integers(0, K_ROWS + 1, n)]
        long_tiles = [([s for s, _, _ in segs], rows) for segs, rows in plan_cta(lens)]
        assert long_tiles == plan_short(lens), lens


def test_long_sample_tiles():
    # a 300-position sample after a 100-position one: 100 + 28 | 128 | 128 - 28 = 100 + the next sample
    segs = [s for s, _ in plan_cta([100, 300, 20])]
    assert segs == [[(0, 0, 100), (1, 0, 28)], [(1, 28, 128)], [(1, 156, 128)], [(1, 284, 16), (2, 0, 20)]]
