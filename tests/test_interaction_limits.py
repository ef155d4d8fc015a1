"""Width limits of the CrossNet, residual-unit and FM kernels, restated in Python (CPU only).

* Residual units (csrc/residual.cu): the shared-memory size of the forward and backward blocks, from
  the layout constants, against the 227 KiB a block may have.  Over 1 <= d, H <= 256 the backward takes
  every pair the forward takes, and the library refuses every pair the restatement refuses.
* CrossNet (csrc/concat_cross.cu) and the FM / FwFM parts (csrc/fm.cu, csrc/fwfm.cu): the vector width a
  row or an embedding is cut into and the unit / lane limits that follow from it.
* The table-gradient reductions (csrc/direct_reduce.cu, csrc/segment_reduce.cu), which
  sparse.check_table_gradients restates for the forwards.

The library is only called with shapes the restatement refuses, so no kernel may launch.  Where a GPU is
present the pointers are real device memory, so that a shape the restatement wrongly called refused runs
on valid memory and fails the test instead of the device; elsewhere they are placeholders.
tests/test_gpu_interaction_widths.py runs shapes just inside the limits on the GPU.
"""
import ctypes as C

import pytest
import torch

from rank_b200 import RankB200Error, _lib
from rank_b200.sparse import check_table_gradients

SMEM_MAX = 227 * 1024            # dynamic shared memory a block may have (kResSmemMax)
REGION = 1 << 22                 # bytes per argument buffer: the widest residual pack is ~1 MiB


# ---- residual units ------------------------------------------------------------------------------
def res_layout(d, H):
    """ResLayout: dp = roundup(d, 4), Hp = roundup(H, 8)."""
    return (d + 3) // 4 * 4, (H + 7) // 8 * 8


def res_rows(H):
    return 32 if H > 128 else 64


def res_fwd_bytes(d, H):
    """[W1^T d x Hp][b1 Hp][W2^T Hp x dp][b2 dp] + X [dp][rows+4] + Hs [Hp][rows+4]."""
    dp, Hp = res_layout(d, H)
    return 4 * (d * Hp + Hp + Hp * dp + dp + (dp + Hp) * (res_rows(H) + 4))


def res_bwd_bytes(d, H, rows):
    """[W1^T d x Hp | b1 Hp, later W1 Hp x dp][W2 d x Hp] + X, G [dp][rows+4] + Hs [Hp][rows+4]."""
    dp, Hp = res_layout(d, H)
    return 4 * (max(d * Hp + Hp, Hp * dp) + d * Hp + (2 * dp + Hp) * (rows + 4))


def res_bwd_rows(d, H):
    """The backward's tile height: res_rows(H), halved while the block does not fit (down to 4)."""
    rows = res_rows(H)
    while rows > 4 and res_bwd_bytes(d, H, rows) > SMEM_MAX:
        rows //= 2
    return rows


def res_fwd_ok(d, H):
    return res_fwd_bytes(d, H) <= SMEM_MAX


def res_bwd_ok(d, H):
    return res_bwd_bytes(d, H, res_bwd_rows(d, H)) <= SMEM_MAX


def res_widest_d(H):
    return max(d for d in range(1, 257) if res_fwd_ok(d, H))


PAIRS = [(d, H) for d in range(1, 257) for H in range(1, 257)]


# ---- CrossNet and FM -----------------------------------------------------------------------------
def vec_of(*values):
    """Widest of 4 / 2 / 1 floats dividing every value (pick_vec; a row's pointers are 16-byte aligned)."""
    v = 4
    while v > 1 and any(x % v for x in values):
        v //= 2
    return v


def crossnet_fwd_refusal(n_dense, dims):
    """The words of rk_crossnet_fwd's refusal of this tiling, or None where it takes it."""
    offs = [n_dense + sum(dims[:f]) for f in range(len(dims))]
    d = n_dense + sum(dims)
    if d > 512:
        return "wider than 512"
    if d // vec_of(n_dense, *dims, *offs) > 128:
        return "exceeds 128 units"
    return None


def crossnet_bwd_ok(d):
    return d // vec_of(d) <= 128


def fm_lanes_ok(D):
    return D // vec_of(D) <= 32


# ---- calling the library -------------------------------------------------------------------------
@pytest.fixture(scope="module")
def addr():
    if torch.cuda.is_available():
        buf = torch.zeros(16 * REGION // 4, dtype=torch.float32, device="cuda")
        yield lambda k: buf.data_ptr() + k * REGION
        torch.cuda.synchronize()
    else:
        yield lambda k: (1 << 24) * (k + 1)


def _refused(rc, *words):
    msg = _lib.load().rk_last_error().decode()
    assert rc < 0, (rc, msg)
    for w in words:
        assert w in msg, msg


def _fields(addr, dims, first_off):
    arr = (_lib.RkField * max(len(dims), 1))()
    off = first_off
    for f, dim in enumerate(dims):
        arr[f] = _lib.RkField(addr(0), addr(1), 1, dim, off)   # one-row tables, every index 0
        off += dim
    return arr


# ---- residual units ------------------------------------------------------------------------------
def test_resunits_backward_takes_every_pair_the_forward_takes():
    fwd = [p for p in PAIRS if res_fwd_ok(*p)]
    assert all(res_bwd_ok(*p) for p in fwd)
    # the tiles are whole micro-tiles of tile_gemm (4 rows), and no narrower than 16
    assert all(res_bwd_rows(*p) % 4 == 0 and res_bwd_rows(*p) >= 16 for p in fwd)
    # the benchmark's shape keeps its tile height, and the reference's default width at H = 128 runs
    assert res_bwd_rows(50, 128) == 64
    assert res_fwd_ok(128, 128) and res_bwd_ok(128, 128)
    # the forward's limit is the block's shared memory, not d, H <= 256: d = 89 does not fit at H = 256
    assert res_widest_d(256) == 88 and not res_fwd_ok(89, 256)


def test_resunits_library_refuses_what_the_restatement_refuses(addr):
    lib = _lib.load()
    refused_fwd = [p for p in PAIRS if not res_fwd_ok(*p)]
    refused_bwd = [p for p in PAIRS if not res_bwd_ok(*p)]
    assert refused_fwd and refused_bwd
    for d, H in refused_fwd:
        rc = lib.rk_resunits_fwd(None, 0, addr(0), d, addr(1), 1, H, 1, addr(2), addr(3), None)
        _refused(rc, "resunits_fwd", "shared memory")
    for d, H in refused_bwd:
        rc = lib.rk_resunits_bwd(addr(2), addr(1), 1, H, d, 1, addr(4), addr(5), None)
        _refused(rc, "resunits_bwd", "shared memory")


@pytest.mark.parametrize("d,H", [(257, 8), (8, 257), (8, 0)])
def test_resunits_widths_outside_1_to_256_are_refused(addr, d, H):
    lib = _lib.load()
    _refused(lib.rk_resunits_fwd(None, 0, addr(0), d, addr(1), 1, H, 1, addr(2), addr(3), None), "[1, 256]")
    _refused(lib.rk_resunits_bwd(addr(2), addr(1), 1, H, d, 1, addr(4), addr(5), None), "[1, 256]")


# ---- CrossNet ------------------------------------------------------------------------------------
def _cross_layouts():
    """Every row width up to 520 floats, ending in a field of 1 to 4 columns after a dense block."""
    for d in range(1, 521):
        for tail in (1, 2, 3, 4):
            if tail <= d:
                yield d - tail, [tail]


def test_crossnet_backward_takes_every_row_the_forward_takes():
    for n_dense, dims in _cross_layouts():
        if crossnet_fwd_refusal(n_dense, dims) is None:
            assert crossnet_bwd_ok(n_dense + sum(dims)), (n_dense, dims)


def test_crossnet_library_refuses_what_the_restatement_refuses(addr):
    lib = _lib.load()
    refused = 0
    for n_dense, dims in _cross_layouts():
        words = crossnet_fwd_refusal(n_dense, dims)
        if words is None:
            continue
        refused += 1
        rc = lib.rk_crossnet_fwd(_fields(addr, dims, n_dense), len(dims), addr(2), n_dense, addr(3), addr(4), 1, 1,
                                 addr(5), addr(6), addr(7), None)
        _refused(rc, "concat", words)
    assert refused
    for d in range(1, 1100):
        if not crossnet_bwd_ok(d):
            rc = lib.rk_crossnet_bwd(addr(2), addr(3), addr(4), 1, d, 1, addr(5), addr(6), addr(7), None)
            _refused(rc, "crossnet_bwd", "too wide")


def test_crossnet_limits_at_the_kernel_instantiations():
    assert crossnet_fwd_refusal(16, [1, 32, 32, 32, 15]) is None          # 128 units of 1 float
    assert crossnet_fwd_refusal(16, [1, 32, 32, 32, 16]) == "exceeds 128 units"
    assert crossnet_fwd_refusal(16, [128, 128, 128, 112]) is None         # 128 units of 4 floats
    assert crossnet_fwd_refusal(16, [128, 128, 128, 116]) == "wider than 512"


# ---- FM / FwFM -----------------------------------------------------------------------------------
def test_fm_lane_limit():
    assert [D for D in range(1, 140) if fm_lanes_ok(D) and D > 32 and D % 2] == []
    assert fm_lanes_ok(62) and not fm_lanes_ok(66) and fm_lanes_ok(128) and not fm_lanes_ok(132)


@pytest.mark.parametrize("F", [1, 2])
def test_fm_library_refuses_what_the_restatement_refuses(addr, F):
    lib = _lib.load()
    firsts = (C.c_void_p * F)(*[addr(8)] * F)
    for D in range(1, 300):
        if fm_lanes_ok(D):
            continue
        second = (_lib.RkField * F)(*[_lib.RkField(addr(0), addr(1), 1, D, f * D) for f in range(F)])
        if F == 1:
            _refused(lib.rk_deepfm_fwd(second, firsts, F, 1, addr(2), addr(3), addr(4), addr(7), None),
                     "deepfm_fwd", "too wide")
            _refused(lib.rk_deepfm_bwd(addr(2), addr(5), addr(6), F, D, 1, addr(9), None), "deepfm_bwd", "too wide")
        else:
            _refused(lib.rk_fwfm_fwd(second, firsts, addr(3), addr(4), F, 1, addr(2), addr(5), addr(7), None),
                     "fwfm_fwd", "too wide")
            _refused(lib.rk_fwfm_bwd(addr(2), addr(5), addr(6), addr(3), F, D, 1, addr(9), addr(10), addr(11),
                                     addr(12), None), "fwfm_bwd", "too wide")


# ---- table-gradient reductions -------------------------------------------------------------------
GRAD_LAYOUTS = [(dim, off, off + dim + extra) for dim in range(1, 140) for off in (0, 1, 2, 3, 16, 17, 18)
                for extra in (0, 1, 2, 3)]


def _grad_refused(dim, off, ld):
    try:
        check_table_gradients([(dim, off, ld)], "test")
    except RankB200Error as e:
        assert "at most" in str(e)
        return True
    return False


def test_table_gradient_check_matches_the_reduction_lanes():
    for dim, off, ld in GRAD_LAYOUTS:
        assert _grad_refused(dim, off, ld) == (dim > 32 * vec_of(dim, off, ld)), (dim, off, ld)
    # a 64-wide field after 16 dense columns and before a 1-wide one: an 81-float row, 1 float per lane
    assert _grad_refused(64, 16, 81) and not _grad_refused(64, 16, 80) and not _grad_refused(32, 17, 81)
    # FM / FwFM: F second-order and F first-order gradient tables in one reduction
    for F, ok in ((16, True), (17, False), (24, False)):
        tables = [(8, f * 8, F * 8) for f in range(F)] + [(1, 0, 1)] * F
        try:
            check_table_gradients(tables, "FM part")
            assert ok
        except RankB200Error as e:
            assert not ok and "RK_MAX_TABLES" in str(e)


def test_reductions_refuse_what_the_check_refuses(addr):
    lib = _lib.load()
    for dim, off, ld in GRAD_LAYOUTS:
        if not _grad_refused(dim, off, ld):
            continue
        g = addr(2) + 4 * off
        direct = (_lib.RkDirectTable * 1)(_lib.RkDirectTable(addr(1), g, ld, addr(3), 1, 1, dim, 0))
        _refused(lib.rk_embgrad_direct_reduce(direct, 1, addr(7), None), "direct_reduce: table 0")
        tabs = (_lib.RkGradTable * 1)(_lib.RkGradTable(g, ld, addr(3), dim, 0))
        n, rows = (C.c_int64 * 1)(1), (C.c_int64 * 1)(1)
        ws = lib.rk_reduce_workspace_bytes(n, 1, tabs, 1)
        _refused(lib.rk_embgrad_segment_reduce(addr(4), addr(5), n, rows, 1, tabs, 1, addr(6), ws, None),
                 "segment_reduce", "too wide")
