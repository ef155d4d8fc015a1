"""The tensor-core entry points refuse NULL operand tiles before they touch the device (CPU only).

The weight tiles that the forward's prologue writes and every CTA fetches by bulk copy are the only
way these kernels get their weights, so a NULL buffer is an argument error, not a request for another
path.  Every other argument is valid: host-side structs and placeholder device addresses that are
never dereferenced because the call is refused first.  Skipped where a GPU is present, so that a
broken check could never launch a kernel on those addresses.
"""
import ctypes as C

import pytest
import torch

from rank_b200 import _lib

pytestmark = pytest.mark.skipif(torch.cuda.is_available(),
                                reason="placeholder device addresses: only run where no kernel can launch")

ADDR = 1 << 24          # placeholder device addresses: 128-byte aligned, distinct, never dereferenced
B, D = 4, 16


def _addr(k):
    return ADDR * (k + 1)


def _fields(F, rows=10):
    arr = (_lib.RkField * F)()
    for f in range(F):
        arr[f] = _lib.RkField(_addr(10 + f), _addr(40 + f), rows, D, f * D)
    return arr


def _assert_refused(rc, what):
    msg = _lib.load().rk_last_error().decode()
    assert rc < 0, (what, rc, msg)
    assert "tiles" in msg, (what, msg)


def test_afm_tc_fwd_refuses_null_tiles():
    lib = _lib.load()
    F, A = 3, 8
    rc = lib.rk_afm_tc_fwd(_fields(F), F, _addr(0), _addr(1), _addr(2), _addr(3), A, B, _addr(4), None,
                           _addr(5), None)
    _assert_refused(rc, "rk_afm_tc_fwd")


def test_afm_tc_bwd_refuses_null_tiles():
    lib = _lib.load()
    F, A = 3, 8
    g_w1 = _addr(6)
    g_b1 = g_w1 + 4 * A * D             # g_w1 | g_b1 | g_w2 | g_b2: one contiguous buffer
    g_w2 = g_b1 + 4 * A
    g_b2 = g_w2 + 4 * A
    n_ctas = 1                          # B = 4 samples fit one tile of 16
    rc = lib.rk_afm_tc_bwd(_fields(F), F, _addr(0), _addr(1), _addr(2), _addr(3), A, B, _addr(4), _addr(5),
                           g_w1, g_b1, g_w2, g_b2, _addr(7), n_ctas, None, _addr(8), None)
    _assert_refused(rc, "rk_afm_tc_bwd")


def test_din_tensor_core_fwd_refuses_null_tiles():
    lib = _lib.load()
    T = 8
    a = _lib.RkDinArgs()
    a.cat, a.n_cat, a.n_dense = None, 0, 0
    a.target = _lib.RkField(_addr(0), _addr(1), 10, D, 0)
    a.history = _lib.RkField(_addr(2), _addr(3), 10, D, 0)
    a.hist_len = _addr(4)
    a.T = T
    a.att_off, a.width, a.l2_from, a.use_softmax = D, 2 * D, 0, 0
    a.precision = 1                     # RK_DIN_BF16_TENSOR
    a.mlp = _addr(5)
    a.B = B
    a.mlp_tiles = None
    rc = lib.rk_din_fwd(C.byref(a), _addr(6), _addr(7), _addr(8), _addr(9), _addr(10), None)
    _assert_refused(rc, "rk_din_fwd")
