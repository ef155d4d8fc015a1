"""BST sequences longer than one 128-row tile (fp32 block), CPU only.

* The C ABI's argument checks for the sequence length: fp32 accepts any T >= 1 (with B = 0 the entry
  points return before any launch), the tensor-core block above 128 positions and T = 0 are refused
  before any CUDA call.  Placeholder device addresses, never dereferenced, as in test_din_long.py;
  skipped where a GPU is present.
* A float64 restatement of the long kernels' decomposition (bst_fwd_long_kernel / bst_bwd_long_kernel in
  csrc/bst.cu): query and key chunks of 128, the online softmax over key chunks, and the backward's
  per-(query chunk, key chunk) contributions to g_x, the position table and the k / v weights, added in
  the kernels' loop order.  It must equal autograd through oracle.interactions.bst_transformer_block.
"""
import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

from rank_b200 import _lib
from oracle import interactions as X

K = 128
D = 16
ADDR = 1 << 24
no_gpu = pytest.mark.skipif(torch.cuda.is_available(),
                            reason="placeholder device addresses: only run where no kernel can launch")
_NAMES = ("pos", "wq", "bq", "wk", "bk", "wv", "bv", "wo", "bo", "ln1_g", "ln1_b", "w1", "b1", "w2", "b2",
          "ln2_g", "ln2_b")


def _blk(precision):
    blk = _lib.RkBstBlock()
    for i, n in enumerate(_NAMES):
        setattr(blk, n, ADDR * (i + 1))
    blk.dropout_p = 0.0
    blk.precision = precision
    return blk


def _fwd(T, B, precision):
    return _lib.load().rk_bst_block_fwd(C.byref(_blk(precision)), 4, ADDR * 30, ADDR * 31, 100, None,
                                        ADDR * 32, B, T, ADDR * 33, None, D, 0, ADDR * 34, None)


def _bwd(T, B, precision):
    lib = _lib.load()
    n_ctas = lib.rk_bst_bwd_ctas(B, T, precision)
    return lib.rk_bst_block_bwd(C.byref(_blk(precision)), 4, ADDR * 30, ADDR * 31, 100, None, ADDR * 32, B, T,
                                ADDR * 33, None, D, 0, ADDR * 35, ADDR * 36, ADDR * 37, n_ctas, ADDR * 34, None)


def _refused(rc, *words):
    msg = _lib.load().rk_last_error().decode()
    assert rc < 0, (rc, msg)
    for w in words:
        assert w in msg, msg


@no_gpu
@pytest.mark.parametrize("call", [_fwd, _bwd])
@pytest.mark.parametrize("T", [129, 1000, 4096])
def test_fp32_accepts_any_length(call, T):
    assert call(T, 0, _lib.BST_FP32) == 0, _lib.load().rk_last_error().decode()


@no_gpu
@pytest.mark.parametrize("call", [_fwd, _bwd])
@pytest.mark.parametrize("T", [129, 300, 5000])
def test_tensor_core_block_above_128_positions_is_refused(call, T):
    _refused(call(T, 4, _lib.BST_BF16_TENSOR), "RK_BST_FP32", str(T))


@no_gpu
@pytest.mark.parametrize("call", [_fwd, _bwd])
@pytest.mark.parametrize("precision", [0, 1])
def test_length_zero_is_refused(call, precision):
    _refused(call(0, 4, precision), "sequence length 0")


def test_grad_floats_cover_any_length():
    lib = _lib.load()
    for T in (1, 128, 129, 1000, 4096):
        assert lib.rk_bst_grad_floats(T) == T * 16 + 1696


# ---- float64 restatement of the chunked algorithm ---------------------------------------------------
def _params(T, seed):
    gen = torch.Generator().manual_seed(seed)
    p = {"position_embedding.weight": torch.randn(T + 1, D, generator=gen)}
    for n in ("w_q", "w_k", "w_v", "w_o", "ffn.0", "ffn.3"):
        p[n + ".weight"] = torch.randn(D, D, generator=gen) / 4
        p[n + ".bias"] = torch.randn(D, generator=gen) / 4
    for n in ("norm1", "norm2"):
        p[n + ".weight"] = 1 + torch.randn(D, generator=gen) / 4
        p[n + ".bias"] = torch.randn(D, generator=gen) / 4
    return {k: v.double() for k, v in p.items()}


def _tail(ctx, qk, p):
    """The per-row rest of the block: w_o, LayerNorm 1, FFN, LayerNorm 2."""
    o1 = F.layer_norm(qk + F.linear(ctx, p["w_o.weight"], p["w_o.bias"]), (D,), p["norm1.weight"], p["norm1.bias"])
    h = F.leaky_relu(F.linear(o1, p["ffn.0.weight"], p["ffn.0.bias"]), 0.01)
    return F.layer_norm(o1 + F.linear(h, p["ffn.3.weight"], p["ffn.3.bias"]), (D,), p["norm2.weight"],
                        p["norm2.bias"])


def chunked_block(x, lens, p, H, g_y):
    """(y, g_x, {parameter: gradient}) of the block as the long kernels compute it."""
    B, T, _ = x.shape
    DH = D // H
    scale = 1.0 / math.sqrt(DH)
    Wq, Wk, Wv = p["w_q.weight"], p["w_k.weight"], p["w_v.weight"]
    qk_all = x + p["position_embedding.weight"][:T]
    heads = lambda a: a.view(B, a.shape[1], H, DH).transpose(1, 2)      # [B, H, rows, DH]
    tail_p = {k: v.clone().requires_grad_() for k, v in p.items()
              if k.startswith(("w_o", "norm", "ffn"))}
    y = torch.empty(B, T, D, dtype=torch.float64)
    g_x = torch.zeros(B, T, D, dtype=torch.float64)
    g_pos = torch.zeros(T + 1, D, dtype=torch.float64)
    g = {n: torch.zeros_like(p[n]) for n in ("w_q.weight", "w_q.bias", "w_k.weight", "w_k.bias", "w_v.weight",
                                             "w_v.bias")}
    written = torch.zeros(B, T, dtype=torch.bool)

    def keys(u0):
        """k, v, qk, x of a key chunk (recomputed per pair in the kernels), and its live mask [B, n]."""
        u = slice(u0, min(u0 + K, T))
        qk_u, x_u = qk_all[:, u], x[:, u]
        live = torch.arange(u0, u.stop).unsqueeze(0) < lens.unsqueeze(1)
        return F.linear(qk_u, Wk, p["w_k.bias"]), F.linear(x_u, Wv, p["w_v.bias"]), qk_u, x_u, live, u

    for t0 in range(0, T, K):
        t = slice(t0, min(t0 + K, T))
        qk = qk_all[:, t]
        q = F.linear(qk, Wq, p["w_q.bias"])
        qh = heads(q)
        rows = qk.shape[1]
        m = torch.full((B, H, rows, 1), -math.inf, dtype=torch.float64)
        l = torch.zeros(B, H, rows, 1, dtype=torch.float64)
        ctx = torch.zeros(B, H, rows, DH, dtype=torch.float64)
        for u0 in range(0, T, K):
            k, v, _, _, live, _ = keys(u0)
            has = (lens > u0).view(B, 1, 1, 1)           # samples with a live key in this chunk
            lv = live.view(B, 1, 1, -1)
            s = torch.where(lv, qh @ heads(k).transpose(-1, -2) * scale, -math.inf)
            mc = torch.where(has, torch.maximum(m, s.amax(-1, keepdim=True)), m)
            alpha = torch.where(has, torch.exp(m - mc), 1.0)
            pr = torch.where(lv, torch.exp(s - torch.where(has, mc, 0.0)), 0.0)
            l = l * alpha + pr.sum(-1, keepdim=True)
            ctx = ctx * alpha + pr @ heads(v)
            m = mc
        ctx = ctx / l
        # the rows' tail and its backward: dctx, and dz1 (the residual into qk)
        ctx_leaf = ctx.transpose(1, 2).reshape(B, rows, D).detach().requires_grad_()
        qk_leaf = qk.detach().requires_grad_()
        y_rows = _tail(ctx_leaf, qk_leaf, tail_p)
        y[:, t] = y_rows.detach()
        y_rows.backward(g_y[:, t])
        dctx, dz1 = heads(ctx_leaf.grad), qk_leaf.grad
        delta = (dctx * ctx).sum(-1, keepdim=True)
        dq = torch.zeros(B, H, rows, DH, dtype=torch.float64)
        for u0 in range(0, T, K):
            k, v, qk_u, x_u, live, u = keys(u0)
            if not bool((lens > u0).any()):
                continue
            lv = live.view(B, 1, 1, -1)
            kh, vh = heads(k), heads(v)
            s = qh @ kh.transpose(-1, -2) * scale
            a = torch.where(lv, torch.exp(s - m) / l, 0.0)
            dS = a * (dctx @ vh.transpose(-1, -2) - delta) * scale
            dq = dq + dS @ kh
            dk = (dS.transpose(-1, -2) @ qh).transpose(1, 2).reshape(B, -1, D)     # this pair's contribution
            dv = (a.transpose(-1, -2) @ dctx).transpose(1, 2).reshape(B, -1, D)
            dk, dv = dk * live.unsqueeze(-1), dv * live.unsqueeze(-1)
            dpos = dk @ Wk
            g_pos[u] += dpos.sum(0)
            contrib = dpos + dv @ Wv
            g_x[:, u] = torch.where(written[:, u].unsqueeze(-1), g_x[:, u] + contrib,
                                    torch.where(live.unsqueeze(-1), contrib, g_x[:, u]))
            written[:, u] |= live
            g["w_k.weight"] += torch.einsum("bun,buk->nk", dk, qk_u)
            g["w_k.bias"] += dk.sum((0, 1))
            g["w_v.weight"] += torch.einsum("bun,buk->nk", dv, x_u)
            g["w_v.bias"] += dv.sum((0, 1))
        dq = dq.transpose(1, 2).reshape(B, rows, D)
        dqk = dz1 + dq @ Wq
        g_pos[t] += dqk.sum(0)
        g_x[:, t] = torch.where(written[:, t].unsqueeze(-1), g_x[:, t] + dqk, dqk)
        written[:, t] = True
        g["w_q.weight"] += torch.einsum("btn,btk->nk", dq, qk)
        g["w_q.bias"] += dq.sum((0, 1))
    g["position_embedding.weight"] = g_pos
    g.update({k: v.grad for k, v in tail_p.items()})
    return y, g_x, g


@pytest.mark.parametrize("T,H", [(129, 4), (300, 1), (300, 16), (1000, 2)])
def test_chunked_decomposition_equals_autograd_through_the_oracle(T, H):
    lens = torch.tensor([min(n, T) for n in (1, 127, 128, 129, 255, 256, 257, T)])
    B = len(lens)
    gen = torch.Generator().manual_seed(T + H)
    x = torch.randn(B, T, D, generator=gen, dtype=torch.float64)
    g_y = torch.randn(B, T, D, generator=gen, dtype=torch.float64)
    p = _params(T, T)
    y, g_x, grads = chunked_block(x, lens, p, H, g_y)

    pr = {k: v.clone().requires_grad_() for k, v in p.items()}
    xr = x.clone().requires_grad_()
    pad = torch.arange(T).expand(B, T) >= lens.unsqueeze(1)
    yr = X.bst_transformer_block(xr, pad, pr, H)
    yr.backward(g_y)
    assert torch.allclose(y, yr.detach(), rtol=0, atol=1e-12), float((y - yr).abs().max())
    assert torch.allclose(g_x, xr.grad, rtol=0, atol=1e-12), float((g_x - xr.grad).abs().max())
    assert set(grads) == set(pr)
    for k, v in pr.items():
        err = float((grads[k] - v.grad).abs().max())
        assert err <= 1e-12 * max(1.0, float(v.grad.abs().max())), (k, err)
