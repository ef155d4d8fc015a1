"""Fused tower layers (SURVEY 8(f) item 3: "tower BN/Dice").

The DNN towers stay the reference's torch modules — same ModuleList, same parameters, buffers and
`state_dict` keys.  `run_tower(layers, x)` walks that list exactly as the reference's
`for layer in self.fcn: net = layer(net)` does, but where it meets the pattern

    Dice(units)  [-> nn.BatchNorm1d(units)]           (DIN/din.py:26-36, 272-285)

or

    nn.BatchNorm1d(units) -> nn.ReLU() | nn.LeakyReLU(slope)    (DeepFM/deepfm.py:100-110, BST/bst.py:203-214)

in training mode on CUDA it runs both modules in one CUDA kernel per direction (csrc/tower.cu),
reading the modules' own parameters and updating their running statistics in place.  An nn.Linear
with at least LINEAR_MIN_OUT outputs keeps torch's forward and input gradient, and takes its weight
and bias gradients from one csrc/linear.cu call.  Anything else (eval mode, other layers,
momentum=None, batches below MIN_BATCH, or above 16384 for the normalisation pairs) runs the modules
themselves.
Set `rank_b200.tower.FUSED = False` to always run the modules.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib

FUSED = True
# Below this batch size the modules run as they are: batch statistics over a few dozen rows make every
# gradient a difference of near-equal sums, and the parity bar against the reference (1e-5) is then
# decided by which fp32 summation order one happens to share with ATen.
MIN_BATCH = 256
# A Linear with fewer than 64 outputs keeps torch's weight gradient: csrc/linear.cu's 128-output tile is then
# mostly padding (BST's final Linear(128, 1) at B = 8192: 24.8 µs against torch's 10.3 µs, scripts/bench_mm.py
# on an NVIDIA B200 at its 1000 W power limit, max SM clock 1965 MHz, L2 warm).
LINEAR_MIN_OUT = 64


class _DiceBn(torch.autograd.Function):
    """(x, alpha, gamma, beta) -> z;  bn1 = Dice.bn (affine=False), bn2 = the following BatchNorm1d or None."""

    @staticmethod
    def forward(ctx, x, alpha, gamma, beta, bn1, bn2):
        lib = _lib.load()
        x = _lib.require_cuda(x, "dice input", torch.float32)
        alpha = _lib.require_cuda(alpha, "Dice.alpha", torch.float32)
        B, U = x.shape
        z = torch.empty_like(x)
        stats = torch.empty(4, U, dtype=torch.float32, device=x.device)

        def running(bn):
            if bn is None or not bn.track_running_stats:
                return None, None, None
            return bn.running_mean.data_ptr(), bn.running_var.data_ptr(), bn.num_batches_tracked.data_ptr()
        rm1, rv1, nb1 = running(bn1)
        rm2, rv2, nb2 = running(bn2)
        rc = lib.rk_dice_bn_fwd(x.data_ptr(), B, U, alpha.data_ptr(), bn1.eps,
                                _lib.ptr(gamma), _lib.ptr(beta), bn2.eps if bn2 is not None else 0.0,
                                bn1.momentum, rm1, rv1, nb1,
                                bn2.momentum if bn2 is not None else 0.0, rm2, rv2, nb2,
                                z.data_ptr(), stats.data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "rk_dice_bn_fwd")
        ctx.save_for_backward(x, alpha, gamma, stats)
        return z

    @staticmethod
    def backward(ctx, g_z):
        lib = _lib.load()
        x, alpha, gamma, stats = ctx.saved_tensors
        B, U = x.shape
        g_z = _lib.require_cuda(g_z, "g_z", torch.float32)
        g_x = torch.empty_like(x)
        g_par = torch.empty(3, U, dtype=torch.float32, device=x.device)     # d alpha | d gamma | d beta
        rc = lib.rk_dice_bn_bwd(x.data_ptr(), g_z.data_ptr(), B, U, alpha.data_ptr(), _lib.ptr(gamma),
                                stats.data_ptr(), g_x.data_ptr(), g_par[0].data_ptr(), g_par[1].data_ptr(),
                                g_par[2].data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "rk_dice_bn_bwd")
        has_bn2 = gamma is not None
        return g_x, g_par[0], (g_par[1] if has_bn2 else None), (g_par[2] if has_bn2 else None), None, None


class _BnAct(torch.autograd.Function):
    """(x, gamma, beta) -> act(batchnorm(x));  slope: 0 = ReLU, LeakyReLU's negative_slope otherwise."""

    @staticmethod
    def forward(ctx, x, gamma, beta, bn, slope):
        lib = _lib.load()
        x = _lib.require_cuda(x, "batch-norm input", torch.float32)
        gamma = _lib.require_cuda(gamma, "BatchNorm1d.weight", torch.float32)
        beta = _lib.require_cuda(beta, "BatchNorm1d.bias", torch.float32)
        B, U = x.shape
        z = torch.empty_like(x)
        stats = torch.empty(2, U, dtype=torch.float32, device=x.device)
        track = bn.track_running_stats
        rc = lib.rk_bn_act_fwd(x.data_ptr(), B, U, gamma.data_ptr(), beta.data_ptr(), bn.eps, bn.momentum,
                               bn.running_mean.data_ptr() if track else None,
                               bn.running_var.data_ptr() if track else None,
                               bn.num_batches_tracked.data_ptr() if track else None, slope,
                               z.data_ptr(), stats.data_ptr(), _lib.stream_ptr())
        _lib.check(rc, "rk_bn_act_fwd")
        ctx.slope = slope
        ctx.save_for_backward(x, gamma, beta, stats)
        return z

    @staticmethod
    def backward(ctx, g_z):
        lib = _lib.load()
        x, gamma, beta, stats = ctx.saved_tensors
        B, U = x.shape
        g_z = _lib.require_cuda(g_z, "g_z", torch.float32)
        g_x = torch.empty_like(x)
        g_par = torch.empty(2, U, dtype=torch.float32, device=x.device)     # d gamma | d beta
        rc = lib.rk_bn_act_bwd(x.data_ptr(), g_z.data_ptr(), B, U, gamma.data_ptr(), beta.data_ptr(), ctx.slope,
                               stats.data_ptr(), g_x.data_ptr(), g_par[0].data_ptr(), g_par[1].data_ptr(),
                               _lib.stream_ptr())
        _lib.check(rc, "rk_bn_act_bwd")
        return g_x, g_par[0], g_par[1], None, None


def _rows(t):
    """t with unit column stride, and its row pitch: the kernel reads strided rows in place."""
    B, n = t.shape
    if (n > 1 and t.stride(1) != 1) or (B > 1 and t.stride(0) < n):
        t = t.contiguous()
    return t, (t.stride(0) if B > 1 else n)


class _Linear(torch.autograd.Function):
    """nn.Linear with torch's forward and input gradient; dW = g^T x and db = sum_b g in one csrc/linear.cu
    call (cuBLAS runs these as a split-K sgemm over a few dozen output tiles plus a separate bias reduce)."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return F.linear(x, weight, bias)

    @staticmethod
    def backward(ctx, g):
        lib = _lib.load()
        x, weight = ctx.saved_tensors
        g_x = g.mm(weight) if ctx.needs_input_grad[0] else None
        B, K = x.shape
        N = weight.shape[0]
        x, ldx = _rows(x)
        g, ldg = _rows(g)
        g_w = torch.empty_like(weight)
        g_b = torch.empty(N, dtype=torch.float32, device=g.device) if ctx.has_bias else None
        partials = torch.empty(lib.rk_linear_wgrad_scratch_floats(B, K, N), dtype=torch.float32, device=g.device)
        rc = lib.rk_linear_wgrad(x.data_ptr(), ldx, g.data_ptr(), ldg, B, K, N, g_w.data_ptr(), _lib.ptr(g_b),
                                 partials.data_ptr() if partials.numel() else None, _lib.stream_ptr())
        _lib.check(rc, "rk_linear_wgrad")
        return g_x, g_w, g_b


def _activation_slope(layer):
    if type(layer) is nn.ReLU:
        return 0.0
    if type(layer) is nn.LeakyReLU:
        return float(layer.negative_slope)
    return None


def _fusable_bn(bn):
    return (isinstance(bn, nn.BatchNorm1d) and bn.training and bn.momentum is not None
            and (bn.track_running_stats or bn.running_mean is None))


def run_tower(layers, x):
    """`for layer in layers: x = layer(x)` with Dice(+BatchNorm1d) and BatchNorm1d+(Leaky)ReLU pairs
    fused on CUDA, and nn.Linear weight gradients from librank."""
    from .din import Dice
    n, i = len(layers), 0
    max_b = None
    while i < n:
        layer = layers[i]
        if (FUSED and isinstance(layer, Dice) and layer.training and x.is_cuda and x.dim() == 2
                and x.dtype == torch.float32 and _fusable_bn(layer.bn) and not layer.bn.affine):
            if max_b is None:
                max_b = _lib.load().rk_dice_bn_max_batch()
            if MIN_BATCH <= x.shape[0] <= max_b:
                nxt = layers[i + 1] if i + 1 < n else None
                bn2 = nxt if (_fusable_bn(nxt) and nxt.affine and nxt.num_features == x.shape[1]) else None
                x = _DiceBn.apply(x, layer.alpha, bn2.weight if bn2 is not None else None,
                                  bn2.bias if bn2 is not None else None, layer.bn, bn2)
                i += 2 if bn2 is not None else 1
                continue
        if (FUSED and _fusable_bn(layer) and layer.affine and x.is_cuda and x.dim() == 2
                and x.dtype == torch.float32 and i + 1 < n and _activation_slope(layers[i + 1]) is not None):
            if max_b is None:
                max_b = _lib.load().rk_dice_bn_max_batch()
            if MIN_BATCH <= x.shape[0] <= max_b:
                x = _BnAct.apply(x, layer.weight, layer.bias, layer, _activation_slope(layers[i + 1]))
                i += 2
                continue
        if (FUSED and type(layer) is nn.Linear and x.is_cuda and x.dim() == 2 and x.dtype == torch.float32
                and layer.weight.dtype == torch.float32 and MIN_BATCH <= x.shape[0]
                and layer.out_features >= LINEAR_MIN_OUT):
            x = _Linear.apply(x, layer.weight, layer.bias)
            i += 1
            continue
        x = layer(x)
        i += 1
    return x
