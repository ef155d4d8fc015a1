"""CrossNet, residual units and the FM / FwFM parts at the widths their kernels accept, against the oracle.

Each kernel picks a vector width and a register or shared-memory tiling from the row width, so a single
model layout runs one of them.  Here synthetic tables and indices (seeded) reach every forward <VEC, R>
of the CrossNet, 1 to 32 lanes per sample at vec 1, 2 and 4 of the FM part, residual units from d = 1
to 256 with partial tiles of every height, and the widest rows each forward takes, whose backward must
take them too.  Outputs and gradients are judged as test_gpu_models.compare judges them (the oracle in
fp32 at 1e-5, the oracle in float64 as the arbiter), gathered rows bit for bit.  Layouts whose table
gradients the reductions cannot produce are refused by the forward before anything is launched.
"""
import pytest
import torch

import rank_b200
from rank_b200 import RankB200Error, _lib
from rank_b200.dcn import _CrossNet, draw_cross_weights
from rank_b200.deepcrossing import _ResidualStack, draw_residual_units
from rank_b200.deepfm import _FMInteraction
from rank_b200.fwfm import _FwFMInteraction
from conftest import rel_err
from oracle import interactions as X
from test_interaction_limits import res_fwd_ok, res_widest_d

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5


def _judge(ours, runs):
    """ours / runs[dtype] = (outputs, {name: gradient}); runs holds the oracle in fp32 and in float64."""
    from test_gpu_models import compare
    (o_outs, o_grads), (r_outs, r_grads), (_, g64) = ours, runs[torch.float32], runs[torch.float64]
    assert set(o_grads) == set(r_grads)
    compare(o_outs, o_grads, r_outs, r_grads, TOL, g64)


def _oracle(fn, leaves, cots, dtype):
    """fn(**leaves) on the CPU in `dtype`; gradients of sum(out * cot) over the outputs with a cotangent.
    Returns ([outputs], {leaf: gradient}) with gradients that exist only."""
    xs = {k: v.detach().to(dtype).requires_grad_() for k, v in leaves.items()}
    outs = fn(**xs)
    loss = sum((o * c.to(dtype)).sum() for o, c in zip(outs, cots) if c is not None)
    loss.backward()
    return [o.detach() for o in outs], {k: v.grad for k, v in xs.items() if v.grad is not None}


def _both(fn, leaves, cots):
    return {dt: _oracle(fn, leaves, cots, dt) for dt in (torch.float32, torch.float64)}


def _ours(outs, cots, leaves):
    """Backward of sum(out * cot) on the GPU; gradients of the `leaves` that received one."""
    loss = sum((o * c.to(DEV)).sum() for o, c in zip(outs, cots) if c is not None)
    loss.backward()
    rank_b200.check_index_errors()
    return {k: v.grad for k, v in leaves.items() if v.grad is not None}


def _tables(gen, dims, rows_of=lambda f: 37 + 101 * f):
    """Tables of nn.Embedding's N(0, 1) init; small heights so rows repeat inside a batch."""
    return [torch.randn(rows_of(f), dim, generator=gen) for f, dim in enumerate(dims)]


def _indices(gen, tables, B):
    return [torch.randint(0, t.shape[0], (B,), generator=gen) for t in tables]


def _launches():
    torch.cuda.synchronize()
    return _lib.load().rk_launch_count()


# ---- CrossNet ------------------------------------------------------------------------------------
# (n_dense, field dims): forward VEC and units (R = 1, 2 or 4 rounds of 32 lanes), backward VEC (from d)
CROSS_LAYOUTS = {
    "v4_d96": (16, [64, 16]),                   # VEC 4, 24 units, R 1
    "v4_d256": (16, [128, 64, 48]),             # VEC 4, 64 units, R 2
    "v4_d388": (16, [128, 128, 116]),           # VEC 4, 97 units, R 4
    "v4_d512": (16, [128, 128, 128, 112]),      # VEC 4, 128 units, R 4
    "v2_d50": (16, [16, 2, 4, 4, 4, 4]),        # the WeChat side features: VEC 2, 25 units, R 1
    "v2_d100": (16, [2, 50, 32]),               # VEC 2, 50 units, R 2; backward VEC 4
    "v2_d130": (16, [2, 64, 48]),               # VEC 2, 65 units, R 4
    "v1_d31": (16, [1, 14]),                    # VEC 1, 31 units, R 1
    "v1_d63": (16, [3, 32, 12]),                # VEC 1, 63 units, R 2
    "v1_d128": (16, [1, 32, 32, 32, 15]),       # VEC 1, 128 units, R 4; backward VEC 4
    "v1_d127": (16, [1, 32, 32, 32, 14]),       # VEC 1, 127 units, R 4 in both directions
    "v2_d90": (16, [2, 40, 32]),                # VEC 2, 45 units, R 2 in both directions
    "v2_d52": (16, [2, 34]),                    # VEC 2, 26 units; backward VEC 4
}
CROSS_CASES = [("v4_d96", 1, 1000, "both"), ("v4_d256", 8, 7, "both"), ("v4_d388", 1, 8195, "cross"),
               ("v4_d512", 8, 1000, "both"), ("v4_d512", 0, 8195, "concat"), ("v2_d50", 8, 8195, "both"),
               ("v2_d100", 0, 1, "both"), ("v2_d130", 1, 1000, "concat"), ("v1_d31", 8, 1000, "cross"),
               ("v1_d63", 1, 7, "both"), ("v1_d128", 8, 8195, "both"), ("v1_d128", 0, 1, "cross"),
               ("v2_d52", 1, 1000, "both"), ("v2_d52", 8, 7, "concat"), ("v1_d127", 8, 1000, "both"),
               ("v2_d90", 1, 8195, "both")]


def _offsets(n_dense, dims):
    return [n_dense + sum(dims[:f]) for f in range(len(dims))]


@pytest.mark.parametrize("layout,L,B,grads", CROSS_CASES)
def test_crossnet_vs_oracle(layout, L, B, grads):
    n_dense, dims = CROSS_LAYOUTS[layout]
    F, d = len(dims), n_dense + sum(dims)
    gen = torch.Generator().manual_seed(d * 31 + L)
    tables = _tables(gen, dims)
    idx = _indices(gen, tables, B)
    dense = torch.randn(B, n_dense, generator=gen)
    torch.manual_seed(d)
    w, b = draw_cross_weights(d, L)
    b = b + 0.1 * torch.randn(L, d, generator=gen)          # the reference's b_l is zero: exercise the bias
    cots = [torch.randn(B, d, generator=gen) / B if grads in ("both", "concat") else None,
            torch.randn(B, d, generator=gen) / B if grads in ("both", "cross") else None]
    leaves = {"dense": dense, **{f"t{f}": t for f, t in enumerate(tables)}}

    def oracle(dense, **ts):
        x0 = X.concat_features(dense, [ts[f"t{f}"] for f in range(F)], idx)
        ws = [w[l].to(x0.dtype).view(d, 1) for l in range(L)]
        bs = [b[l].to(x0.dtype).view(d, 1) for l in range(L)]
        return [x0, X.cross_network(x0, ws, bs)]

    runs = _both(oracle, leaves, cots)
    dl = {k: v.to(DEV).requires_grad_() for k, v in leaves.items()}
    concat_all, cross_vec = _CrossNet.apply(F, _offsets(n_dense, dims), dl["dense"], w.to(DEV), b.to(DEV),
                                            *[i.to(DEV) for i in idx], *[dl[f"t{f}"] for f in range(F)])
    assert torch.equal(concat_all.detach().cpu(), runs[torch.float32][0][0])
    got = _ours([concat_all, cross_vec], cots, dl)
    _judge(([cross_vec], got), {dt: (outs[1:], g) for dt, (outs, g) in runs.items()})


@pytest.mark.parametrize("dims,words", [([1, 32, 32, 32, 16], "exceeds 128 units"),     # d = 129 at VEC 1
                                        ([128, 128, 128, 116], "wider than 512")])      # a 516-float row
def test_crossnet_refuses_rows_beyond_its_units(dims, words):
    gen = torch.Generator().manual_seed(1)
    tables = [t.to(DEV).requires_grad_() for t in _tables(gen, dims)]
    idx = [i.to(DEV) for i in _indices(gen, tables, 64)]
    d = 16 + sum(dims)
    w, b = (t.to(DEV) for t in draw_cross_weights(d, 1))
    before = _launches()
    with pytest.raises(RankB200Error, match=words):
        _CrossNet.apply(len(dims), _offsets(16, dims), torch.zeros(64, 16, device=DEV), w, b, *idx, *tables)
    assert _launches() == before


@pytest.mark.parametrize("d", [1, 31, 32, 33, 512])
def test_cross_layer_widths(d):
    B = 1000
    gen = torch.Generator().manual_seed(d)
    leaves = {"x0": torch.randn(B, d, generator=gen), "xl": torch.randn(B, d, generator=gen)}
    cots = [torch.randn(B, d, generator=gen) / B]
    torch.manual_seed(11)
    w, b = draw_cross_weights(d, 1)
    runs = _both(lambda x0, xl: [x0 * (xl @ w.to(xl.dtype).t()) + b.to(xl.dtype) + xl], leaves, cots)
    dl = {k: v.to(DEV).requires_grad_() for k, v in leaves.items()}
    torch.manual_seed(11)
    out = rank_b200.cross_layer(dl["x0"], dl["xl"], 0)
    _judge(([out], _ours([out], cots, dl)), runs)


# ---- residual units ------------------------------------------------------------------------------
RES_D = [1, 3, 4, 31, 33, 50, 64, 128, 200, 256]
RES_H = [1, 7, 8, 100, 128, 129, 256]
RES_B = [1, 31, 63, 65, 1000]
# every (d, H) the forward takes; B cycles so that partial tiles of 64 (H <= 128) and 32 rows (H > 128) occur
# at every width, and every other pair runs three units behind a gather of fields instead of residual_unit
RES_CASES = [(d, H, RES_B[k % len(RES_B)], "fields" if k % 2 else "unit")
             for k, (d, H) in enumerate([(d, H) for d in RES_D for H in RES_H if res_fwd_ok(d, H)])]


def _unpack_units(d, H, n_units, seed):
    """The nn.Linear draws draw_residual_units(d, H, n_units) packs, as the oracle's (W1, b1, W2, b2)."""
    torch.manual_seed(seed)
    units = []
    for _ in range(n_units):
        first, second = torch.nn.Linear(d, H), torch.nn.Linear(H, d)
        units.append(tuple(p.detach() for p in (first.weight, first.bias, second.weight, second.bias)))
    torch.manual_seed(seed)
    return units, draw_residual_units(d, H, n_units)


def _split_row(d):
    """A dense block and fields tiling d: one column, then fields of at most 32 at odd offsets."""
    n_dense = max(1, min(16, d // 2))
    dims = [1] if d > n_dense else []
    while n_dense + sum(dims) < d:
        dims.append(min(32, d - n_dense - sum(dims)))
    return n_dense, dims


def _run_residual(d, H, B, how, n_units):
    gen = torch.Generator().manual_seed(d * 1000 + H)
    seed = 7 * d + H
    units, pack = _unpack_units(d, H, n_units, seed)
    cots = [torch.randn(B, d, generator=gen) / B]
    if how == "unit":
        leaves = {"x": torch.randn(B, d, generator=gen)}
        runs = _both(lambda x: [X.residual_units(x, [tuple(t.to(x.dtype) for t in u) for u in units])], leaves, cots)
        dl = {k: v.to(DEV).requires_grad_() for k, v in leaves.items()}
        torch.manual_seed(seed)
        out = rank_b200.residual_unit(dl["x"], H, 0)
        _judge(([out], _ours([out], cots, dl)), runs)
        return
    n_dense, dims = _split_row(d)
    assert n_dense + sum(dims) == d and max(dims, default=0) <= 32
    F = len(dims)
    tables = _tables(gen, dims)
    idx = _indices(gen, tables, B)
    leaves = {"dense": torch.randn(B, n_dense, generator=gen), **{f"t{f}": t for f, t in enumerate(tables)}}

    def oracle(dense, **ts):
        x0 = X.concat_features(dense, [ts[f"t{f}"] for f in range(F)], idx)
        return [X.residual_units(x0, [tuple(t.to(x0.dtype) for t in u) for u in units])]

    runs = _both(oracle, leaves, cots)
    dl = {k: v.to(DEV).requires_grad_() for k, v in leaves.items()}
    out = _ResidualStack.apply(F, tuple(_offsets(n_dense, dims)), H, n_units, dl["dense"], pack.to(DEV),
                               *[i.to(DEV) for i in idx], *[dl[f"t{f}"] for f in range(F)])
    _judge(([out], _ours([out], cots, dl)), runs)


@pytest.mark.parametrize("d,H,B,how", RES_CASES)
def test_residual_units_vs_oracle(d, H, B, how):
    _run_residual(d, H, B, how, 3 if how == "fields" and B != 1000 else 1)


@pytest.mark.parametrize("H", [7, 64, 128, 129, 256])
def test_residual_units_at_the_widest_row(H):
    """The widest d the forward's shared memory takes: the backward must take it too."""
    _run_residual(res_widest_d(H), H, 1000, "fields", 2)


def test_residual_unit_reference_default_width():
    """residual_unit on a 128-wide input with the reference's internal_dim = 128."""
    _run_residual(128, 128, 1000, "unit", 1)


# ---- DeepFM's FM part ----------------------------------------------------------------------------
# D covers vec 1 (odd), 2 and 4 and 1 to 32 lanes per sample; F and B cycle; `grads` picks the cotangents
FM_CASES = [(1, 1, 8192, "all"), (3, 2, 1, "deep"), (5, 7, 333, "second"), (31, 16, 8192, "all"),
            (2, 1, 333, "all"), (6, 2, 8192, "second"), (34, 7, 1, "all"), (62, 16, 333, "deep"),
            (4, 16, 8192, "all"), (12, 7, 333, "all"), (36, 2, 1, "second"), (64, 1, 8192, "deep"),
            (100, 7, 333, "all"), (128, 16, 8192, "all"), (128, 2, 333, "second"), (31, 1, 1, "deep")]


def _fm_inputs(D, F, B, seed):
    gen = torch.Generator().manual_seed(seed)
    second = _tables(gen, [D] * F, rows_of=lambda f: 23 + 57 * f)
    first = [torch.randn(t.shape[0], 1, generator=gen) for t in second]
    return gen, first, second, _indices(gen, second, B)


@pytest.mark.parametrize("D,F,B,grads", FM_CASES)
def test_fm_part_vs_oracle(D, F, B, grads):
    gen, first, second, idx = _fm_inputs(D, F, B, D * 100 + F)
    cots = [torch.randn(B, F * D, generator=gen) / B if grads in ("all", "deep") else None,
            torch.randn(B, 1, generator=gen) / B if grads == "all" else None,
            torch.randn(B, 1, generator=gen) / B if grads in ("all", "second") else None]
    leaves = {**{f"first{f}": t for f, t in enumerate(first)}, **{f"second{f}": t for f, t in enumerate(second)}}
    runs = _both(lambda **ts: list(X.deepfm_fm_part([ts[f"first{f}"] for f in range(F)],
                                                    [ts[f"second{f}"] for f in range(F)], idx)), leaves, cots)
    dl = {k: v.to(DEV).requires_grad_() for k, v in leaves.items()}
    outs = _FMInteraction.apply(F, *[i.to(DEV) for i in idx], *[dl[f"first{f}"] for f in range(F)],
                                *[dl[f"second{f}"] for f in range(F)])
    assert torch.equal(outs[0].detach().cpu(), runs[torch.float32][0][0])
    got = _ours(outs, cots, dl)
    if F == 1:
        # one field has no pairs: the oracle's second-order term is exactly zero, and ours holds at most the
        # rounding of e^2 - e^2, judged against the scale of the squares it cancels (as compare judges a
        # numerically zero gradient against the model's gradient scale)
        assert not runs[torch.float32][0][2].any()
        scale = 0.5 * float((second[0][idx[0]] ** 2).sum(1).max())
        assert float(outs[2].detach().abs().max()) <= TOL * scale
        runs = {dt: (o[1:2], g) for dt, (o, g) in runs.items()}
        outs = outs[1:2]
    else:
        runs = {dt: (o[1:], g) for dt, (o, g) in runs.items()}
        outs = outs[1:]
    _judge((list(outs), got), runs)


@pytest.mark.parametrize("D", [33, 66, 129])
def test_fm_part_refuses_embeddings_beyond_32_lanes(D):
    """The kernel refuses them; with table gradients the reductions' own limit (the same one) refuses first."""
    _, first, second, idx = _fm_inputs(D, 2, 64, D)
    idx = [i.to(DEV) for i in idx]
    before = _launches()
    with pytest.raises(RankB200Error, match="too wide"):
        _FMInteraction.apply(2, *idx, *[t.to(DEV) for t in first + second])
    with pytest.raises(RankB200Error, match="at most"):
        _FMInteraction.apply(2, *idx, *[t.to(DEV).requires_grad_() for t in first + second])
    assert _launches() == before


# ---- FwFM ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("F", [2, 16])
@pytest.mark.parametrize("D", [1, 4, 32])
def test_fwfm_vs_oracle(F, D):
    B = 4097
    gen, first, second, idx = _fm_inputs(D, F, B, D * 100 + F + 1)
    P = F * (F - 1) // 2
    leaves = {**{f"first{f}": t for f, t in enumerate(first)}, **{f"second{f}": t for f, t in enumerate(second)},
              "field_weight": torch.randn(P, generator=gen), "bias": torch.full((1,), -0.5)}
    cots = [torch.randn(B, generator=gen) / B]

    def oracle(field_weight, bias, **ts):
        z = X.fwfm_logit([ts[f"first{f}"] for f in range(F)], [ts[f"second{f}"] for f in range(F)], idx,
                         field_weight, bias)
        return [torch.sigmoid(z).view(-1)]

    runs = _both(oracle, leaves, cots)
    dl = {k: v.to(DEV).requires_grad_() for k, v in leaves.items()}
    y = _FwFMInteraction.apply(F, *[i.to(DEV) for i in idx], *[dl[f"first{f}"] for f in range(F)],
                               *[dl[f"second{f}"] for f in range(F)], dl["field_weight"], dl["bias"])
    _judge(([y], _ours([y], cots, dl)), runs)


# ---- layouts whose table gradients cannot be reduced: refused before any launch --------------------
def _wide_field_at_odd_column(B=500):
    """16 dense columns, then fields of 64 and 1: an 81-float row, so the 64-wide field's gradient would
    be reduced one float per lane, 64 lanes (at most 32)."""
    gen = torch.Generator().manual_seed(81)
    tables = _tables(gen, [64, 1])
    return gen, torch.randn(B, 16, generator=gen), tables, _indices(gen, tables, B)


def test_crossnet_refuses_a_wide_field_at_an_odd_column():
    gen, dense, tables, idx = _wide_field_at_odd_column()
    w, b = draw_cross_weights(81, 2)
    args = (2, [16, 80], dense.to(DEV), w.to(DEV), b.to(DEV), *[i.to(DEV) for i in idx])
    before = _launches()
    with pytest.raises(RankB200Error, match="at most 32 columns"):
        _CrossNet.apply(*args, *[t.to(DEV).requires_grad_() for t in tables])
    assert _launches() == before
    # without table gradients the forward still serves
    with torch.no_grad():
        concat_all, cross_vec = _CrossNet.apply(*args, *[t.to(DEV) for t in tables])
    x0 = X.concat_features(dense, tables, idx)
    assert torch.equal(concat_all.cpu(), x0)
    assert rel_err(cross_vec, X.cross_network(x0, [w[l].view(81, 1) for l in range(2)],
                                              [b[l].view(81, 1) for l in range(2)])) <= TOL
    rank_b200.check_index_errors()


def test_residual_units_refuse_a_wide_field_at_an_odd_column():
    gen, dense, tables, idx = _wide_field_at_odd_column()
    units, pack = _unpack_units(81, 64, 1, 5)
    args = (2, (16, 80), 64, 1, dense.to(DEV), pack.to(DEV), *[i.to(DEV) for i in idx])
    before = _launches()
    with pytest.raises(RankB200Error, match="at most 32 columns"):
        _ResidualStack.apply(*args, *[t.to(DEV).requires_grad_() for t in tables])
    assert _launches() == before
    with torch.no_grad():
        out = _ResidualStack.apply(*args, *[t.to(DEV) for t in tables])
    assert rel_err(out, X.residual_units(X.concat_features(dense, tables, idx), units)) <= TOL
    rank_b200.check_index_errors()


@pytest.mark.parametrize("F", [17, 24])
@pytest.mark.parametrize("which", ["fm", "fwfm"])
def test_more_than_16_fields_are_refused_with_table_gradients(F, which):
    D, B = 4, 300
    _, first, second, idx = _fm_inputs(D, F, B, F)
    fw = [torch.randn(F * (F - 1) // 2), torch.zeros(1)] if which == "fwfm" else []
    op = _FMInteraction if which == "fm" else _FwFMInteraction
    args = [i.to(DEV) for i in idx]
    before = _launches()
    with pytest.raises(RankB200Error, match="RK_MAX_TABLES"):
        op.apply(F, *args, *[t.to(DEV).requires_grad_() for t in first + second], *[t.to(DEV) for t in fw])
    assert _launches() == before
    # the forward alone takes up to 24 fields
    with torch.no_grad():
        got = op.apply(F, *args, *[t.to(DEV) for t in first + second], *[t.to(DEV) for t in fw])
    if which == "fm":
        want = X.deepfm_fm_part(first, second, idx)
        assert torch.equal(got[0].cpu(), want[0])
        assert rel_err(got[1], want[1]) <= TOL and rel_err(got[2], want[2]) <= TOL
    else:
        assert rel_err(got, torch.sigmoid(X.fwfm_logit(first, second, idx, *fw)).view(-1)) <= TOL
    rank_b200.check_index_errors()
