"""rank_b200.Adam without a GPU: construction, validation, state_dict interchange with torch.optim.Adam, and
the descriptor layout of rk_adam_step."""
import ctypes

import pytest
import torch

import rank_b200
from rank_b200 import _lib


def _params():
    torch.manual_seed(0)
    return [torch.nn.Parameter(torch.randn(5, 3)), torch.nn.Parameter(torch.randn(3))]


@pytest.mark.parametrize("kw", [dict(weight_decay=0.01), dict(amsgrad=True), dict(maximize=True), dict(lr=-1e-3),
                                dict(eps=-1.0), dict(betas=(1.0, 0.999)), dict(betas=(0.9, -0.1)),
                                dict(lr=torch.tensor(1e-3))])
def test_constructor_refuses_what_it_does_not_implement(kw):
    with pytest.raises(ValueError):
        rank_b200.Adam(_params(), **kw)


def test_groups_carry_torch_adam_keys():
    opt = rank_b200.Adam(_params(), lr=3e-3)
    ref = torch.optim.Adam(_params(), lr=3e-3, fused=True)
    assert set(opt.param_groups[0]) == set(ref.param_groups[0])
    g = opt.param_groups[0]
    assert g["lr"] == 3e-3 and g["betas"] == (0.9, 0.999) and g["eps"] == 1e-8 and g["weight_decay"] == 0.0
    assert rank_b200.Adam is rank_b200.optim.Adam


def test_cpu_parameters_are_refused_before_any_update():
    ps = _params()
    opt = rank_b200.Adam(ps)
    for p in ps:
        p.grad = torch.ones_like(p)
    before = [p.detach().clone() for p in ps]
    with pytest.raises(rank_b200.RankB200Error):
        opt.step()
    assert all(torch.equal(p, b) for p, b in zip(ps, before))
    assert not opt.state                                  # nothing was initialised either


def test_parameters_without_gradient_are_skipped():
    ps = _params()
    assert rank_b200.Adam(ps).step() is None


@pytest.mark.parametrize("foreach", [True, False])
def test_torch_state_dict_loads_with_the_step_in_fused_format(foreach):
    ps = _params()
    ref = torch.optim.Adam(ps, lr=1e-2, foreach=foreach)
    for p in ps:
        p.grad = torch.randn_like(p)
    ref.step()
    ref.step()
    opt = rank_b200.Adam(ps)
    opt.load_state_dict(ref.state_dict())
    for p in ps:
        st = opt.state[p]
        assert st["step"].dtype == torch.float32 and st["step"].dim() == 0 and float(st["step"]) == 2.0
        assert torch.equal(st["exp_avg"], ref.state[p]["exp_avg"])
    assert opt.param_groups[0]["lr"] == 1e-2 and opt.param_groups[0]["fused"] is True
    back = torch.optim.Adam(ps)
    back.load_state_dict(opt.state_dict())                # and the reverse: torch continues as fused Adam
    assert back.param_groups[0]["fused"] is True and float(back.state[ps[0]]["step"]) == 2.0


def test_state_dict_with_weight_decay_is_refused():
    ps = _params()
    ref = torch.optim.Adam(ps, weight_decay=0.1)
    with pytest.raises(ValueError):
        rank_b200.Adam(ps).load_state_dict(ref.state_dict())


def test_descriptor_layout_matches_header():
    assert ctypes.sizeof(_lib.RkAdamTensor) == 104                     # rk_adam_tensor_t
    assert _lib.RkAdamTensor.capacity.offset == 64 and _lib.RkAdamTensor.eps.offset == 96
    assert _lib.RK_ADAM_MAX_TENSORS >= 64


def test_entry_point_validates_without_a_gpu():
    lib = _lib.load()
    assert lib.rk_adam_step(None, 0, None, None) == 0                  # nothing to do
    assert lib.rk_adam_step(None, _lib.RK_ADAM_MAX_TENSORS + 1, None, None) < 0
    d = (_lib.RkAdamTensor * 1)()
    d[0].param = d[0].exp_avg = d[0].exp_avg_sq = d[0].step = 16
    d[0].rows, d[0].dim = 4, 4
    assert lib.rk_adam_step(d, 1, None, None) < 0                      # neither grad nor touched_count
    d[0].grad, d[0].touched_count = 16, 16
    assert lib.rk_adam_step(d, 1, None, None) < 0                      # both
    assert b"exactly one" in lib.rk_last_error()
