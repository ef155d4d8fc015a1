"""Pins oracle/ against outputs of the unmodified reference (CPU, no GPU needed)."""
import importlib.util
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN_DIR, HAVE_REFERENCE, REFERENCE_ROOT, golden_files, grad_floor, load_golden, rel_err
import golden_cases
from oracle import interactions as X
from oracle import models as oracle_models

MODEL_FIXTURES = [p for p in golden_files() if "smoke" not in p and "loader" not in p and "checkpoint" not in p]
TOL = 2e-6   # same torch ops in (almost) the same order: far inside the 1e-5 bar
BAR = 1e-5   # the project's fp32 parity bar
ZERO = 1e-4  # a gradient below ZERO x the model's largest one is mathematically zero: rounding noise only


def _oracle_grads_float64(fx, vocab_dir):
    model = golden_cases.build(fx, oracle_models, vocab_dir, oracle=True)
    model.load_state_dict(fx["state_dict"], strict=True)
    return golden_cases.replay(model.double(), fx, golden_cases.to_double(fx["inputs"]),
                               golden_cases.to_double(fx["cotangents"]))[1]


@pytest.mark.parametrize("path", MODEL_FIXTURES, ids=[os.path.basename(p) for p in MODEL_FIXTURES])
def test_oracle_matches_reference_fixture(path, small_vocab_dir):
    fx = load_golden(path)
    model = golden_cases.build(fx, oracle_models, small_vocab_dir, oracle=True)
    missing = model.load_state_dict(fx["state_dict"], strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    outs, grads = golden_cases.replay(model, fx, fx["inputs"], fx["cotangents"])
    assert len(outs) == len(fx["outputs"])
    for i, (o, ref) in enumerate(zip(outs, fx["outputs"])):
        if torch.is_tensor(ref):
            assert rel_err(o, ref) <= TOL, f"output {i}"
        else:
            assert o == ref
    assert set(grads) == set(fx["grads"])
    floor = grad_floor(fx["grads"])
    gmax = max(float(g.abs().max()) for g in fx["grads"].values())
    grads64 = None
    for k, g in fx["grads"].items():
        e = rel_err(grads[k], g, floor)
        if e <= TOL:
            continue
        # The recorded gradients carry the summation order of the host that recorded them; with another
        # thread count or vector width the CPU kernels add the same terms in another order.
        if float(g.abs().max()) < ZERO * gmax:
            # mathematically zero (a Linear bias feeding BatchNorm): both sides hold only the rounding noise
            # of cancelling sums, so the bar is taken against the model's gradient scale, as in
            # tests/test_gpu_models.py::compare
            err = float((grads[k].double() - g.double()).abs().max())
            assert err <= TOL * gmax, f"grad {k} (numerically zero): abs err {err / gmax:.3e} of the scale"
        else:
            # both fp32 results against the oracle in float64: the recorded one must lie within the 1e-5 bar
            # of it (the oracle does the reference's arithmetic) and the oracle's own fp32 result no further
            # from it than TOL or twice the recorded one's rounding error
            if grads64 is None:
                grads64 = _oracle_grads_float64(fx, small_vocab_dir)
            e_ref, e_ours = rel_err(g, grads64[k], floor), rel_err(grads[k], grads64[k], floor)
            assert e_ref <= BAR and e_ours <= max(TOL, 2.0 * e_ref), \
                f"grad {k}: {e:.3e} vs recorded; vs float64: oracle {e_ours:.3e}, recorded {e_ref:.3e}"


def test_din_attention_reference_smoke():
    """The reference's own smoke input (DIN/din_attention.py:54-68), incl. keys_length = 0."""
    fx = load_golden(os.path.join(GOLDEN_DIR, "din_attention_smoke.pt"))
    for soft, key, state in ((False, "out_raw", "rng_before_raw"), (True, "out_softmax", "rng_before_softmax")):
        torch.set_rng_state(fx[state])
        net = torch.nn.Sequential(torch.nn.Linear(16, 64), torch.nn.ReLU(), torch.nn.Linear(64, 32),
                                  torch.nn.ReLU(), torch.nn.Linear(32, 1))
        mlp = tuple(p.detach() for p in net.parameters())
        out = X.din_local_activation(fx["query"], fx["keys"], fx["keys_length"], mlp, soft)
        assert rel_err(out, fx[key]) <= TOL
    assert torch.count_nonzero(fx["out_raw"][0]) == 0   # length 0, raw mode -> zeros


def test_dense_embedding_grad_matches_autograd():
    gen = torch.Generator().manual_seed(0)
    idx = torch.randint(0, 7, (50,), generator=gen)
    g = torch.randn(50, 4, generator=gen)
    w = torch.zeros(7, 4, requires_grad=True)
    (w[idx] * g).sum().backward()
    mine = X.dense_embedding_grad(idx.numpy(), g.numpy(), 7)
    assert np.allclose(mine, w.grad.numpy(), rtol=1e-6, atol=1e-6)


def test_stable_occurrence_order():
    cols = [np.array([2, 0, 2, 1]), np.array([0, 0])]
    keys, perm = X.stable_occurrence_order(cols, [3, 5])
    assert keys.tolist() == [0, 1, 2, 2, 4, 4]      # field 1 starts after field 0's sentinel key (3)
    assert perm.tolist() == [1, 3, 0, 2, 0, 1]


@pytest.mark.skipif(not HAVE_REFERENCE, reason="needs the reference checkout (RANK_REFERENCE_ROOT); "
                    "test_oracle_matches_shipped_checkpoint_fixture checks the same checkpoints against its recorded outputs")
@pytest.mark.parametrize("which", ["DCN", "DeepCrossing"])
def test_oracle_loads_shipped_checkpoint_and_matches_reference(which):
    """The two real trained state_dicts the reference ships, on the real vocabulary sizes."""
    rel = {"DCN": "DCN/dcn.py", "DeepCrossing": "DeepCrossing/deepcrossing.py"}[which]
    spec = importlib.util.spec_from_file_location("ref_" + which, os.path.join(REFERENCE_ROOT, "algorithm", rel))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    vocab = os.path.join(REFERENCE_ROOT, "dataset/wechat_algo_data1/vocabulary/")
    sd = torch.load(os.path.join(REFERENCE_ROOT, "algorithm", which, "model_dir/best_model.pth"),
                    map_location="cpu")
    if which == "DCN":
        a, b = ref.DCNModel(vocab, num_cross_layer=3), oracle_models.OracleDCN(vocab, num_cross_layer=3)
    else:
        a, b = ref.DeepCrossingModel(vocab, 128, 2), oracle_models.OracleDeepCrossing(vocab, 128, 2)
    a.load_state_dict(sd)
    b.load_state_dict(sd)
    gen = torch.Generator().manual_seed(4)
    B = 64
    dense = torch.rand(B, 16, generator=gen)
    cat = {c: torch.randint(0, e.num_embeddings, (B,), generator=gen) for c, e in a.embeddings.items()}
    torch.manual_seed(99)
    pa, la = a(dense, cat)
    torch.manual_seed(99)
    pb, lb = b(dense, cat)
    assert rel_err(lb, la) <= TOL and rel_err(pb, pa) <= TOL


@pytest.mark.parametrize("which", ["dcn", "deepcrossing"])
def test_oracle_matches_shipped_checkpoint_fixture(which, tmp_path):
    """tests/golden/checkpoint_*.pt: the reference's two trained state_dicts run through the unmodified
    reference classes (make_checkpoint_golden.py) — outputs and every gradient."""
    import golden_cases
    import rank_b200
    fx = golden_cases.expand_checkpoint(load_golden(os.path.join(GOLDEN_DIR, f"checkpoint_{which}.pt")))
    vocab = rank_b200.write_vocab_dir(str(tmp_path), fx["vocab_lines"]) + "/"
    model = golden_cases.build(fx, oracle_models, vocab, oracle=True)
    model.load_state_dict(fx["state_dict"], strict=True)
    outs, grads = golden_cases.replay(model, fx, fx["inputs"], fx["cotangents"])
    for o, r in zip(outs, fx["outputs"]):
        assert rel_err(o, r) <= TOL
    assert set(grads) == set(fx["grads"])
    for k, g in fx["grads"].items():
        assert rel_err(grads[k], g) <= TOL, k
