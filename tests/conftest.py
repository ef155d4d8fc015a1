import glob
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
# a checkout of the reference project, for the tests that run it live; those that can fall back to
# outputs recorded from it under tests/golden do so when it is absent
REFERENCE_ROOT = os.environ.get("RANK_REFERENCE_ROOT", "")
HAVE_REFERENCE = bool(REFERENCE_ROOT) and os.path.isdir(REFERENCE_ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def golden_files(prefix=""):
    return sorted(glob.glob(os.path.join(GOLDEN_DIR, prefix + "*.pt")))


def load_golden(path):
    return torch.load(path, map_location="cpu", weights_only=False)


@pytest.fixture(scope="session")
def small_vocab_dir(tmp_path_factory):
    """Vocabulary directory with the line counts the golden fixtures were made with."""
    import rank_b200
    fx = load_golden(os.path.join(GOLDEN_DIR, "dcn_l3.pt"))
    path = tmp_path_factory.mktemp("vocab_small")
    return rank_b200.write_vocab_dir(str(path), fx["vocab_lines"]) + "/"


@pytest.fixture(scope="session")
def wechat_vocab_dir(tmp_path_factory):
    """Vocabulary directory with the real WeChat-challenge line counts."""
    import rank_b200
    path = tmp_path_factory.mktemp("vocab_wechat")
    return rank_b200.write_vocab_dir(str(path)) + "/"


def to_device(obj, device):
    if torch.is_tensor(obj):
        return obj.to(device)
    if isinstance(obj, dict):
        return {k: to_device(v, device) for k, v in obj.items()}
    if isinstance(obj, (list, tuple)):
        return type(obj)(to_device(v, device) for v in obj)
    return obj


def grad_floor(ref_grads):
    """Scale floor for gradient comparisons: tensors that are mathematically zero (e.g. the key
    bias of a softmax attention) hold only rounding noise, so they are compared against a small
    fraction of the model's largest gradient instead of against themselves."""
    return 1e-3 * max(float(g.abs().max()) for g in ref_grads.values())


def rel_err(a, b, floor=1e-30):
    """max |a-b| / max(|b|, floor) over the tensor — the 'relative' of the 1e-5 bar."""
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    if a.shape != b.shape:
        raise AssertionError(f"shape {tuple(a.shape)} vs {tuple(b.shape)}")
    if a.numel() == 0:
        return 0.0
    scale = max(float(b.abs().max()), floor)
    return float((a - b).abs().max()) / scale


def pytest_terminal_summary(terminalreporter, exitstatus, config):
    """How often the float64 arbiter of tests/test_gpu_models.py::compare decided a gradient
    comparison (fp32 comparison > tol, accepted against the float64 run), and the worst errors."""
    mod = sys.modules.get("test_gpu_models")
    stats = getattr(mod, "ARBITER", None)
    if not stats or not stats["comparisons"]:
        return
    tr = terminalreporter
    tr.write_line(f"float64 arbiter: fired {stats['fired']} of {stats['comparisons']} gradient comparisons; "
                  f"worst e_ref {stats['worst_e_ref']:.3e}, worst e_ours {stats['worst_e_ours']:.3e}")
    for case in stats["cases"]:
        tr.write_line("  arbiter: %s %s fp32-vs-fp32 %.3e, ours-vs-f64 %.3e, oracle-vs-f64 %.3e" % case)
    out_dir = os.path.join(ROOT, "gpurun_out")
    if os.path.isdir(out_dir):
        import json
        with open(os.path.join(out_dir, "arbiter_stats.json"), "w") as f:
            json.dump(stats, f, indent=1)
