"""rank_b200.loader.EncodedWechat against the reference's own WechatDataset + DataLoader (when the
reference checkout is present) and against batches recorded from it (tests/golden/loader_*.pt)."""
import importlib.util
import os

import pytest
import torch
from torch.utils.data import DataLoader

import rank_b200
from rank_b200.loader import EncodedWechat
from conftest import GOLDEN_DIR, HAVE_REFERENCE, REFERENCE_ROOT
import loader_cases

REF = {"deepfm": "DeepFM/deepfm.py", "dcn": "DCN/dcn.py", "deepcrossing": "DeepCrossing/deepcrossing.py",
       "din": "DIN/din.py", "bst": "BST/bst.py"}
BATCH = 8


def _same(a, b, path="batch"):
    if torch.is_tensor(b):
        assert torch.is_tensor(a) and a.dtype == b.dtype and a.shape == b.shape, path
        assert torch.equal(a, b) or (a.is_floating_point() and torch.equal(torch.nan_to_num(a), torch.nan_to_num(b))
                                     and torch.equal(a.isnan(), b.isnan())), path
    elif isinstance(b, dict):
        assert isinstance(a, dict) and list(a.keys()) == list(b.keys()), path
        for k in b:
            _same(a[k], b[k], f"{path}/{k}")
    else:
        raise TypeError(path)


def _reference_batches(kind, path, vocab_dir):
    spec = importlib.util.spec_from_file_location("ref_" + kind, os.path.join(REFERENCE_ROOT, "algorithm", REF[kind]))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    ds = ref.WechatDataset(path, vocab_dir, 5) if kind == "bst" else ref.WechatDataset(path, vocab_dir)
    kw = {"collate_fn": ref.din_collate_fn} if kind == "din" else {}
    return list(DataLoader(ds, batch_size=BATCH, shuffle=False, **kw))


@pytest.mark.parametrize("kind", sorted(REF))
@pytest.mark.parametrize("history", ["string", "list"])
def test_batches_equal_the_reference_dataloader(kind, history, tmp_path):
    """Through a parquet file, as the reference reads its data.  Without a reference checkout the
    string-history frame is compared with the batches the reference produced for it
    (tests/golden/make_golden.py wrote them from the same parquet file); its batches for list
    histories were not recorded."""
    if not HAVE_REFERENCE and history != "string":
        pytest.skip("needs the reference checkout (RANK_REFERENCE_ROOT): no recorded batches for list histories")
    vocab_dir = loader_cases.write_vocab(str(tmp_path / "vocab")) + "/"
    path = os.path.join(str(tmp_path), f"{kind}.parquet")
    loader_cases.make_frame(history).to_parquet(path)
    if HAVE_REFERENCE:
        want = _reference_batches(kind, path, vocab_dir)
    else:
        want = torch.load(os.path.join(GOLDEN_DIR, "loader_batches.pt"), weights_only=False)[kind]
    enc = EncodedWechat(path, vocab_dir, kind, max_seq_length=5)       # reads the same parquet file
    got = list(enc.batches(BATCH))
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        _same(g, w, f"{kind}[{i}]")


@pytest.mark.parametrize("kind", sorted(REF))
def test_batches_equal_the_recorded_reference_batches(kind, tmp_path):
    fx = torch.load(os.path.join(GOLDEN_DIR, "loader_batches.pt"), weights_only=False)
    vocab_dir = loader_cases.write_vocab(str(tmp_path / "vocab")) + "/"
    enc = EncodedWechat(loader_cases.make_frame("string"), vocab_dir, kind, max_seq_length=5)
    got = list(enc.batches(BATCH))
    assert len(got) == len(fx[kind])
    for i, (g, w) in enumerate(zip(got, fx[kind])):
        _same(g, w, f"{kind}[{i}]")


def test_shuffled_batches_and_packed_staging(tmp_path):
    vocab_dir = loader_cases.write_vocab(str(tmp_path / "vocab")) + "/"
    enc = EncodedWechat(loader_cases.make_frame("string"), vocab_dir, "dcn")
    gen = torch.Generator().manual_seed(3)
    order = torch.randperm(len(enc), generator=torch.Generator().manual_seed(3))
    packed = rank_b200.PackedBatch.like(enc.batch(range(BATCH)), "cpu", pin=False)
    seen = 0
    for i, b in enumerate(enc.batches(BATCH, shuffle=True, generator=gen, drop_last=True, packed=packed)):
        assert b is packed
        _same(packed.host_views, enc.batch(order[i * BATCH:(i + 1) * BATCH].numpy()))
        seen += 1
    assert seen == len(enc) // BATCH
