#!/usr/bin/env python
"""Input-path timings: the host loader against batches gathered on the device (csrc/batch.cu, rank_b200.device_data).

    python scripts/bench_input.py --out-dir DIR [--rows 1048576] [--batch 8192]

On a seeded synthetic WeChat-shaped encoded frame (`--rows` rows; DIN histories 30 % empty, lengths 1..50
otherwise; Zipf ids over the real vocabulary sizes; BST sequences of 20):
1. host_rows_per_s: one shuffled epoch of EncodedWechat.batches per kind, with the host's core count;
2. gather: rk_batch_gather device time per batch (CUDA events around a CUDA graph of one launch per batch of
   the epoch, replayed twice: >= 200 launches; the frame is larger than L2 and read in shuffled order), and
   the bytes it moves (each column read and written once, the order entries, DIN's offsets, ids, padding
   and lengths) over that time;
3. epoch: wall time of one epoch of DIN training (tensor-core activation unit, raw attention, batch
   `--batch`; the bench's step: zero_grad, forward, loss, backward, replayed from one CUDA graph), the
   epoch's randperm included, synchronised at the end, fed
     (a) host:   EncodedWechat.batch padded to the fixed width -> PackedBatch.fill -> Prefetcher -> replay;
     (b) device: BatchFeed.next() captured inside the step's graph -> replay;
   next to the step alone (the same graph replayed on resident inputs).
Prints one JSON object and writes it to DIR/bench_input.json, with the GPU's name, power limit and SM clocks
read in the same run.  Needs a CUDA device.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

T_DIN, T_BST = 50, 20


def gpu_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = ""
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": {"query": q, "value": out}}


def synthetic_encoded(kind, n, seed=1):
    """An EncodedWechat holding seeded synthetic arrays of the shapes and dtypes the encoder produces."""
    from rank_b200 import synthetic
    from rank_b200.loader import SIDE, SIX, EncodedWechat
    gen = torch.Generator().manual_seed(seed)
    rows = synthetic.table_rows()
    enc = object.__new__(EncodedWechat)
    enc.kind, enc.n, enc.max_seq_length = kind, n, T_BST
    enc.label = synthetic.labels(gen, n).numpy()
    enc.category = {c: synthetic.zipf_indices(gen, rows[c], (n,)).numpy() for c in (SIX if kind == "deepfm" else SIDE)}
    if kind != "deepfm":
        enc.dense = synthetic.dense_block(gen, n).numpy()
    if kind == "din":
        enc.target = {"feedid": synthetic.zipf_indices(gen, rows["feedid"], (n,)).numpy()}
        lengths = torch.randint(1, T_DIN + 1, (n,), generator=gen) * (torch.rand(n, generator=gen) >= 0.3)
        enc.seq_offsets = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(lengths.numpy(), out=enc.seq_offsets[1:])
        enc.seq_flat = synthetic.zipf_indices(gen, rows["feedid"], (int(enc.seq_offsets[-1]),)).numpy()
    if kind == "bst":
        length = torch.randint(1, T_BST + 1, (n,), generator=gen)
        seq = synthetic.zipf_indices(gen, rows["feedid"], (n, T_BST))
        enc.seq = (seq * (torch.arange(T_BST) < length.unsqueeze(1))).numpy()
        enc.seq_length = length.numpy()
    return enc


def pad(batch, width):
    from rank_b200.loader import DIN_SEQ
    seq = batch["sequence"][DIN_SEQ]
    out = dict(batch)
    out["sequence"] = {DIN_SEQ: F.pad(seq, (0, width - seq.shape[1])),
                       DIN_SEQ + "_length": batch["sequence"][DIN_SEQ + "_length"]}
    return out


def host_rate(enc, B):
    t0 = time.perf_counter()
    rows = sum(len(b["label"]) for b in enc.batches(B, shuffle=True, generator=torch.Generator().manual_seed(3)))
    return rows / (time.perf_counter() - t0)


def gather_time(enc, data, B, dev):
    """ms per rk_batch_gather launch and the bytes each moves."""
    feed = data.feed(B)
    feed.start_epoch(shuffle=True, generator=torch.Generator().manual_seed(4))
    k = len(feed)
    starts = torch.arange(0, k * B, B, dtype=torch.int64, device=dev)
    cursors = [starts[i:i + 1] for i in range(k)]

    def launches():
        for c in cursors:
            data._gather(feed._outs, feed.order, k * B, c, 0, B, feed.width, feed.status)

    launches()                                            # warm-up, and outside capture: module load
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        launches()
    g.replay()
    torch.cuda.synchronize()
    times = []
    for _ in range(2):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        g.replay()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b) / k)
    feed.check()
    row_bytes = sum(t[0].numel() * t.element_size() for p, t in feed._outs if p[-1] != "his_read_comment_7d_seq"
                    and p[-1] != "his_read_comment_7d_seq_length")
    moved = B * (2 * row_bytes + 8)                       # every column read + written, one order entry per row
    if enc.kind == "din":
        mean_len = float(enc.seq_offsets[-1]) / enc.n
        moved += B * (16 + 8 * mean_len + 8 * feed.width + 8)   # offsets, ids read, padded ids + length written
    ms = statistics.median(times)
    return {"launches": 2 * k, "device_ms_per_batch": ms, "bytes_per_batch": int(moved),
            "gb_per_s": moved / (ms * 1e-3) / 1e9}


def din_epochs(enc, data, B, dev, reps):
    import rank_b200
    from rank_b200.staging import PackedBatch, Prefetcher
    vocab = rank_b200.write_vocab_dir(tempfile.mkdtemp(prefix="rk_vocab_")) + "/"
    torch.manual_seed(0)
    model = rank_b200.DIN(vocab, dropout_rate=0.0, use_softmax=False, l2_lambda=0.2).to(dev)
    model.activation_unit_precision = "bf16"
    model.train()
    W = data.seq_width
    example = pad(enc.batch(np.arange(B)), W)
    static = PackedBatch.like(example, dev)
    static.fill(example)
    static.to_device()
    feed = data.feed(B)

    def step(b):
        prob, _, l2 = model(b["dense"], b["category"], b["sequence"], b["target"])
        loss = F.binary_cross_entropy(prob.squeeze(), b["label"]) + l2
        loss.backward()

    def capture(body):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                model.zero_grad(set_to_none=True)
                body()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        model.zero_grad(set_to_none=True)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            body()
        return g

    model.draw_ephemeral()
    model.ephemeral_frozen = True
    g_static = capture(lambda: step(static.device_views))
    g_feed = capture(lambda: step(feed.next()))
    k = len(feed)
    gen = torch.Generator().manual_seed(5)

    def step_alone():
        for _ in range(k):
            g_static.replay()

    hosts = [PackedBatch.like(example, dev) for _ in range(2)]      # pinned, filled alternately
    pf = Prefetcher(static)

    def host_fed():
        order = torch.randperm(enc.n, generator=gen).numpy()
        hosts[0].fill(pad(enc.batch(order[:B]), W))
        slot = pf.submit(hosts[0])
        for i in range(k):
            nxt = None
            if i + 1 < k:
                hosts[(i + 1) % 2].fill(pad(enc.batch(order[(i + 1) * B:(i + 2) * B]), W))
                nxt = pf.submit(hosts[(i + 1) % 2])
            pf.consume(slot)
            g_static.replay()
            slot = nxt

    def device_fed():
        feed.start_epoch(shuffle=True, generator=gen)
        for _ in range(k):
            g_feed.replay()

    out = {name: [] for name in ("step_alone", "host_fed", "device_fed")}
    for fn in (step_alone, host_fed, device_fed):          # warm-up
        fn()
    torch.cuda.synchronize()
    for _ in range(reps):                                 # alternate, so drift of a shared machine hits all alike
        for name, fn in (("step_alone", step_alone), ("host_fed", host_fed), ("device_fed", device_fed)):
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            out[name].append(time.perf_counter() - t0)
    feed.check()
    rank_b200.check_index_errors()
    res = {"batches_per_epoch": k, "batch": B, "seq_width": W, "reps": reps,
           "workload": "DIN raw attention, tensor-core activation unit, zero_grad+fwd+loss+bwd graph replay"}
    for name, ts in out.items():
        s = statistics.median(ts)
        res[name] = {"epoch_s": s, "ms_per_batch": 1e3 * s / k, "samples_per_s": k * B / s, "all_epoch_s": ts}
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out-dir", required=True)
    ap.add_argument("--rows", type=int, default=1 << 20)
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_input.py needs a CUDA device")
    from rank_b200.loader import KINDS
    dev = torch.device("cuda:0")
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else os.cpu_count()
    result = {"device": gpu_info(), "rows": args.rows, "host_cores": cores, "torch_threads": torch.get_num_threads(),
              "host_rows_per_s": {}, "gather": {}}
    encs = {}
    for kind in KINDS:
        enc = encs[kind] = synthetic_encoded(kind, args.rows)
        result["host_rows_per_s"][kind] = host_rate(enc, args.batch)
        data = enc.to_device(dev, seq_width=T_DIN if kind == "din" else None)
        result["gather"][kind] = gather_time(enc, data, args.batch, dev)
        print(kind, result["host_rows_per_s"][kind], result["gather"][kind], file=sys.stderr)
        if kind == "din":
            result["epoch"] = din_epochs(enc, data, args.batch, dev, args.reps)
        del data
    result["device_after"] = gpu_info()
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "bench_input.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
