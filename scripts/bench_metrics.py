#!/usr/bin/env python
"""Timings of the device metrics (csrc/metrics.cu, rank_b200.metrics).

    python scripts/bench_metrics.py --out-dir DIR

1. BinaryMetrics.compute() at n = 2^20 and 8 * 2^20, untied (uniform fp32 scores) and tied (scores
   rounded to 1e-3), without and with groups (Zipf users over the 19 627-row userid table):
     device_ms : CUDA events around rk_metrics_compute (the kernels alone);
     wall_ms   : host clock around compute(), both device->host reads included;
   and for the AUC alone, on the same data:
     torch_ms  : an exact AUC in plain torch on the same GPU (torch.sort + unique_consecutive + cumsum);
     sklearn_ms: roc_auc_score on the host, the device->host copy of scores and labels included.
2. The per-step cost of update() inside a captured DIN training step (zero_grad, forward, loss,
   backward; batch 8192, T = 50, tensor-core activation unit), against the reference's per-step
   `loss.item(); label.cpu(); prob.cpu()` after the same step.

Prints one JSON object and writes it to DIR/bench_metrics.json, with the GPU name and power limit read
in the same run.  Needs a CUDA device.
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

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

USERS = 19627


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = ""
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": {"query": q, "value": out}}


def torch_auc(s, y):
    """Exact tie-averaged AUC with stock torch ops: runs of equal scores, pos_r (2 neg_before_r + neg_r)."""
    ss, idx = torch.sort(s)
    pos = y[idx].to(torch.int64)
    _, counts = torch.unique_consecutive(ss, return_counts=True)
    ends = torch.cumsum(counts, 0)
    cpos = torch.cumsum(pos, 0)
    pos_end = cpos[ends - 1]
    pos_r = pos_end - torch.cat([pos_end.new_zeros(1), pos_end[:-1]])
    neg_r = counts - pos_r
    neg_before = torch.cumsum(neg_r, 0) - neg_r
    u2 = int((pos_r * (2 * neg_before + neg_r)).sum())
    P = int(pos_r.sum())
    N = int(neg_r.sum())
    return u2 / (2 * P * N)


def median_ms(fn, reps, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(1e3 * (time.perf_counter() - t0))
    return statistics.median(ts)


def bench_compute(dev, reps):
    from sklearn.metrics import roc_auc_score
    from rank_b200 import _lib, synthetic
    from rank_b200.metrics import BinaryMetrics
    lib = _lib.load()
    gen = torch.Generator().manual_seed(1)
    rows = []
    for n in (1 << 20, 8 << 20):
        users = synthetic.zipf_indices(gen, USERS, (n,)).to(dev)
        y = (torch.rand(n, generator=gen) < synthetic.LABEL_RATE).float().to(dev)
        for tied in (False, True):
            s = torch.rand(n, generator=gen)
            if tied:
                s = torch.round(s * 1000) / 1000
            s = s.to(dev)
            for groups in (None, USERS):
                m = BinaryMetrics(n, dev, groups)
                m.update(s, y, users if groups else None)
                out = m.compute()
                G = groups or 0
                args = (m.scores.data_ptr(), m.labels.data_ptr(), _lib.ptr(m.groups), n, G, m._ws.data_ptr(),
                        m._ws.numel(), m._result.data_ptr())
                for _ in range(3):
                    _lib.check(lib.rk_metrics_compute(*args, _lib.stream_ptr()), "rk_metrics_compute")
                evs = []
                for _ in range(reps):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    _lib.check(lib.rk_metrics_compute(*args, _lib.stream_ptr()), "rk_metrics_compute")
                    b.record()
                    evs.append((a, b))
                torch.cuda.synchronize()
                row = {"n": n, "tied": tied, "groups": groups,
                       "device_ms": statistics.median(a.elapsed_time(b) for a, b in evs),
                       "wall_ms": median_ms(m.compute, reps), "auc": out["auc"], "uauc": out.get("uauc")}
                if groups is None:
                    ref = torch_auc(s, y)
                    assert abs(ref - out["auc"]) <= 1e-12, (ref, out["auc"])
                    row["torch_ms"] = median_ms(lambda: torch_auc(s, y), reps)
                    row["sklearn_ms"] = median_ms(lambda: roc_auc_score(y.cpu().numpy(), s.cpu().numpy()), 2,
                                                  warmup=1)
                rows.append(row)
                print(json.dumps(row), file=sys.stderr)
                del m
    return rows


def bench_step(dev, steps):
    import rank_b200
    from rank_b200 import synthetic
    from rank_b200.metrics import BinaryMetrics
    B, T = 8192, 50
    vocab = rank_b200.write_vocab_dir(tempfile.mkdtemp(prefix="rk_vocab_")) + "/"
    torch.manual_seed(0)
    model = rank_b200.DIN(vocab, dropout_rate=0.0, use_softmax=False, l2_lambda=0.2).to(dev)
    model.activation_unit_precision = "bf16"
    model.train()
    static = synthetic.to_device(synthetic.din_batch(B, T, 7), dev)
    metrics = BinaryMetrics(B * (2 * steps + 16), dev, num_groups=USERS)
    out = {}

    def body(with_metrics):
        prob, _, l2 = model(static["dense"], static["category"], static["sequence"], static["target"])
        loss = F.binary_cross_entropy(prob.squeeze(), static["label"]) + l2
        loss.backward()
        if with_metrics:
            metrics.update(prob.detach(), static["label"], static["category"]["userid"])
        return loss, prob

    graphs = {}
    for with_metrics in (False, True):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                model.zero_grad(set_to_none=True)
                body(with_metrics)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        model.zero_grad(set_to_none=True)
        if hasattr(model, "draw_ephemeral"):
            model.draw_ephemeral()
            model.ephemeral_frozen = True
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            res = body(with_metrics)
        graphs[with_metrics] = (g, res)
    metrics.reset()

    def device_ms(g):
        for _ in range(5):
            g.replay()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            g.replay()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / steps

    plain, with_update = graphs[False][0], graphs[True][0]
    # alternate the two graphs so drift of the shared machine hits both alike
    d_plain, d_upd = [], []
    for _ in range(3):
        d_plain.append(device_ms(plain))
        metrics.reset()
        d_upd.append(device_ms(with_update))
        metrics.reset()
    out["graph_step_ms"] = statistics.median(d_plain)
    out["graph_step_with_update_ms"] = statistics.median(d_upd)
    out["update_cost_us"] = 1e3 * (out["graph_step_with_update_ms"] - out["graph_step_ms"])

    loss, prob = graphs[False][1]

    def reference_pattern():
        for _ in range(steps):
            plain.replay()
            loss.item()
            static["label"].cpu()
            prob.cpu()

    def device_pattern():
        for _ in range(steps):
            with_update.replay()

    w_ref, w_dev = [], []
    for _ in range(3):
        w_ref.append(median_ms(reference_pattern, 1, warmup=1) / steps)
        metrics.reset()
        w_dev.append(median_ms(device_pattern, 1, warmup=1) / steps)
        metrics.reset()
    out["wall_step_item_cpu_ms"] = statistics.median(w_ref)
    out["wall_step_update_ms"] = statistics.median(w_dev)
    out.update(batch=B, T=T, steps=steps, workload="DIN raw attention, tensor-core activation unit, graph replay")
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out-dir", required=True)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--steps", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_metrics.py needs a CUDA device")
    dev = torch.device("cuda:0")
    result = {"device": gpu_info(), "compute": bench_compute(dev, args.reps), "step": bench_step(dev, args.steps)}
    result["device_after"] = gpu_info()
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "bench_metrics.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
