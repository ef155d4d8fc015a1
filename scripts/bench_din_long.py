#!/usr/bin/env python
"""DIN (fp32 activation unit) across history widths, below and above one 128-row tile.

    python scripts/bench_din_long.py --out-dir DIR [--batch 8192] [--widths 50,128,129,256,512,1024]

Batches come from synthetic.din_batch(B, T): 30 % of the histories empty, the rest of uniform length 1..T;
Zipf ids over the real vocabulary sizes.  For every width T and both attention modes (raw, softmax):
  hot_us     the hot path alone: DIN.hot_path forward + its backward against fixed cotangents (rk_din_fwd,
             rk_plan_build, rk_din_bwd, the embedding-gradient reduction), one CUDA graph;
  step_us    the whole training step (forward, loss, backward), one CUDA graph;
both timed with CUDA events around each replay, L2 overwritten (a 256 MB fill) between replays.
  live       history positions that run through the activation unit: sum_b min(len_b, T);
  us_per_live_k  hot_us per 1000 live positions;
  gbps       algorithmic bytes / hot_us, with the SURVEY.md 8(d) DIN row per live position:
             forward 8 B of index + 64 B of embedding row, backward the row re-read (64 B) + 3 x 64 B of
             gradient rows (per-occurrence write, sorted read, unique write) = 328 B per live position
             (the per-sample columns and the empty softmax histories are left out);
  tflops     activation-unit FLOPs / hot_us: 2 (4D*64 + 64*32 + 32) per live position forward, the same
             again backward (the weight gradient is never needed).
At --aten-width (default 256) the oracle port of the reference model is also timed on the same GPU through
stock ATen kernels, eagerly and from a graph (bench.py's aten_cuda_run).
Prints one JSON object and writes it to DIR/bench_din_long.json with the GPU's name, power limit and
maximum SM clock read in the same run.  Needs a CUDA device.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import bench  # noqa: E402

BYTES_PER_LIVE = 8 + 64 + 64 + 3 * 64
D = 16
FLOPS_PER_LIVE = 2 * 2 * (4 * D * 64 + 64 * 32 + 32)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def graph_time(body, model, steps, flush):
    """Mean device time (us) of `body` replayed from a CUDA graph, L2 overwritten before every replay."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            model.zero_grad(set_to_none=True)
            body()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    model.zero_grad(set_to_none=True)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        body()
    for _ in range(3):
        graph.replay()
    evs = []
    for i in range(steps):
        flush.fill_(i & 0xff)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        graph.replay()
        e.record()
        evs.append((s, e))
    torch.cuda.synchronize()
    del graph
    return 1e3 * sum(s.elapsed_time(e) for s, e in evs) / steps


def measure(vocab, B, T, soft, steps, flush, dev):
    import rank_b200
    from rank_b200 import synthetic
    torch.manual_seed(0)
    model = rank_b200.DIN(vocab, dropout_rate=0.0, use_softmax=soft, l2_lambda=0.2).to(dev)
    model.train()
    model.draw_ephemeral()
    model.ephemeral_frozen = True           # one fixed draw of the per-call weights: a graph cannot hold CPU draws
    b = synthetic.to_device(synthetic.din_batch(B, T, 1000), dev)
    length = b["sequence"]["his_read_comment_7d_seq_length"].clamp(max=T)
    live = int(length.sum())
    gen = torch.Generator(device=dev).manual_seed(7)
    cots = []

    def hot():
        outs = model.hot_path(b["dense"], b["category"], b["sequence"], b["target"])
        if not cots:
            cots.extend(torch.randn(o.shape, generator=gen, device=dev) / B for o in outs)
        torch.autograd.backward(list(outs), cots)

    def step():
        prob, _, l2 = model(b["dense"], b["category"], b["sequence"], b["target"])
        (F.binary_cross_entropy(prob.squeeze(), b["label"]) + l2).backward()

    hot_us = graph_time(hot, model, steps, flush)
    step_us = graph_time(step, model, steps, flush)
    rank_b200.check_index_errors()
    return {"T": T, "mode": "softmax" if soft else "raw", "hot_us": round(hot_us, 1), "step_us": round(step_us, 1),
            "live": live, "us_per_live_k": round(1e3 * hot_us / live, 4),
            "gbps": round(BYTES_PER_LIVE * live / (hot_us * 1e-6) / 1e9, 1),
            "tflops": round(FLOPS_PER_LIVE * live / (hot_us * 1e-6) / 1e12, 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", required=True)
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--widths", default="50,128,129,256,512,1024")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--aten-width", type=int, default=256)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_din_long needs a CUDA device")
    import rank_b200
    dev = torch.device("cuda:0")
    vocab = rank_b200.write_vocab_dir(tempfile.mkdtemp(prefix="rk_vocab_")) + "/"
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {"gpu": gpu_info(), "batch": args.batch, "bytes_per_live_position": BYTES_PER_LIVE,
           "flops_per_live_position": FLOPS_PER_LIVE, "rows": []}
    for T in [int(t) for t in args.widths.split(",")]:
        for soft in (False, True):
            row = measure(vocab, args.batch, T, soft, args.steps, flush, dev)
            print(json.dumps(row), flush=True)
            out["rows"].append(row)
            torch.cuda.empty_cache()

    class Wide(bench.DINWorkload):
        def make_batch(self, B, seed):
            from rank_b200 import synthetic
            return synthetic.din_batch(B, args.aten_width, seed)

    out["aten_cuda"] = {"T": args.aten_width, "mode": "raw",
                        **bench.aten_cuda_run(Wide(), args.batch, args.steps, 3, dev, flush, vocab)}
    print(json.dumps(out["aten_cuda"]), flush=True)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "bench_din_long.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
