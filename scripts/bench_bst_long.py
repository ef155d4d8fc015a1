#!/usr/bin/env python
"""BST (fp32 block) across sequence lengths, below and above one 128-row tile.

    python scripts/bench_bst_long.py --out-dir DIR [--batch 2048] [--widths 20,50,128,129,256,512,1024]

Batches come from synthetic.bst_batch(B, T): lengths uniform in 1..T, Zipf ids over the real vocabulary sizes.
One transformer block, nhead 4, sum pooling.  For every length T:
  hot_us     the hot path alone: BSTModel.hot_path forward + its backward against fixed cotangents (side gather,
             rk_bst_block_fwd, rk_plan_build, rk_bst_block_bwd, the embedding-gradient reduction), one CUDA graph;
  step_us    the whole training step (forward, loss, backward), one CUDA graph;
both timed with CUDA events around each replay, L2 overwritten (a 256 MB fill) between replays.
  pairs      (query, live key) pairs of the attention: sum_b T * min(len_b, T);
  us_per_mpair   hot_us per 10^6 pairs;
  attn_tfma  attention FMAs / hot_us (10^12 FMA/s), with FMA_PER_PAIR per pair: 2 x 16 forward (scores, context)
             and 5 x 16 backward (scores recomputed, dP = dctx . v, dq, dk, dv), summed over the heads.  The
             kernels execute more than that (the max pass, the backward's recomputed forward); the rate is of
             the algorithmic count, and the hot path's other work (projections, FFN, gathers) is in hot_us.
At --aten-width (default 256) the oracle port of the reference model is also timed on the same GPU through
stock ATen kernels, eagerly and from a graph (bench.py's aten_cuda_run).
Prints one JSON object and writes it to DIR/bench_bst_long.json with the GPU's name, power limit and
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

D = 16
FMA_PER_PAIR = (2 + 5) * D
NHEAD = 4


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


def measure(vocab, B, T, steps, flush, dev):
    import rank_b200
    from rank_b200 import synthetic
    torch.manual_seed(0)
    model = rank_b200.BSTModel(vocab, dropout_rate=0.0, nhead=NHEAD, num_transformer_blocks=1,
                               max_seq_length=T).to(dev)
    model.train()
    b = synthetic.to_device(synthetic.bst_batch(B, T, 1000), dev)
    pairs = T * int(b["seq_length"].clamp(max=T).sum())
    gen = torch.Generator(device=dev).manual_seed(7)
    cots = []

    def hot():
        outs = model.hot_path(b["dense"], b["category"], b["seq_feedid"], b["seq_length"])
        if not cots:
            cots.extend(torch.randn(o.shape, generator=gen, device=dev) / B for o in outs)
        torch.autograd.backward(list(outs), cots)

    def step():
        logit = model(b["dense"], b["category"], b["seq_feedid"], b["seq_length"])[1]
        F.binary_cross_entropy_with_logits(logit.squeeze(), b["label"]).backward()

    hot_us = graph_time(hot, model, steps, flush)
    step_us = graph_time(step, model, steps, flush)
    rank_b200.check_index_errors()
    return {"T": T, "kernels": "long" if T > 128 else "short", "hot_us": round(hot_us, 1),
            "step_us": round(step_us, 1), "pairs": pairs, "us_per_mpair": round(1e6 * hot_us / pairs, 3),
            "attn_tfma": round(FMA_PER_PAIR * pairs / (hot_us * 1e-6) / 1e12, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", required=True)
    ap.add_argument("--batch", type=int, default=2048)
    ap.add_argument("--widths", default="20,50,128,129,256,512,1024")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--aten-width", type=int, default=256)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_bst_long needs a CUDA device")
    import rank_b200
    dev = torch.device("cuda:0")
    vocab = rank_b200.write_vocab_dir(tempfile.mkdtemp(prefix="rk_vocab_")) + "/"
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {"gpu": gpu_info(), "batch": args.batch, "nhead": NHEAD, "fma_per_pair": FMA_PER_PAIR, "rows": []}
    for T in [int(t) for t in args.widths.split(",")]:
        row = measure(vocab, args.batch, T, args.steps, flush, dev)
        print(json.dumps(row), flush=True)
        out["rows"].append(row)
        torch.cuda.empty_cache()

    class Wide(bench.BSTWorkload):
        def model(self, ns, oracle, vocab_dir):
            cls = ns.OracleBST if oracle else ns.BSTModel
            return cls(vocab_dir, dropout_rate=0.0, nhead=NHEAD, num_transformer_blocks=1,
                       max_seq_length=args.aten_width)

        def make_batch(self, B, seed):
            from rank_b200 import synthetic
            return synthetic.bst_batch(B, args.aten_width, seed)

    out["aten_cuda"] = {"T": args.aten_width,
                        **bench.aten_cuda_run(Wide(), args.batch, args.steps, 3, dev, flush, vocab)}
    print(json.dumps(out["aten_cuda"]), flush=True)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "bench_bst_long.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
