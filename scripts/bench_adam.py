#!/usr/bin/env python
"""The full training step — zero_grad, forward, loss, backward AND the optimizer — with four optimizer set-ups.

    python scripts/bench_adam.py --out-dir DIR [--steps 100] [--warmup 10] [--workloads deepfm,dcn,din_tc,bst_tc]

Workloads, models and batches are bench.py's (DeepFM at B = 1024, the others at 8192).  Variants:
  a  dense table gradients, forward/backward replayed from a CUDA graph, then the default torch.optim.Adam
     (foreach, step count on the host) run eagerly: what the reference does;
  b  dense table gradients, torch.optim.Adam(fused=True, capturable=True) inside the graph;
  c  dense table gradients, rank_b200.Adam inside the graph;
  d  touched-rows table gradients (sparse.set_table_gradients("touched")), rank_b200.Adam inside the graph.
All four start from the same weights and see the same batches and per-call weight draws; their steps alternate
within one process.  Per step: CUDA events around the step (for a: the replay plus the eager optimizer), 256 MiB
written between steps to evict L2, outside the events, as bench.py does.
  opt_ms    : the optimizer alone.  a: events between the end of the replay and the end of the eager optimizer;
              b, c, d: a CUDA graph of optimizer.step() alone, over gradients of one eager backward, replayed with
              L2 evicted before each replay;
  opt_bytes : bytes the update needs, from shapes: p, m, v read and written plus the gradient read (28 B per
              element), or, for touched tables, 24 B per element plus the touched rows (8 B row id + 4 B per
              value) of that backward;
  b_equals_c: the parameters of b and c are bit-identical after all steps.
Prints one JSON object and writes it to DIR/bench_adam.json, with the GPU name, power limit and max SM clock
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

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import torch  # noqa: E402

import bench  # noqa: E402

VARIANTS = ("a", "b", "c", "d")


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = ""
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": {"query": q, "value": out}}


class TrainStep(bench.Stepper):
    """bench.Stepper (zero_grad, forward, loss, backward replayed from a CUDA graph) with the optimizer step
    inside the graph, or run eagerly after each replay."""

    def __init__(self, model, wl, example, opt, in_graph, mode):
        from rank_b200 import sparse
        self.opt, self.in_graph = opt, in_graph
        sparse.set_table_gradients(mode)        # read while the graph is captured; replays keep what it recorded
        try:
            super().__init__(model, wl, example, True, None)
        finally:
            sparse.set_table_gradients("dense")

    def _body(self):
        super()._body()
        if self.in_graph:
            self.opt.step()

    def run(self, seed, before_replay=None, mid=None):
        loss = super().run(seed, before_replay)
        if not self.in_graph:
            if mid is not None:
                mid.record()
            self.opt.step()
        return loss


def make_optimizer(kind, model, lr):
    import rank_b200
    if kind == "a":
        return torch.optim.Adam(model.parameters(), lr)
    if kind == "b":
        return torch.optim.Adam(model.parameters(), lr, fused=True, capturable=True)
    return rank_b200.Adam(model.parameters(), lr)


def optimizer_alone(st, kind, flush, reps, pool):
    """Device time and bytes of the optimizer by itself, over the gradients of one eager backward."""
    from rank_b200 import sparse
    model, opt = st.model, st.opt
    model.zero_grad(set_to_none=True)
    if hasattr(model, "ephemeral_frozen"):
        model.ephemeral_frozen = False
    st.load(pool[0])
    sparse.set_table_gradients("touched" if kind == "d" else "dense")
    try:
        torch.manual_seed(1)
        st.wl.loss(model, st.static).backward()
    finally:
        sparse.set_table_gradients("dense")
    nbytes = 0
    touched = {}
    for p in model.parameters():
        t = getattr(p, "touched_grad", None)
        if t is not None:
            touched[p] = t
            nbytes += 24 * p.numel() + int(t.count.item()) * (8 + 4 * p.shape[1])
        elif p.grad is not None:
            nbytes += 28 * p.numel()
    if kind == "a":
        return None, nbytes
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for p, t in touched.items():
            p.touched_grad = t
        opt.step()
    evs = []
    for i in range(reps + 3):
        flush.fill_(i & 0xff)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        graph.replay()
        e.record()
        if i >= 3:
            evs.append((s, e))
    torch.cuda.synchronize()
    return statistics.median(s.elapsed_time(e) for s, e in evs), nbytes


def run_workload(key, steps, warmup, flush, lr):
    import rank_b200
    from rank_b200.staging import PackedBatch
    wl = bench.WORKLOADS[key]()
    dev = torch.device("cuda", 0)
    B = wl.batch
    vocab = rank_b200.write_vocab_dir(tempfile.mkdtemp(prefix="rk_vocab_")) + "/"
    raw = [wl.make_batch(B, 1000 + i) for i in range(4)]
    pool = [PackedBatch.like(b, dev).fill(b) for b in raw]
    for pb in pool:
        pb.to_device()
    torch.cuda.synchronize()
    steppers = {}
    for v in VARIANTS:
        torch.manual_seed(0)                                 # identical weights in all four
        model = wl.model(rank_b200, False, vocab).to(dev)
        model.train()
        opt = make_optimizer(v, model, lr)
        steppers[v] = TrainStep(model, wl, pool[0], opt, in_graph=v != "a", mode="touched" if v == "d" else "dense")
    times = {v: [] for v in VARIANTS}
    opt_a = []
    for i in range(warmup + steps):
        for v in VARIANTS:
            st = steppers[v]
            st.load(pool[i % 4])
            flush.fill_(i & 0xff)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            mid = torch.cuda.Event(enable_timing=True) if v == "a" else None
            s.record()
            st.run(10_000 + i, mid=mid)
            e.record()
            if i >= warmup:
                times[v].append((s, e))
                if mid is not None:
                    opt_a.append((mid, e))
    torch.cuda.synchronize()
    pb, pc = list(steppers["b"].model.parameters()), list(steppers["c"].model.parameters())
    b_equals_c = all(torch.equal(x, y) for x, y in zip(pb, pc))
    pd = list(steppers["d"].model.parameters())
    d_vs_c = max(float((x - y).detach().abs().max()) for x, y in zip(pd, pc))
    out = {"workload": wl.name, "batch": B, "steps": steps, "lr": lr, "b_equals_c": b_equals_c,
           "d_vs_c_max_abs_diff": d_vs_c,
           "params": sum(p.numel() for p in pc), "tensors": len(pc)}
    for v in VARIANTS:
        ms = [s.elapsed_time(e) for s, e in times[v]]
        opt_ms, nbytes = optimizer_alone(steppers[v], v, flush, steps, pool)
        if v == "a":
            opt_ms = statistics.median(s.elapsed_time(e) for s, e in opt_a)
        out[v] = {"ms_per_step_mean": statistics.mean(ms), "ms_per_step_median": statistics.median(ms),
                  "opt_ms": opt_ms, "opt_bytes": nbytes, "opt_gbs": nbytes / (opt_ms * 1e-3) / 1e9}
        print(json.dumps({"workload": key, "variant": v, **out[v]}), file=sys.stderr)
    del steppers
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out-dir", required=True)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--lr", type=float, default=1e-3)
    ap.add_argument("--workloads", default="deepfm,dcn,din_tc,bst_tc")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_adam.py needs a CUDA device"
    torch.cuda.set_device(0)
    flush = torch.empty(bench.L2_FLUSH_BYTES, dtype=torch.uint8, device="cuda")
    result = {"card": gpu_info(), "workloads": {}}
    for key in args.workloads.split(","):
        result["workloads"][key] = run_workload(key, args.steps, args.warmup, flush, args.lr)
    result["card_after"] = gpu_info()["nvidia_smi"]
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "bench_adam.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
