#!/usr/bin/env python
"""Weight and bias gradients of the towers' nn.Linear layers (dW = g^T x, db = g.sum(0); the GEMM's K is the batch).

For every Linear that run_tower meets in bench.py's workloads (DIN, BST, DCN at B = 8192, DeepFM at B = 1024) it
times rk_linear_wgrad (csrc/linear.cu) next to what autograd runs (g.t() @ x, then g.sum(0)), each captured in a
CUDA graph, with L2 warm (the same operands replayed) and flushed (256 MB written between replays, the flush timed
alone and subtracted).  TFLOP/s count the 2*B*N*K FLOP of dW; the peak is 128 fp32 FMA lanes x 2 per SM at the
SM clock read in the same run.  "tf32" is the share of the data-sheet dense TF32 tensor rate of one B200 (1,125
TFLOP/s) that the three products of rk_linear_wgrad's 3xTF32 scheme (6*B*N*K FLOP) would take at that time.
--cublas-variants adds the other cuBLAS forms of dW.   python scripts/bench_mm.py
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rank_b200 import _lib  # noqa: E402

SHAPES = {   # workload: (B, [(in, out), ...])
    "din": (8192, [(82, 512), (512, 256), (256, 128)]),
    "bst": (8192, [(66, 512), (512, 256), (256, 128), (128, 1)]),
    "dcn": (8192, [(50, 512), (512, 256), (256, 128)]),
    "deepfm": (1024, [(96, 512), (512, 256), (256, 128)]),
}


TF32_DENSE_TFLOPS = 1125.0          # NVIDIA HGX B200 data sheet, one GPU, dense


def graph_us(fn, flush=None, n=50):
    """Mean µs of fn per replay of a CUDA graph holding it (after `flush` in the same graph, timed alone too)."""
    for _ in range(3):
        fn()
    def make(body):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            body()
        return g
    def time(g):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g.replay()
        torch.cuda.synchronize()
        s.record()
        for _ in range(n):
            g.replay()
        e.record()
        torch.cuda.synchronize()
        return 1e3 * s.elapsed_time(e) / n
    if flush is None:
        return time(make(fn))
    return time(make(lambda: (flush(), fn()))) - time(make(flush))


def max_sm_clock_mhz():
    out = subprocess.run(["nvidia-smi", "--query-gpu=clocks.max.sm", "--format=csv,noheader,nounits"],
                         capture_output=True, text=True, check=True).stdout
    return float(out.split()[0])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cublas-variants", action="store_true")
    args = ap.parse_args()
    dev = torch.device("cuda")
    lib = _lib.load()
    props = torch.cuda.get_device_properties(dev)
    mhz = max_sm_clock_mhz()
    peak = props.multi_processor_count * 128 * 2 * mhz * 1e6 / 1e12
    print(f"{props.name}, {props.multi_processor_count} SMs, max SM clock {mhz:.0f} MHz: fp32 FMA peak "
          f"{peak:.1f} TFLOP/s", flush=True)
    junk = torch.empty(256 << 18, device=dev)
    flush = lambda: junk.fill_(1.0)                   # noqa: E731
    totals = {}
    for work, (B, shapes) in SHAPES.items():
        for k_in, n_out in shapes:
            x = torch.randn(B, k_in, device=dev)
            g = torch.randn(B, n_out, device=dev)
            dW, db = torch.empty(n_out, k_in, device=dev), torch.empty(n_out, device=dev)
            partials = torch.empty(max(1, lib.rk_linear_wgrad_scratch_floats(B, k_in, n_out)), device=dev)

            def ours():
                _lib.check(lib.rk_linear_wgrad(x.data_ptr(), k_in, g.data_ptr(), n_out, B, k_in, n_out, dW.data_ptr(),
                                               db.data_ptr(), partials.data_ptr(), _lib.stream_ptr()),
                           "rk_linear_wgrad")

            def torch_ref():
                g.t() @ x
                g.sum(0)

            ours()
            ref_w, ref_b = g.t() @ x, g.sum(0)
            assert (dW - ref_w).abs().max() <= 1e-4 * ref_w.abs().max() and (db - ref_b).abs().max() <= 1e-3
            flop = 2.0 * B * n_out * k_in
            row = {}
            for l2, fl in (("warm", None), ("flushed", flush)):
                row[("ours", l2)] = graph_us(ours, fl)
                row[("torch", l2)] = graph_us(torch_ref, fl)
            for key, us in row.items():
                totals[(work,) + key] = totals.get((work,) + key, 0.0) + us
            print(f"{work:6s} B={B} {k_in:3d}->{n_out:3d}: " + ", ".join(
                f"{impl} {l2} {us:6.1f} us ({flop / us / 1e6:5.1f} TFLOP/s, {100 * flop / us / 1e6 / peak:4.1f}% peak, "
                f"tf32 {100 * 3 * flop / us / 1e6 / TF32_DENSE_TFLOPS:4.1f}%)"
                for (impl, l2), us in row.items()), flush=True)
            if args.cublas_variants:
                res = {"dW g.t().contiguous()@x": graph_us(lambda: g.t().contiguous() @ x),
                       "dW (x.t()@g).t()": graph_us(lambda: (x.t() @ g).t()),
                       "dW x.t().contiguous()@g": graph_us(lambda: x.t().contiguous() @ g),
                       "db ones@g": graph_us(lambda: torch.ones(1, B, device=dev) @ g)}
                print("        warm: " + ", ".join(f"{k} {v:.1f}us" for k, v in res.items()), flush=True)
    for work in SHAPES:
        print(f"{work:6s} tower dW + db total: " + ", ".join(
            f"{impl} {l2} {totals[(work, impl, l2)]:.1f} us" for impl in ("ours", "torch") for l2 in ("warm", "flushed")))


if __name__ == "__main__":
    main()
