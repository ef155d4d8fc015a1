#!/usr/bin/env python
"""Timings of the data-parallel evaluation metrics (BinaryMetrics.all_gather, csrc/metrics.cu rk_metrics_merge).

    torchrun --nproc-per-node N scripts/bench_metrics_dp.py --out-dir DIR

An evaluation set of 2^20 and of 8 * 2^20 samples is split evenly over the N ranks, with scores rounded to
1e-3 (ties), 3.56 % positives and Zipf users over the 19 627-row userid table.  Every rank fills its
BinaryMetrics with update(), then, per size:
    gather_ms : CUDA events around all_gather() (one all_gather_into_tensor per buffer + the merge launch),
                median over --reps, after a barrier each time so that no rank waits for a late one;
    compute_ms: CUDA events around compute() on the merged buffers (its two device->host reads included);
    host_ms   : the hand-written alternative, host clock: every rank copies its samples to the host,
                all_gather_object collects them, rank 0 runs sklearn's roc_auc_score and a per-user
                roc_auc_score loop (uAUC).  Once; --no-host skips it.
The L2 cache is not flushed between repetitions: at 2^20 samples the gathered and merged buffers (32 MB)
fit in it, at 8 * 2^20 (256 MB) they do not.  Rank 0 prints one JSON object, with every GPU's name and power
limit read in the same run, and writes it to DIR/bench_metrics_dp_n{N}.json.  Needs CUDA devices and NCCL.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

USERS = 19627


def gpu_info():
    q = "index,name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    except (OSError, subprocess.TimeoutExpired):
        out = []
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": {"query": q, "value": out}}


def rank_data(total, rank, world, seed=1):
    """This rank's share of the evaluation set, drawn from one global stream so that the union over the
    ranks is the same set at every N."""
    rng = np.random.default_rng(seed)
    w = np.arange(1, USERS + 1, dtype=np.float64) ** -1.05
    users = rng.permutation(USERS)[rng.choice(USERS, size=total, p=w / w.sum())].astype(np.int64)
    labels = (rng.random(total) < 0.0356).astype(np.float32)
    scores = np.round(rng.random(total), 3).astype(np.float32)
    per = total // world
    sl = slice(rank * per, (rank + 1) * per)
    return scores[sl], labels[sl], users[sl]


def sklearn_metrics(s, y, u):
    from sklearn.metrics import roc_auc_score
    auc = roc_auc_score(y, s)
    order = np.argsort(u, kind="stable")
    cuts = np.flatnonzero(np.diff(u[order])) + 1
    total, count = 0.0, 0
    for idx in np.split(order, cuts):
        yy = y[idx]
        if yy.min() != yy.max():
            total += roc_auc_score(yy, s[idx])
            count += 1
    return auc, total / count


def event_ms(fn, reps):
    ts = []
    for _ in range(reps):
        dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return {"median": statistics.median(ts), "min": min(ts), "reps": reps}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out-dir", required=True)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--sizes", default=f"{2 ** 20},{8 * 2 ** 20}")
    ap.add_argument("--no-host", action="store_true", help="skip the host all_gather_object + sklearn alternative")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_metrics_dp.py needs CUDA devices")
    import rank_b200
    from rank_b200.metrics import BinaryMetrics
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    rank, world = dist.get_rank(), dist.get_world_size()
    rows = []
    for total in (int(x) for x in args.sizes.split(",")):
        s, y, u = rank_data(total, rank, world)
        m = BinaryMetrics(len(s), dev, USERS)
        m.update(*(torch.from_numpy(a).to(dev) for a in (s, y, u)))
        merged = m.all_gather()                   # the eager first call: configuration check, allocation
        out = merged.compute()
        row = {"n": total, "per_rank": len(s), "gather_ms": event_ms(m.all_gather, args.reps),
               "compute_ms": event_ms(merged.compute, args.reps), "auc": out["auc"], "uauc": out["uauc"]}
        if not args.no_host:
            dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n = int(m._state[0])
            mine = tuple(t[:n].cpu().numpy() for t in (m.scores, m.labels, m.groups))
            every = [None] * world
            dist.all_gather_object(every, mine)
            if rank == 0:
                auc, uauc = sklearn_metrics(*(np.concatenate([e[i] for e in every]) for i in range(3)))
                row["host_ms"] = 1e3 * (time.perf_counter() - t0)
                row["host_vs_device"] = {"auc": abs(auc - out["auc"]), "uauc": abs(uauc - out["uauc"])}
            dist.barrier()
        if rank == 0:
            print(json.dumps(row), file=sys.stderr)
        rows.append(row)
        del m, merged
        torch.cuda.empty_cache()
    if rank == 0:
        result = {"world": world, **gpu_info(), "abi": rank_b200._lib.ABI_VERSION, "rows": rows}
        os.makedirs(args.out_dir, exist_ok=True)
        with open(os.path.join(args.out_dir, f"bench_metrics_dp_n{world}.json"), "w") as f:
            json.dump(result, f, indent=1)
        print(json.dumps(result))
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
