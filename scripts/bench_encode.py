#!/usr/bin/env python
"""Frame encoding timings: the host encoder against DeviceWechat.from_frame (csrc/encode.cu).

    python scripts/bench_encode.py --out-dir DIR [--rows 3320000] [--kinds din,bst,dcn,deepcrossing,deepfm]

Workload: a seeded synthetic frame shaped like the WeChat challenge training set (`--rows` rows; ids as
decimal strings over the real vocabulary sizes plus 2 % unknown ids; `device` integer-typed, as in the
challenge data; DIN histories comma-joined as the ETL writes them, 30 % empty, the rest 1..50 items; 16 dense
columns and the label), written to parquet under a temporary directory and read back with pandas.  The
vocabulary files hold the decimal ids 1..V.

Per kind, each a wall time ending in a device synchronise:
  host:      EncodedWechat(frame, ...).to_device(device) (pandas / numpy on the host, then the upload);
  device:    DeviceWechat.from_frame(frame, ...), split into its encode kernels (CUDA events around every
             encode entry point, `_lib.CallTimer`) and its host-to-device copies (torch.profiler, in a
             separate run); the rest is host work (Arrow conversion, dense columns, vocabulary files);
  pyarrow:   a vectorised host restatement with pyarrow.compute (`index_in` per column, `split_pattern` +
             `index_in` for DIN's history), then the same upload; a baseline kept in this script only.
The parquet read is timed once.  Prints one JSON object and writes it to DIR/bench_encode.json, with the
GPU's name and power limit read in the same run.  Needs a CUDA device.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import pandas as pd  # noqa: E402
import pyarrow as pa  # noqa: E402
import pyarrow.compute as pc  # noqa: E402
import torch  # noqa: E402

ENCODE_ENTRIES = ("rk_vocab_build", "rk_encode_strings", "rk_encode_split_count", "rk_encode_split")


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = ""
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": {"query": q, "value": out}}


def write_vocab(path, lines):
    from rank_b200.loader import VOCAB_FILES
    os.makedirs(path, exist_ok=True)
    for col, n in lines.items():
        with open(os.path.join(path, VOCAB_FILES[col]), "w") as f:
            f.write("\n".join(str(i) for i in range(1, n + 1)) + "\n")
    return path + "/"


def make_frame(n, lines, seed=0):
    from rank_b200.loader import DENSE_FEATURES, DIN_SEQ
    rng = np.random.default_rng(seed)

    def ids(col, k):
        v = rng.integers(1, lines[col] + 1, k)
        v[rng.random(k) < 0.02] += lines[col]          # unknown ids
        return pc.cast(pa.array(v), pa.large_string())

    cols = {c: ids(c, n) for c in ("userid", "feedid", "authorid", "bgm_song_id", "bgm_singer_id", "manual_tag_list")}
    cols["device"] = pa.array(rng.integers(1, 3, n))
    lens = rng.integers(1, 51, n) * (rng.random(n) >= 0.3)
    offsets = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    items = pa.LargeListArray.from_arrays(pa.array(offsets), ids("feedid", int(offsets[-1])))
    cols[DIN_SEQ] = pc.binary_join(items, pa.scalar(",", pa.large_string()))
    for c in DENSE_FEATURES:
        cols[c] = pa.array(np.log1p(rng.poisson(3.0, n)).astype(np.float64))
    cols["read_comment"] = pa.array((rng.random(n) < 0.3).astype(np.int64))
    return pa.table(cols)


def pyarrow_encode(frame, vocab_dir, kind, max_seq_length, device):
    """EncodedWechat's arrays computed with pyarrow.compute on the host (string columns only), uploaded."""
    from rank_b200.loader import (DENSE_FEATURES, DIN_SEQ, VOCAB_FILES, _float_column, category_columns,
                                  load_vocab_index)
    n = len(frame)
    tables = {}

    def lookup(col, values):
        if col not in tables:
            index = load_vocab_index(vocab_dir, VOCAB_FILES[col])
            tables[col] = (pa.array(list(index), type=pa.large_string()),
                           np.fromiter(index.values(), dtype=np.int64, count=len(index)))
        keys, pos = tables[col]
        at = pc.index_in(values, value_set=keys).to_numpy(zero_copy_only=False)
        hit = ~np.isnan(at) if at.dtype.kind == "f" else np.ones(len(at), dtype=bool)
        out = np.zeros(len(values), dtype=np.int64)
        out[hit] = pos[at[hit].astype(np.int64)]
        return out

    def strings(s):
        a = pa.array(s, type=pa.large_string(), from_pandas=True)
        return a.combine_chunks() if isinstance(a, pa.ChunkedArray) else a

    def cat(col):
        s = frame[col]
        if pd.api.types.is_numeric_dtype(s.dtype):
            return np.zeros(n, dtype=np.int64)
        return lookup(col, strings(s))

    arrays = [_float_column(frame, "read_comment", n)]
    arrays += [cat(c) for c in category_columns(kind)]
    if kind != "deepfm":
        arrays.append(np.stack([_float_column(frame, c, n) for c in DENSE_FEATURES], axis=1))
    if kind == "din":
        arrays.append(cat("feedid"))
        split = pc.split_pattern(strings(frame[DIN_SEQ]), ",")
        offsets = np.asarray(split.offsets, dtype=np.int64)
        arrays += [lookup("feedid", split.flatten()), offsets - offsets[0]]
    if kind == "bst":
        seq = np.zeros((n, max_seq_length), dtype=np.int64)
        if max_seq_length:
            seq[:, 0] = cat("feedid")
        arrays += [seq, np.full(n, min(1, max_seq_length), dtype=np.int64)]
    return [torch.from_numpy(np.ascontiguousarray(a)).to(device) for a in arrays]


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", required=True)
    ap.add_argument("--rows", type=int, default=3_320_000)
    ap.add_argument("--kinds", default="din,bst,dcn,deepcrossing,deepfm")
    ap.add_argument("--max-seq-length", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_encode.py needs a CUDA device")
    import rank_b200
    from rank_b200 import _lib
    from rank_b200.loader import EncodedWechat
    from rank_b200.vocab import WECHAT_VOCAB_LINES

    dev = torch.device("cuda:0")
    os.makedirs(args.out_dir, exist_ok=True)
    result = {"rows": args.rows, "host_cores": os.cpu_count(), **gpu_info(), "kinds": {}}
    with tempfile.TemporaryDirectory(prefix="rk_bench_encode_") as tmp:
        vocab = write_vocab(os.path.join(tmp, "vocab"), WECHAT_VOCAB_LINES)
        path = os.path.join(tmp, "frame.parquet")
        import pyarrow.parquet as pq
        pq.write_table(make_frame(args.rows, WECHAT_VOCAB_LINES), path)
        result["parquet_mb"] = round(os.path.getsize(path) / 2 ** 20, 1)
        read_s, frame = timed(lambda: pd.read_parquet(path))
        result["parquet_read_s"] = round(read_s, 3)
        T = args.max_seq_length
        rank_b200.DeviceWechat.from_frame(frame.iloc[:1000], vocab, "din", dev)      # warm-up: module load
        for kind in args.kinds.split(","):
            host_s, want = timed(lambda: EncodedWechat(frame, vocab, kind, max_seq_length=T).to_device(dev))
            dev_s, got = timed(lambda: rank_b200.DeviceWechat.from_frame(frame, vocab, kind, dev, max_seq_length=T))
            same = all(torch.equal(a, b) for (_, a), (_, b) in zip(got._leaves, want._leaves) if a is not None)
            if kind == "din":
                same = same and torch.equal(got.seq_flat, want.seq_flat) and torch.equal(got.seq_offsets,
                                                                                         want.seq_offsets)
            del want, got
            with _lib.CallTimer() as ct:
                rank_b200.DeviceWechat.from_frame(frame, vocab, kind, dev, max_seq_length=T)
            calls = ct.summary()
            kernel_ms = sum(ms for name, (_, ms) in calls.items() if name in ENCODE_ENTRIES)
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                rank_b200.DeviceWechat.from_frame(frame, vocab, kind, dev, max_seq_length=T)
                torch.cuda.synchronize()
            copy_us = sum(e.device_time_total for e in prof.key_averages() if "HtoD" in e.key)
            pa_s, _ = timed(lambda: pyarrow_encode(frame, vocab, kind, T, dev))
            row = {"host_s": round(host_s, 3), "device_s": round(dev_s, 3), "device_kernels_ms": round(kernel_ms, 2),
                   "device_copies_ms": round(copy_us / 1e3, 2), "pyarrow_s": round(pa_s, 3),
                   "host_rows_per_s": round(args.rows / host_s), "device_rows_per_s": round(args.rows / dev_s),
                   "pyarrow_rows_per_s": round(args.rows / pa_s), "bit_identical": bool(same),
                   "encode_calls": {k: v[0] for k, v in calls.items() if k in ENCODE_ENTRIES}}
            result["kinds"][kind] = row
            print(kind, json.dumps(row), flush=True)
    with open(os.path.join(args.out_dir, "bench_encode.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
