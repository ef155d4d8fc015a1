#!/usr/bin/env python
"""bench.py — train samples/s (fwd+bwd) of the CTR hot path + unchanged torch tower on B200.

    python bench.py --gpus N --steps K --warmup W [--workload dcn] [--impl reference] [--dump-outputs DIR]

One "step" = zero_grad, forward, loss, backward of the whole model on one synthetic
WeChat-shaped batch (per-GPU batch fixed: weak scaling; for N > 1 the dense-gradient allreduce
is part of the step).  Rank 0 prints ONE JSON line (see DESIGN.md "Measurement").
  value     : device-timed (CUDA events), inputs already resident in HBM, max over ranks
  e2e       : same metric through the public module API with pinned HOST inputs, H2D copies and
              the D2H read of the loss inside the timed region
  roofline  : algorithmic bytes of the hot path (SURVEY.md §8d) / device time of a CUDA graph that
              holds ONLY the hot path of a step (model.hot_path forward + its backward incl. the
              embedding-gradient reduction), against MEASURED_PEAKS.json; by construction a subset of
              the step, and checked to be <= ms_per_step
  aten_cuda_baseline : the oracle port of the reference model on the SAME GPU through stock
              ATen/cuBLAS kernels (what the reference does with --device cuda), eager and replayed
              from a CUDA graph — the kernel-level bar of SURVEY.md §2.2 / §8d
  cpu_baseline / --impl reference : the oracle port of the reference model on the host cores
  other_workloads : one-line summaries of the other configurations (N = 1, default workload only)
  --dump-outputs DIR : after the timed steps, what the last of them handed its caller (loss, forward
              outputs, parameter gradients) as DIR/<name>.npy, so that two builds can be compared on the
              same seeded inputs
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

METRIC = "train samples/sec (fwd+bwd)"
L2_FLUSH_BYTES = 256 << 20
DUMP_BYTES = 64_000_000


# ------------------------------------------------------------------------------- workloads
class Workload:
    """One BASELINE.json config: how to build the model (ours or the oracle port), its batch,
    its loss, and the algorithmic bytes/flops per sample of its hot path (SURVEY.md §8d)."""
    name = ""
    batch = 8192
    bytes_per_sample = 0          # fwd + bwd, algorithmic
    flops_per_sample = 0
    bound = "hbm"
    dtype = "f32"
    hot_calls = ()                # ABI entry points that make up the hot path of a step

    def model(self, ns, oracle, vocab_dir):
        raise NotImplementedError

    def make_batch(self, B, seed):
        raise NotImplementedError

    def loss(self, model, batch):
        raise NotImplementedError

    def hot(self, model, batch):
        """The tensors model.hot_path hands to the torch tower (the librank_b200 part of forward)."""
        raise NotImplementedError


class DeepFMWorkload(Workload):
    name, batch, bytes_per_sample, flops_per_sample = "deepfm_d16", 1024, 2896, 600
    hot_calls = ("rk_deepfm_fwd", "rk_plan_build", "rk_deepfm_bwd", "rk_embgrad_segment_reduce")

    def model(self, ns, oracle, vocab_dir):
        cls = ns.OracleDeepFM if oracle else ns.DeepFM
        return cls(vocab_dir, embedding_dim=16, dropout_rate=0.0)

    def make_batch(self, B, seed):
        from rank_b200 import synthetic
        return synthetic.deepfm_batch(B, seed)

    def loss(self, model, batch):
        prob = model(batch["category"])[0]
        return F.binary_cross_entropy(prob.squeeze(), batch["label"])

    def hot(self, model, batch):
        return model.hot_path(batch["category"])


class FwFMWorkload(Workload):
    # FwFM/fwfm.py defaults: batch 1024, embedding_dim 8, six fields.  Algorithmic bytes per sample:
    # fwd 48 idx + 192 rows + 24 first-order + 192 emb + 4 y = 460; bwd 48 idx + 192 emb + 8 (y, g_y)
    # + 3 x (192 + 24) gradient rows (written per occurrence, read sorted, written unique) = 896.
    name, batch, bytes_per_sample, flops_per_sample = "fwfm_d8", 1024, 1356, 1000
    hot_calls = ("rk_fwfm_fwd", "rk_plan_build", "rk_fwfm_bwd", "rk_embgrad_segment_reduce")

    def model(self, ns, oracle, vocab_dir):
        from rank_b200 import synthetic
        cls = ns.OracleFwFM if oracle else ns.FwFM
        return cls(synthetic.fwfm_field_dims(), 8)

    def make_batch(self, B, seed):
        from rank_b200 import synthetic
        return synthetic.fwfm_batch(B, seed)

    def loss(self, model, batch):
        return F.binary_cross_entropy(model(batch["x"]), batch["label"])

    def hot(self, model, batch):
        return model.hot_path(batch["x"])


class DCNWorkload(Workload):
    name, batch, bytes_per_sample, flops_per_sample = "dcn_l3_dnn512-256-128", 8192, 1704, 2300
    hot_calls = ("rk_crossnet_fwd", "rk_plan_build", "rk_crossnet_bwd", "rk_embgrad_segment_reduce")

    def model(self, ns, oracle, vocab_dir):
        cls = ns.OracleDCN if oracle else ns.DCNModel
        return cls(vocab_dir, hidden_units=[512, 256, 128], num_cross_layer=3)

    def make_batch(self, B, seed):
        from rank_b200 import synthetic
        return synthetic.side_batch(B, seed)

    def loss(self, model, batch):
        logit = model(batch["dense"], batch["category"])[1]
        return F.binary_cross_entropy_with_logits(logit.squeeze(), batch["label"])

    def hot(self, model, batch):
        return model.hot_path(batch["dense"], batch["category"])


class AFMWorkload(Workload):
    # 10 fields, D=32, A=128.  Default module setting: attention MLP on tcgen05 (split-bf16 operands,
    # fp32 TMEM accumulation, ReLU decisions re-checked in fp32), inside the 1e-5 parity bar.
    name, batch, bytes_per_sample, flops_per_sample = "afm_f10_d32_a128", 8192, 6816, 1_150_000
    hot_calls = ("rk_afm_tc_fwd", "rk_plan_build", "rk_afm_tc_bwd", "rk_embgrad_segment_reduce")
    dtype = "bf16x3 tensor-core attention MLP (fp32 accumulate), f32 elsewhere"
    precision = "tensor"

    def __init__(self):
        from rank_b200 import synthetic
        self.fc = synthetic.afm_feature_columns(10)

    def model(self, ns, oracle, vocab_dir):
        cls = ns.OracleAFM if oracle else ns.AFM
        m = cls(self.fc, 32, 128)
        if not oracle:
            m.attention_precision = self.precision
        return m

    def make_batch(self, B, seed):
        from rank_b200 import synthetic
        return synthetic.afm_batch(B, self.fc, seed)

    def loss(self, model, batch):
        prob = model(batch["dense"], batch["category"])[0]
        return F.binary_cross_entropy(prob.squeeze(), batch["label"])

    def hot(self, model, batch):
        return model.hot_path(batch["dense"], batch["category"])


class AFMFp32Workload(AFMWorkload):
    # the fp32 SIMT kernels (csrc/afm.cu): compute-bound on the fp32 FMA pipe (SURVEY.md §8d)
    name, dtype, precision = "afm_f10_d32_a128_fp32simt", "f32", "fp32"
    hot_calls = ("rk_afm_fwd", "rk_plan_build", "rk_afm_bwd", "rk_embgrad_segment_reduce")


class DINWorkload(Workload):
    name, batch, bytes_per_sample, flops_per_sample = "din_t50_raw", 8192, 18648, 1_240_000
    hot_calls = ("rk_din_fwd", "rk_plan_build", "rk_din_bwd", "rk_embgrad_segment_reduce")
    use_softmax = False

    precision = "fp32"

    def model(self, ns, oracle, vocab_dir):
        cls = ns.OracleDIN if oracle else ns.DIN
        m = cls(vocab_dir, dropout_rate=0.0, use_softmax=self.use_softmax, l2_lambda=0.2)
        if not oracle:
            m.activation_unit_precision = self.precision
        return m

    def make_batch(self, B, seed):
        from rank_b200 import synthetic
        return synthetic.din_batch(B, 50, seed)

    def loss(self, model, batch):
        prob, _, l2 = model(batch["dense"], batch["category"], batch["sequence"], batch["target"])
        return F.binary_cross_entropy(prob.squeeze(), batch["label"]) + l2

    def hot(self, model, batch):
        return model.hot_path(batch["dense"], batch["category"], batch["sequence"], batch["target"])


class DINSoftmaxWorkload(DINWorkload):
    name, use_softmax = "din_t50_softmax", True


class DINTensorCoreWorkload(DINWorkload):
    # activation-unit MLP on tcgen05 (split-bf16 operands, fp32 TMEM accumulation)
    name, precision, dtype = "din_t50_raw_tcgen05", "bf16", "bf16x3 tensor-core MLP, f32 elsewhere"


class DINSoftmaxTensorCoreWorkload(DINSoftmaxWorkload):
    name, precision, dtype = "din_t50_softmax_tcgen05", "bf16", "bf16x3 tensor-core MLP, f32 elsewhere"


class BSTWorkload(Workload):
    name, batch, bytes_per_sample, flops_per_sample = "bst_t20_h4_b1", 8192, 7968, 261_000
    hot_calls = ("rk_gather_concat_fwd", "rk_bst_block_fwd", "rk_plan_build", "rk_bst_block_bwd",
                 "rk_embgrad_segment_reduce")

    precision = "fp32"

    def model(self, ns, oracle, vocab_dir):
        cls = ns.OracleBST if oracle else ns.BSTModel
        m = cls(vocab_dir, dropout_rate=0.0, nhead=4, num_transformer_blocks=1, max_seq_length=20)
        if not oracle:
            m.block_precision = self.precision
        return m

    def make_batch(self, B, seed):
        from rank_b200 import synthetic
        return synthetic.bst_batch(B, 20, seed)

    def loss(self, model, batch):
        logit = model(batch["dense"], batch["category"], batch["seq_feedid"], batch["seq_length"])[1]
        return F.binary_cross_entropy_with_logits(logit.squeeze(), batch["label"])

    def hot(self, model, batch):
        return model.hot_path(batch["dense"], batch["category"], batch["seq_feedid"], batch["seq_length"])


class BSTTensorCoreWorkload(BSTWorkload):
    # Q/K/V, output projection and FFN of the block on tcgen05 (split-bf16 operands, fp32 TMEM accumulation)
    name, precision, dtype = "bst_t20_h4_b1_tcgen05", "bf16", "bf16x3 tensor-core projections/FFN, f32 elsewhere"


class DeepCrossingWorkload(Workload):
    name, batch, bytes_per_sample, flops_per_sample = "deepcrossing_h128_n2", 8192, 1304, 154_000
    bound = "hbm"
    hot_calls = ("rk_resunits_fwd", "rk_plan_build", "rk_resunits_bwd", "rk_embgrad_segment_reduce")

    def model(self, ns, oracle, vocab_dir):
        cls = ns.OracleDeepCrossing if oracle else ns.DeepCrossingModel
        return cls(vocab_dir, residual_internal_dim=128, residual_network_num=2)

    def make_batch(self, B, seed):
        from rank_b200 import synthetic
        return synthetic.side_batch(B, seed)

    def loss(self, model, batch):
        logit = model(batch["dense"], batch["category"])[1]
        return F.binary_cross_entropy_with_logits(logit.squeeze(), batch["label"])

    def hot(self, model, batch):
        return model.hot_path(batch["dense"], batch["category"])


# BASELINE.json configs[3]: DIN, history 50, local activation unit as a tensor-core MLP, batch 8192 — the
# configuration the north star sets its roofline and 1->8 scaling targets on
DEFAULT_WORKLOAD = "din_tc"
WORKLOADS = {"deepfm": DeepFMWorkload, "fwfm": FwFMWorkload, "dcn": DCNWorkload, "afm": AFMWorkload, "afm_fp32": AFMFp32Workload, "din": DINWorkload,
             "din_softmax": DINSoftmaxWorkload, "din_tc": DINTensorCoreWorkload,
             "din_softmax_tc": DINSoftmaxTensorCoreWorkload, "bst": BSTWorkload, "bst_tc": BSTTensorCoreWorkload,
             "deepcrossing": DeepCrossingWorkload}


# ------------------------------------------------------------------------------- helpers
# fused forward + backward kernels whose ncu dram__bytes (profiles/r0N_traffic.json, one
# `ncu --set full` capture per kernel) are reported as roofline.traffic
TRAFFIC_KERNELS = {
    "din_softmax_tc": ("din_fwd_tc_kernel", "din_bwd_tc_kernel"),
    "dcn": ("crossnet_fwd_kernel", "crossnet_bwd_kernel"), "afm_fp32": ("afm_fwd_kernel", "afm_bwd_kernel"),
    "bst": ("bst_fwd_kernel", "bst_bwd_kernel"), "din_tc": ("din_fwd_tc_kernel", "din_bwd_tc_kernel"),
    "afm": ("afm_fwd_tc_kernel", "afm_bwd_tc_kernel"), "fwfm": ("fwfm_fwd_kernel", "fwfm_bwd_kernel"),
    "bst_tc": ("bst_fwd_tc_kernel", "bst_bwd_tc_kernel"),
}


def measured_traffic(workload_key):
    """DRAM bytes per launch (read + write) of the workload's fused fwd+bwd kernels, from the
    committed ncu capture of this round; None when no capture exists for them."""
    names = TRAFFIC_KERNELS.get(workload_key)
    table = {}
    for rnd in ("r01", "r02"):             # later rounds' captures override earlier ones, kernel by kernel
        path = os.path.join(ROOT, "profiles", f"{rnd}_traffic.json")
        if os.path.exists(path):
            with open(path) as f:
                table.update(json.load(f))
    if not names or not table:
        return None, None
    if not all(n in table for n in names):
        return None, None
    per = {n: table[n]["dram_read_bytes"] + table[n]["dram_write_bytes"] for n in names}
    return sum(per.values()), per


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], bf16_tflops=p["bf16_tflops_sustained"], source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms while the timed region runs."""
    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines, self.marks = index, None, [], []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.QUERY}",
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
            t_end = time.time() + 3.0          # let nvidia-smi finish starting up before any timing
            while not self.lines and time.time() < t_end and self.proc.poll() is None:
                time.sleep(0.01)
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.06)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        return False

    def mark(self):
        """Call at the start and at the end of the timed region."""
        self.marks.append(time.time())

    def absorb(self, other):
        """Add the in-region samples of a second sampler (another timed region of the same run)."""
        if len(other.marks) >= 2:
            t0, t1 = other.marks[0], other.marks[-1]
            extra = [(ts, l) for ts, l in other.lines if t0 - 0.06 <= ts <= t1 + 0.06]
            self.extra = getattr(self, "extra", []) + [l for _, l in extra]

    def summary(self):
        """Clocks / throttle reasons of the samples taken during the timed region (the sampler
        itself is started before the warm-up so that its start-up does not disturb the region;
        a region shorter than the sampling period takes the samples nearest to it)."""
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lines = self.lines
        if len(self.marks) >= 2 and lines:
            t0, t1 = self.marks[0], self.marks[-1]
            inside = [l for ts, l in lines if t0 - 0.06 <= ts <= t1 + 0.06]
            if not inside:
                nearest = sorted(lines, key=lambda x: min(abs(x[0] - t0), abs(x[0] - t1)))[:3]
                inside = [l for _, l in nearest]
            lines = inside
        else:
            lines = [l for _, l in lines]
        lines = list(lines) + getattr(self, "extra", [])
        for line in lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "reasons": sorted(reasons),
                "samples": len(sm)}


def dist_setup(n_gpus):
    # stdout carries exactly one JSON line: whatever NCCL logs (its version banner at
    # NCCL_DEBUG=VERSION, the transport lines at INFO) goes to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return world, rank, local


def capture_outputs(model):
    """{"outputs": the tensors of the latest forward of `model`}.  Under a CUDA graph that is the captured
    forward, whose outputs every replay rewrites in place.  Detached views: they keep no autograd graph alive."""
    seen = {}

    def hook(module, inputs, out):
        seen["outputs"] = [o.detach() for o in ([out] if torch.is_tensor(out) else out) if torch.is_tensor(o)]

    model.register_forward_hook(hook)
    return seen


def dump_outputs(out_dir, loss, outputs, model):
    """What one training step hands its caller, one file per array: DIR/loss.npy, DIR/output_<i>.npy (the
    forward's tensors) and DIR/grad.<parameter name>.npy, in float32 (float64 stays float64).  When they
    exceed DUMP_BYTES in all, every array of more than one row keeps the same share of its rows, chosen by
    a generator seeded with 0 and kept in ascending order, so two runs still compare row for row."""
    import numpy as np
    arrays = {"loss": loss}
    arrays.update({f"output_{i}": o for i, o in enumerate(outputs)})
    arrays.update({f"grad.{k}": p.grad for k, p in model.named_parameters() if p.grad is not None})
    arrays = {k: v.detach().to(torch.float64 if v.dtype == torch.float64 else torch.float32).cpu().numpy()
              for k, v in arrays.items()}
    rows = {k for k, a in arrays.items() if a.ndim and a.shape[0] > 1}
    whole = sum(a.nbytes for k, a in arrays.items() if k not in rows)
    share = min(1.0, (DUMP_BYTES - whole) / max(sum(arrays[k].nbytes for k in rows), 1))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if share < 1.0 and name in rows:
            keep = int(a.shape[0] * share)
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def cpu_reference_run(wl, steps, warmup, batch_size, budget_s=None, dump_dir=None):
    """The oracle port of the reference model on the host cores: fwd + loss + bwd per step."""
    from oracle import models as oracle_models
    import rank_b200
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    vocab = rank_b200.write_vocab_dir(tempfile.mkdtemp(prefix="rk_vocab_")) + "/"
    torch.manual_seed(0)
    model = wl.model(oracle_models, True, vocab)
    model.train()
    seen = capture_outputs(model) if dump_dir else None
    batches = [wl.make_batch(batch_size, 100 + i) for i in range(2)]
    times = []
    t_begin = time.perf_counter()
    for i in range(warmup + steps):
        b = batches[i % len(batches)]
        t0 = time.perf_counter()
        model.zero_grad(set_to_none=True)
        torch.manual_seed(i)
        loss = wl.loss(model, b)
        loss.backward()
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
        if budget_s is not None and i >= warmup + 2 and time.perf_counter() - t_begin > budget_s:
            break
    if seen is not None:
        dump_outputs(dump_dir, loss, seen["outputs"], model)
    ms = 1e3 * sum(times) / len(times)
    return dict(value=batch_size / (ms / 1e3), ms_per_step=ms, steps=len(times), cores=threads,
                loss=float(loss.detach()))


# ------------------------------------------------------------------------------- reference arm
def run_reference(args, wl):
    world, rank, _ = dist_setup(args.gpus)
    if rank != 0:
        return
    B = args.batch or wl.batch
    r = cpu_reference_run(wl, args.steps, args.warmup, B, dump_dir=args.dump_outputs)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": "samples/s",
        "n_gpus": args.gpus, "steps": r["steps"], "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": wl.name, "batch_per_step": B, "dropout": 0.0,
                   "what": "oracle port of the reference nn.Module (the reference is Python and cannot "
                           "travel to the GPU box), torch CPU fp32, all host threads"},
        "cpu_baseline": {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "kind": "port",
                         "sample": f"{r['steps']} full steps of batch {B} (fwd+loss+bwd), host CPU"},
        "e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# ------------------------------------------------------------------------------- our arm
class Stepper:
    """One training step (zero_grad, forward, loss, backward) on static device buffers, replayed
    from a CUDA graph (default) or run eagerly (--no-graph).  The per-call random weights of
    DCN / DeepCrossing / DIN are re-drawn on the CPU generator before every step, as the
    reference does inside forward, and shipped to a fixed device buffer outside the graph.
    `hot_only`: the graph holds only model.hot_path forward + its backward against fixed cotangents
    (no tower, no loss): the hot path of a step and nothing else."""

    def __init__(self, model, wl, example, use_graph, reducer, hot_only=False):
        self.model, self.wl, self.reducer, self.hot_only = model, wl, reducer, hot_only
        from rank_b200.staging import PackedBatch
        self.packed = PackedBatch.like(example.host_views, example.device)   # fixed addresses: graph inputs
        self.static = self.packed.device_views
        self.packed.dev.copy_(example.dev)            # the warm-up steps below run on a real batch
        self.has_ephemeral = hasattr(model, "draw_ephemeral")
        self.graph = None
        self.grads = None
        self.cots = None
        if use_graph:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for i in range(3):
                    self._eager(i)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            model.zero_grad(set_to_none=True)
            if self.has_ephemeral:
                model.draw_ephemeral()
                model.ephemeral_frozen = True
            try:
                self.graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.graph):
                    self._body()
            except Exception:
                # the symmetric-memory all-reduce could not be captured on this build: NCCL's can
                if self.reducer is None or self.reducer.symmetric is None:
                    raise
                self.reducer.use_nccl()
                torch.cuda.synchronize()
                model.zero_grad(set_to_none=True)
                self.graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.graph):
                    self._body()
            self.grads = [p.grad for p in model.parameters()]
        self.collective_in_graph = self.graph is not None and self.reducer is not None

    def _body(self):
        if self.hot_only:
            outs = [o for o in self.wl.hot(self.model, self.static) if o.requires_grad]
            if self.cots is None:
                gen = torch.Generator(device=outs[0].device).manual_seed(7)
                self.cots = [torch.randn(o.shape, generator=gen, device=o.device) / o.shape[0] for o in outs]
            self.loss = outs[0]
            torch.autograd.backward(outs, self.cots)
        else:
            self.loss = self.wl.loss(self.model, self.static)
            self.loss.backward()
            if self.reducer is not None:
                # the gradient all-reduce is part of the step: stream-ordered behind the backward, captured in
                # the same CUDA graph (no host work between the last kernel and the collective)
                self.reducer.allreduce()

    def _eager(self, seed):
        self.model.zero_grad(set_to_none=True)
        torch.default_generator.manual_seed(seed)
        self._body()

    def load(self, packed, from_host=False):
        """ONE copy of the whole packed batch into the static inputs: pinned host -> device when
        `from_host`, device -> device otherwise."""
        self.packed.dev.copy_(packed.host if from_host else packed.dev, non_blocking=True)

    def run(self, seed, before_replay=None):
        """`before_replay()` is called after the step's own uploads (the per-call weights) have been queued and
        before the step's kernels are."""
        if self.graph is None:
            if before_replay is not None:
                before_replay()
            self._eager(seed)
        else:
            if self.has_ephemeral and not self.hot_only:
                torch.default_generator.manual_seed(seed)   # same draw on every rank
                self.model.draw_ephemeral()
            if before_replay is not None:
                before_replay()
            self.graph.replay()
        return self.loss


def aten_cuda_run(wl, B, steps, warmup, dev, flush, vocab):
    """The oracle port of the reference model on THIS GPU through stock ATen/cuBLAS kernels — what the
    reference does when its scripts run with --device cuda (e.g. DCN/dcn.py:161-180, DIN/din.py:294-323):
    zero_grad + forward + loss + backward per step, eager (per-call weights drawn on the CPU and moved to
    the device inside forward, as the reference does) and replayed from a CUDA graph (per-call weights
    frozen to one draw: a graph cannot hold the CPU draws; everything else identical).  L2 is flushed
    between steps as for our arm."""
    from oracle import models as oracle_models
    from rank_b200 import synthetic
    torch.manual_seed(0)
    model = wl.model(oracle_models, True, vocab).to(dev)
    model.train()
    pool = [synthetic.to_device(wl.make_batch(B, 1000 + i), dev) for i in range(4)]

    def step(batch, seed):
        model.zero_grad(set_to_none=True)
        torch.manual_seed(seed)
        loss = wl.loss(model, batch)
        loss.backward()
        return loss

    def timed(fn, n):
        evs = []
        for i in range(n):
            flush.fill_(i & 0xff)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn(i)
            e.record()
            evs.append((s, e))
        torch.cuda.synchronize()
        return sum(s.elapsed_time(e) for s, e in evs) / n

    for i in range(warmup):
        step(pool[i % 4], i)
    torch.cuda.synchronize()
    eager_ms = timed(lambda i: step(pool[i % 4], 100 + i), steps)
    out = {"eager_ms_per_step": eager_ms, "eager_value": B / (eager_ms * 1e-3), "unit": "samples/s",
           "what": "oracle port of the reference nn.Module on cuda: stock ATen/cuBLAS kernels, fwd+loss+bwd, "
                   "same batch, dropout 0; eager = per-call weights drawn on the CPU and copied inside forward "
                   "(as the reference), graph = the same step captured with one frozen draw",
           "steps": steps}
    try:
        if hasattr(model, "last_ephemeral"):
            model.frozen_ephemeral = model.last_ephemeral
        static = synthetic.to_device(wl.make_batch(B, 999), dev)

        def copy_in(dst, src):
            if torch.is_tensor(dst):
                dst.copy_(src)
            else:
                for k in dst:
                    copy_in(dst[k], src[k])

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for i in range(3):
                step(static, i)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        model.zero_grad(set_to_none=True)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            loss = wl.loss(model, static)
            loss.backward()

        def replay(i):
            graph.replay()

        for i in range(3):
            copy_in(static, pool[i % 4])
            graph.replay()
        torch.cuda.synchronize()
        evs = []
        for i in range(steps):
            copy_in(static, pool[i % 4])
            flush.fill_(i & 0xff)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            graph.replay()
            e.record()
            evs.append((s, e))
        torch.cuda.synchronize()
        graph_ms = sum(s.elapsed_time(e) for s, e in evs) / steps
        out.update(graph_ms_per_step=graph_ms, graph_value=B / (graph_ms * 1e-3))
        del graph
    except Exception as exc:       # a capture failure of the stock path is a result, not a bench failure
        msg = f"{type(exc).__name__}: {exc}"
        if "capture" in msg.lower():
            # what happens on every model with an nn.Embedding: ATen's embedding_dense_backward copies a device-side
            # segment count to the host to size its buffers, and a host sync invalidates a stream capture
            msg = ("the stock path cannot be captured: ATen's embedding_dense_backward synchronises with the host "
                   "(cudaErrorStreamCaptureInvalidated); the eager figure is the reference-on-CUDA bar")
        out["graph_error"] = msg[:300]
        torch.cuda.synchronize()
    del model
    return out


def measure_ours(args, wl, key, world, rank, local, dev, primary):
    """Everything measured for one workload.  `primary`: the workload of the JSON line (all legs);
    otherwise a shorter run for the `other_workloads` summaries."""
    import rank_b200
    from rank_b200 import _lib, sparse
    from rank_b200.parallel import GradientAllReducer
    from rank_b200.staging import PackedBatch, Prefetcher

    lib = _lib.load()
    B = args.batch or wl.batch
    steps = args.steps if primary else min(args.steps, 50)
    vocab = rank_b200.write_vocab_dir(tempfile.mkdtemp(prefix="rk_vocab_")) + "/"
    torch.manual_seed(0)                    # identical replicas on every rank
    model = wl.model(rank_b200, False, vocab).to(dev)
    model.train()
    seen = capture_outputs(model) if primary and args.dump_outputs else None
    reducer = GradientAllReducer(model) if world > 1 else None

    n_pool = 4
    # every batch of the pool is collated once into a packed pinned buffer (rank_b200.staging) and
    # also kept on the device: `value` steps copy device -> device (untimed), `e2e` steps do the one
    # host -> device copy inside the timed region
    raw = [wl.make_batch(B, 1000 + 17 * rank + i) for i in range(n_pool)]
    pool = [PackedBatch.like(b, dev).fill(b) for b in raw]
    for pb in pool:
        pb.to_device()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(8):
        pool[i % n_pool].fill(raw[i % n_pool])
    fill_ms = (time.perf_counter() - t0) / 8 * 1e3      # host-side collate into the pinned buffer
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    stepper = Stepper(model, wl, pool[0], not args.no_graph, reducer)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    host_loop = [0.0]

    def timed(st, n_steps, first_seed, from_host):
        evs = []
        loss = None
        host_t0 = time.perf_counter()
        pf = Prefetcher(st.packed) if from_host else None
        # the step's result is read back into PINNED memory: a pageable destination would turn the D2H copy into a
        # host synchronisation and expose the host's per-step work (weight draws, graph launch) on the GPU timeline
        loss_host = torch.empty(max(n_steps, 1), dtype=torch.float32, pin_memory=True) if from_host else None
        slot = None
        for i in range(n_steps):
            flush.fill_(i & 0xff)           # evict L2 between steps; outside the timed events
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            if from_host:
                # Input pipeline with prefetch (rank_b200.staging.Prefetcher): every step's inputs cross PCIe in
                # ONE H2D copy of the packed pinned batch, issued on a copy stream; the copy of step i+1 starts
                # after this step's start event and must have finished before its end event, so each of the K
                # copies lies entirely inside a timed bracket, overlapped with the step's kernels.
                s.record()
                start = torch.cuda.Event()
                start.record()
                if slot is None:
                    slot = pf.submit(pool[i % n_pool], after=start)          # the first step waits for its own copy
                pf.consume(slot)                                             # D2D into the graph's static inputs
                nxt_slot = [None]

                def prefetch_next(i=i):
                    # the next batch's copy may start once this step's own small upload (the per-call weights) has
                    # run: the host-to-device copy engine serves whichever copy is ready first, and a 4 MB prefetch
                    # in front of that upload delays the whole step by ~100 us
                    if i + 1 < n_steps:
                        uploaded = torch.cuda.Event()
                        uploaded.record()
                        nxt_slot[0] = pf.submit(pool[(i + 1) % n_pool], after=uploaded)
                loss = st.run(first_seed + i, before_replay=prefetch_next)
                nxt = nxt_slot[0]
                loss_host[i:i + 1].copy_(loss.detach().reshape(1), non_blocking=True)      # D2H read of the step's result
                if nxt is not None:
                    pf.wait(nxt)
                e.record()
                slot = nxt
            else:
                st.load(pool[i % n_pool])                       # device-to-device, untimed
                s.record()
                loss = st.run(first_seed + i)
                e.record()
            evs.append((s, e))
        host_loop[0] = (time.perf_counter() - host_t0) / max(n_steps, 1) * 1e3     # host time to queue one step
        torch.cuda.synchronize()
        return sum(s.elapsed_time(e) for s, e in evs), float(loss.detach().reshape(-1)[0])

    with ClockSampler(local) as clocks:      # started before the warm-up, sampled through the timed region
        for i in range(args.warmup):
            stepper.load(pool[i % n_pool])
            stepper.run(i)
        if world > 1:
            # NCCL builds its channels lazily over the first collectives: settle them (and the host
            # threads of all ranks) before the timed region, beyond the W model steps above
            for i in range(10):
                stepper.load(pool[i % n_pool])
                stepper.run(100 + i)
                barrier()
        barrier()
        clocks.mark()
        total_ms, last_loss = timed(stepper, steps, 10_000, from_host=False)
        host_value_ms = host_loop[0]
        barrier()
        clocks.mark()
    if seen is not None and rank == 0:           # before the legs below reuse the step's buffers
        dump_outputs(args.dump_outputs, stepper.loss, seen["outputs"], model)
    launches = stepper_launches_per_replay(stepper, lib) * steps if stepper.graph is not None else None
    # end to end: pinned host inputs -> H2D -> step -> D2H loss
    for i in range(3):
        timed(stepper, 1, 50 + i, from_host=True)
    barrier()
    with ClockSampler(local) as clocks_e2e:      # the end-to-end region is a timed region too: sample it as well
        barrier()                                # (the samplers start at different speeds on different ranks)
        clocks_e2e.mark()
        e2e_ms, _ = timed(stepper, steps, 20_000, from_host=True)
        host_e2e_ms = host_loop[0]
        barrier()
        clocks_e2e.mark()
    clocks.absorb(clocks_e2e)

    t = torch.tensor([total_ms, e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    total_ms, e2e_ms = float(t[0]), float(t[1])
    ms_per_step = total_ms / steps

    # ---- the hot path alone: a CUDA graph of model.hot_path forward + backward (incl. the embedding-
    # gradient reduction) against fixed cotangents; same static inputs, same L2 flush between replays
    # (--no-graph, the profiling mode: the hot path runs eagerly too — a capture after eager steps on the legacy
    # stream is refused by CUDA, and ncu wants plain launches anyway)
    hot = Stepper(model, wl, pool[0], not args.no_graph, None, hot_only=True)
    for i in range(3):
        hot.load(pool[i % n_pool])
        hot.run(i)
    hot_total, _ = timed(hot, steps, 0, from_host=False)
    hot_ms = hot_total / steps
    hot_launches = stepper_launches_per_replay(hot, lib)
    evs = []
    for i in range(steps):                    # the same graph without the flush: tables / code still in L2
        hot.load(pool[i % n_pool])
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        hot.run(i)
        e.record()
        evs.append((s, e))
    torch.cuda.synchronize()
    hot_warm_ms = sum(s.elapsed_time(e) for s, e in evs) / steps
    del hot

    # ---- per-call diagnostic: eager steps queued behind a spin kernel, CUDA events around each ABI call.
    # Every bracket also holds the launch gaps around its kernels (~3-6 us per call on this box), so these
    # are upper bounds used for the SHARES of the calls, not for the roofline.
    calls = {}
    if primary or args.calls:
        eager = Stepper(model, wl, pool[0], False, None)
        if hasattr(model, "ephemeral_frozen"):
            model.ephemeral_frozen = False
        side_was = sparse.PLAN_ON_SIDE_STREAM
        sparse.PLAN_ON_SIDE_STREAM = False      # time the occurrence plan in-stream, not overlapped
        n_diag = min(steps, 20)
        with _lib.CallTimer() as ct:
            for i in range(n_diag):
                eager.load(pool[i % n_pool])
                flush.fill_(i & 0xff)
                _lib.check(lib.rk_debug_spin(4000, _lib.stream_ptr()), "rk_debug_spin")
                eager.run(30_000 + i)
                torch.cuda.synchronize()
        sparse.PLAN_ON_SIDE_STREAM = side_was
        calls = {k: {"calls_per_step": n / n_diag, "ms_per_step": ms / n_diag} for k, (n, ms) in sorted(ct.summary().items())}

    pk = peaks()
    achieved = (B * wl.bytes_per_sample) / (hot_ms * 1e-3) / 1e9 if hot_ms > 0 else 0.0
    res = {
        "workload": wl.name, "batch_per_gpu": B, "steps": steps, "value": world * B * steps / (total_ms / 1e3),
        "ms_per_step": ms_per_step, "e2e_value": world * B * steps / (e2e_ms / 1e3), "loss": last_loss,
        "dtype": wl.dtype, "clocks": clocks.summary(),
        "gpu_launches": int(launches) if launches is not None else None,
        "h2d_bytes": pool[0].nbytes, "h2d_payload": pool[0].payload_bytes, "fill_ms": fill_ms,
        "host_queue_ms": {"value_loop": host_value_ms, "e2e_loop": host_e2e_ms},
        "graph": stepper.graph is not None,
        "allreduce": None if reducer is None else ("nccl" if reducer.symmetric is None else "symmetric memory: " + reducer.symmetric[0]),
        "roofline": {
            "bound": wl.bound, "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s",
            "frac": achieved / pk["hbm_gbs"], "peak_source": pk["source"],
            "what": "hot path = CUDA graph of model.hot_path forward + backward incl. the embedding-gradient "
                    "reduction (" + ", ".join(wl.hot_calls) + "), replayed with the L2 flushed before each replay",
            "algorithmic_bytes_per_sample": wl.bytes_per_sample, "hot_ms_per_step": hot_ms,
            "hot_ms_per_step_warm_l2": hot_warm_ms, "hot_launches_per_step": int(hot_launches),
            "hot_share_of_step": hot_ms / ms_per_step if ms_per_step > 0 else None,
            "hot_le_step": bool(hot_ms <= ms_per_step),
            "frac_warm_l2": (B * wl.bytes_per_sample) / (hot_warm_ms * 1e-3) / 1e9 / pk["hbm_gbs"] if hot_warm_ms > 0 else None,
        },
        "hotpath_calls_eager_events": calls,
    }
    if wl.flops_per_sample >= 100_000:       # the dense part: share of the tensor / FMA roof as well
        res["roofline"]["flops_per_sample"] = wl.flops_per_sample
        res["roofline"]["achieved_tflops"] = B * wl.flops_per_sample / (hot_ms * 1e-3) / 1e12
    traffic, traffic_by = measured_traffic(key)
    res["roofline"]["traffic"] = traffic
    res["roofline"]["traffic_by_kernel"] = traffic_by
    if traffic is not None:
        res["roofline"]["traffic_note"] = ("ncu dram__bytes_read+write of the fused fwd+bwd kernels (one --set full "
                                           "capture, cold cache); below the algorithmic bytes where tables and "
                                           "outputs live in the 126 MB L2")
    if world == 1 and rank == 0 and not args.no_aten:
        del stepper
        model.zero_grad(set_to_none=True)
        res["aten_cuda_baseline"] = aten_cuda_run(wl, B, min(steps, 50), 3, dev, flush, vocab)
        a = res["aten_cuda_baseline"]
        a["ours_over_aten_eager"] = a["eager_ms_per_step"] / ms_per_step
        if "graph_ms_per_step" in a:
            a["ours_over_aten_graph"] = a["graph_ms_per_step"] / ms_per_step
    del model, pool, flush
    torch.cuda.empty_cache()
    return res


OTHERS = ("din_softmax_tc", "din", "dcn", "deepfm", "fwfm", "afm", "bst", "bst_tc", "deepcrossing")


def run_ours(args, wl):
    world, rank, local = dist_setup(args.gpus)
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    r = measure_ours(args, wl, args.workload, world, rank, local, dev, primary=True)
    if rank == 0:
        B, steps = r["batch_per_gpu"], r["steps"]
        line = {
            "metric": METRIC, "value": r["value"], "unit": "samples/s",
            "n_gpus": world, "steps": steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": r["dtype"],
            "data": "synthetic",
            "config": {"workload": r["workload"], "batch_per_gpu": B, "global_batch": world * B, "dropout": 0.0,
                       "parallelism": f"dp{world}", "l2": "256 MiB written between steps, outside the timed events",
                       "step": "zero_grad+fwd+loss+bwd" + ("+grad allreduce" if world > 1 else ""),
                       "allreduce": r.get("allreduce"),
                       "launch": "cuda graph replay per step" if r["graph"] else "eager",
                       "indices": "zipf(1.05), fresh batch each step from a pool of 4"},
            "clocks": r["clocks"],
            "e2e": {"value": r["e2e_value"], "unit": "samples/s",
                    "h2d_bytes_per_step": r["h2d_bytes"], "d2h_bytes_per_step": 4,
                    "h2d_copies_per_step": 1, "h2d_payload_bytes": r["h2d_payload"],
                    "note": "timed per step: ONE H2D copy of a packed pinned batch + one D2D into the graph's static "
                            "inputs + graph replay + D2H of the loss.  The input pipeline prefetches "
                            "(staging.Prefetcher): the H2D copy of step i+1 runs on a copy stream between the start "
                            "and end events of step i (the first step waits for its own copy), so all K copies lie "
                            "inside timed brackets.  Collating a dict batch into the pinned buffer "
                            "(PackedBatch.fill, host side) is outside the events",
                    "host_fill_ms_per_batch": r["fill_ms"],
                    # host time to QUEUE one step (weight draws, copies, graph launch): when it approaches the
                    # device time of a step the loop is host-bound and the brackets hold idle device time
                    "host_queue_ms_per_step": r["host_queue_ms"]},
            "gpu_launches": r["gpu_launches"],
            "roofline": r["roofline"],
            "hotpath_calls_eager_events": r["hotpath_calls_eager_events"],
            "loss": r["loss"],
        }
        if "aten_cuda_baseline" in r:
            line["aten_cuda_baseline"] = r["aten_cuda_baseline"]
        if world == 1 and not args.no_cpu_baseline:
            c = cpu_reference_run(wl, 50, 2, B, budget_s=15.0)
            line["cpu_baseline"] = {"value": c["value"], "unit": "samples/s", "cores": c["cores"], "kind": "port",
                                    "sample": f"{c['steps']} full steps of batch {B} (fwd+loss+bwd) of the oracle "
                                              "port, torch CPU fp32"}
    if world == 1 and args.workload == DEFAULT_WORKLOAD and not args.no_others and not args.batch:
        others = {}
        for k in OTHERS:
            if k == args.workload:
                continue
            try:
                o = measure_ours(args, WORKLOADS[k](), k, world, rank, local, dev, primary=False)
                a = o.get("aten_cuda_baseline", {})
                others[k] = {
                    "workload": o["workload"], "batch": o["batch_per_gpu"], "steps": o["steps"],
                    "value": o["value"], "ms_per_step": o["ms_per_step"], "e2e_value": o["e2e_value"],
                    "hot_ms_per_step": o["roofline"]["hot_ms_per_step"], "hot_share_of_step": o["roofline"]["hot_share_of_step"],
                    "roofline_frac": o["roofline"]["frac"], "hot_launches_per_step": o["roofline"]["hot_launches_per_step"],
                    "gpu_launches_per_step": (o["gpu_launches"] or 0) / o["steps"],
                    "aten_cuda_eager_ms": a.get("eager_ms_per_step"), "aten_cuda_graph_ms": a.get("graph_ms_per_step"),
                    "ours_over_aten_eager": a.get("ours_over_aten_eager"), "ours_over_aten_graph": a.get("ours_over_aten_graph"),
                    "sm_mhz": o["clocks"].get("sm_mhz"), "reasons": o["clocks"].get("reasons"),
                }
            except Exception as exc:      # one workload failing must not lose the line
                others[k] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
                try:
                    torch.cuda.synchronize()
                except Exception:         # a sticky device error: nothing more can run in this process
                    break
        line["other_workloads"] = others
    if rank == 0:
        emit(line)
    if world > 1:
        torch.distributed.destroy_process_group()


def stepper_launches_per_replay(stepper, lib):
    """Kernels of librank_b200 inside one captured step = what one eager step launches."""
    probe = Stepper(stepper.model, stepper.wl, stepper.packed, False, None, hot_only=stepper.hot_only)
    probe.cots = stepper.cots
    probe.load(stepper.packed)
    frozen = getattr(stepper.model, "ephemeral_frozen", None)
    n0 = lib.rk_launch_count()
    probe.run(1)
    torch.cuda.synchronize()
    n = lib.rk_launch_count() - n0
    if frozen is not None:
        stepper.model.ephemeral_frozen = frozen
    stepper.model.zero_grad(set_to_none=True)
    if stepper.grads is not None:
        for p, g in zip(stepper.model.parameters(), stepper.grads):
            p.grad = g
    return n


_JSON_FD = None


def claim_stdout():
    """stdout carries exactly ONE line, the JSON result.  Libraries write there too (NCCL prints its
    version banner on stdout when the first communicator is created), so file descriptor 1 is pointed
    at stderr for the whole run and the result line goes to a private duplicate of the real stdout."""
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the workload's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-aten", action="store_true", help="skip the reference-on-CUDA (stock ATen) baseline")
    ap.add_argument("--no-others", action="store_true", help="skip the other workloads' one-line summaries")
    ap.add_argument("--calls", action="store_true", help="per-call event diagnostic for the other workloads too")
    ap.add_argument("--no-graph", action="store_true", help="launch every step eagerly instead of a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's loss, forward outputs and parameter "
                         "gradients to DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    claim_stdout()
    args.warmup = max(args.warmup, 3)
    wl = WORKLOADS[args.workload]()
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
