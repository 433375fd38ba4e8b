#!/usr/bin/env python
"""bench.py — CoPER-ConvE hot-path throughput on B200 (contract: see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--shape S] [--prec P] [--impl ours|reference]
                    [--dump-outputs DIR]

Every GPU workload block times exactly K steps after max(W, 3) warm-up steps (the first two calls of a step run eager and
capture its CUDA graph).

A "step" = one full training step of the hot path over one synthetic batch of B (e1, rel) queries with
1-N labels: lookups -> conv -> fused CPG-FC -> 1-N scorer + label-smoothed BCE -> backward -> global-norm
clip -> AMSGrad.  `value` = train rows/s with inputs resident in HBM; `eval` = filtered-rank queries/s
(forward + 1-N scores + filtered rank); `e2e` = the same through the public API from pinned HOST batches
with the loss / ranks read back every step.  One JSON line on stdout (rank 0).

Workloads (BASELINE.json configs):
  N = 1   headline = WN18RR shape (configs[1]), fp32-class fp16x3 engine (3-term compensated fp16 planes on tcgen05:
          same accuracy class and the same 1e-5 parity bar as tf32x3, which stays selectable with --prec); `configs`
          holds one block per other named shape (FB15k-237, NELL-995, YAGO3-10 in fp16x3; synth-10m in bf16) with
          value / e2e / eval / per-stage
          rooflines; `rooflines` has EVERY stage of the headline (tensor-bound stages against the measured bf16 peak,
          HBM-bound ones against the measured copy bandwidth); `hbm_kernels` times gather / segmented scatter /
          filtered rank at sizes where HBM bandwidth (not launch latency) is what is measured.
  N > 1   headline = synth-10m (10 M entities, d = 256), bf16, entity-sharded scorer, replicated front end, fixed
          B = 512 -> "scaling": "strong" (north_star's scaling target).  `strong_scaling_base` is the same workload
          on ONE GPU measured by rank 0 in the same run (the driver's own N = 1 run is the WN18RR headline, so the
          strong-scaling ratio is value / (N * strong_scaling_base.value)); `wn18rr_weak` keeps the data-parallel
          WN18RR weak-scaling numbers (global batch N * 512).
  --shape / --prec / --front-end select one workload explicitly (then no extra blocks are produced).
"""
from __future__ import annotations

import argparse
import copy
import gc
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
DTYPE_NAME = {"fp32": "f32", "bf16": "bf16", "tf32x3": "tf32x3", "fp16x3": "fp16x3"}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            d["_source"] = "measured (MEASURED_PEAKS.json)"
            return d
        except Exception:
            pass
    d = dict(FALLBACK_PEAKS)
    d["_source"] = "fallback (B200_PROFILING.md)"
    return d


def load_traffic():
    """DRAM bytes per stage from the committed ncu captures (profiles/r0N_traffic.json), newest round first."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            return json.load(open(os.path.join(ROOT, "profiles", name))), name
        except Exception:
            continue
    return {}, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu, self.proc, self.path = gpu_index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path).read().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.path)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def workload_name(shape, s, B):
    return "CoPER-ConvE %s shape (N=%d entities, R'=%d, d=%d, dr=%d, B=%d, full 1-N labels)" % (
        shape, s["num_ent"], s["num_rel"], s["ent_emb_size"], s["rel_emb_size"], B)


# ------------------------------------------------------------------------------------------ CPU legs (oracle port)
def oracle_cfg_of(md, H, num_ent=None):
    from oracle import conve_oracle as O
    return O.OracleConfig(num_ent=num_ent or md["num_ent"], num_rel=md["num_rel"], ent_emb_size=md["ent_emb_size"],
                          rel_emb_size=md["rel_emb_size"], context_rel_out=list(md["context_rel_out"]),
                          conv_in_height=H, hidden_dropout=0.0, output_dropout=0.0,
                          batch_norm_momentum=md["batch_norm_momentum"],
                          batch_norm_train_stats=md["batch_norm_train_stats"])


def _cpu_port(shape, num_ent=None, B=None):
    """TorchPort (oracle/torch_port.py) + one batch at `shape`, optionally against a SLICE of num_ent entity rows."""
    import torch
    from coper_b200 import synthetic
    from oracle import conve_oracle as O
    from oracle.torch_port import TorchPort
    s = synthetic.SHAPES[shape]
    N = num_ent or s["num_ent"]
    B = B or s["batch"]
    md = synthetic.descriptors(shape, dropout=False)
    cfg = oracle_cfg_of(md, s["H"], N)
    params = O.init_params(cfg, seed=0)
    hb = synthetic.make_batches(N, s["num_rel"], B, 1, seed=1)[0]
    dense = O.csr_to_dense(hb["e2_multi_rowptr"], hb["e2_multi_col"], N)
    torch.set_num_threads(os.cpu_count() or 1)
    return TorchPort(params, cfg, torch.float32), (hb["e1"], hb["rel"], hb["e2"], dense)


def _time_port(port, batch, steps, warmup, eval_batches):
    e1, rel, e2, labels = batch
    for _ in range(warmup):
        port.train_step(e1, rel, labels)
    t0 = time.perf_counter()
    for _ in range(steps):
        port.train_step(e1, rel, labels)
    train_s = (time.perf_counter() - t0) / max(steps, 1)
    eval_s = None
    if eval_batches:
        port.eval_batch(e1, rel, e2, labels)
        t0 = time.perf_counter()
        for _ in range(eval_batches):
            port.eval_batch(e1, rel, e2, labels)
        eval_s = (time.perf_counter() - t0) / eval_batches
    return train_s, eval_s


def run_cpu_baseline(shape, budget_s):
    """cpu_baseline leg of our own arm: the reference algorithm restated on torch-CPU (oracle/torch_port.py; TensorFlow
    1.14 is not installable here), all host cores, a bounded sample (~budget_s seconds) of the same workload."""
    from coper_b200 import synthetic
    from oracle.torch_port import time_cpu_baseline
    from oracle import conve_oracle as O
    s = synthetic.SHAPES[shape]
    md = synthetic.descriptors(shape, dropout=False)
    cfg = oracle_cfg_of(md, s["H"])
    params = O.init_params(cfg, seed=0)
    hb = synthetic.make_batches(s["num_ent"], s["num_rel"], s["batch"], 1, seed=1)[0]
    dense = O.csr_to_dense(hb["e2_multi_rowptr"], hb["e2_multi_col"], s["num_ent"])
    r = time_cpu_baseline(params, cfg, (hb["e1"], hb["rel"], hb["e2"], dense), budget_s=budget_s)
    return {"value": r["train_rows_per_s"], "unit": "train rows/s", "eval_value": r["eval_queries_per_s"],
            "eval_unit": "eval queries/s", "cores": r["cores"], "kind": "port",
            "sample": "%d train steps + %d eval batches of B=%d at the %s shape, torch-CPU fp32 materialising "
                      "restatement of models.py/metrics.py (TensorFlow unavailable offline)"
                      % (r["train_steps"], r["eval_batches"], s["batch"], shape),
            "train_ms": r["train_ms"], "eval_ms": r["eval_ms"]}


def reference_arm(args, shape, B, scaling, workload):
    """`--impl reference`: the reference's CPU implementation of the path (oracle port, kind "port") on all host cores,
    exactly W warm-up + K timed steps, on the configuration our own arm labels.  Shapes whose dense fp32 [B, N] labels
    and logits do not fit a bounded CPU step (synth-10m: 2 x 20 GB per step) are timed on an entity SLICE and
    extrapolated linearly in N (the scorer, loss, gradient and optimizer all stream N rows); the slice is stated.
    --steps sets the timed train steps only: the eval batches (2 to 8) and the small slice's train steps (K // 2, at
    least 2) are counts of their own, stated in `sample`."""
    from coper_b200 import synthetic
    s = synthetic.SHAPES[shape]
    N = s["num_ent"]
    K, W = args.steps, args.warmup
    slice_n = None
    if N > 400_000:
        slice_n = 1 << 18                                  # 262 144 rows: ~1 s per CPU step
    if slice_n is None:
        port, batch = _cpu_port(shape, B=B)
        train_s, eval_s = _time_port(port, batch, K, W, eval_batches=max(2, min(K, 8)))
        sample = "%d warm-up + %d timed train steps and %d eval batches of B=%d at the full %s shape" % (
            W, K, max(2, min(K, 8)), B, shape)
    else:
        # t(N) = t_front + c * N: two slices give both terms
        small_n = slice_n // 8
        port, batch = _cpu_port(shape, num_ent=slice_n, B=B)
        t_big, e_big = _time_port(port, batch, K, W, eval_batches=2)
        del port, batch
        gc.collect()
        port, batch = _cpu_port(shape, num_ent=small_n, B=B)
        t_small, e_small = _time_port(port, batch, max(2, K // 2), 1, eval_batches=2)
        c_t = max(t_big - t_small, 0.0) / (slice_n - small_n)
        c_e = max(e_big - e_small, 0.0) / (slice_n - small_n)
        train_s = t_small + c_t * (N - small_n)
        eval_s = e_small + c_e * (N - small_n)
        sample = ("bounded sample: %d warm-up + %d timed train steps of B=%d against an entity slice of %d rows (and %d "
                  "rows for the N-independent part), extrapolated linearly to N=%d (dense fp32 labels + logits of the "
                  "full shape are 2 x %.0f GB per step); measured %.3f s / %.3f s per step" % (
                      W, K, B, slice_n, small_n, N, B * N * 4 / 1e9, t_big, t_small))
    value, evalue = B / train_s, B / eval_s
    cores = os.cpu_count() or 1
    line = {"impl": "reference", "metric": "train_rows_per_s", "value": value, "unit": "train rows/s",
            "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": train_s * 1e3, "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "note": "CPU restatement of the reference path (oracle/torch_port.py), "
                                                     "torch-CPU fp32, %d threads" % cores},
            "eval": {"value": evalue, "unit": "eval queries/s", "ms_per_batch": eval_s * 1e3},
            "cpu_baseline": {"value": value, "unit": "train rows/s", "cores": cores, "kind": "port",
                             "sample": sample + "; torch-CPU fp32 materialising restatement of models.py / metrics.py "
                                                "(TensorFlow 1.14 unavailable offline)"},
            "e2e": {"value": value, "unit": "train rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                    "eval_value": evalue}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ GPU measurement
class Ctx:
    """torch / dist handles + timing helpers shared by every measured block."""

    def __init__(self, rank, world, local_rank):
        import torch
        import torch.distributed as dist
        from coper_b200 import _lib
        self.torch, self.dist = torch, dist
        self.rank, self.world, self.local_rank = rank, world, local_rank
        self.lib = _lib.load()

    def barrier(self, collective=True):
        if self.world > 1 and collective:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, model, fn, steps, warmup, collective=True):
        """W warm-up + K timed calls bracketed by barrier + synchronize, CUDA events, max over ranks."""
        torch = self.torch
        for i in range(warmup):
            fn(i)
        self.barrier(collective)
        k0 = self.lib.coper_launch_count() + model.graph_kernel_launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        self.barrier(collective)
        ms = e0.elapsed_time(e1)
        if self.world > 1 and collective:
            t = torch.tensor([ms], device="cuda")
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps, (self.lib.coper_launch_count() + model.graph_kernel_launches - k0)


def working_set_mb(s, B):
    N, d, dr = s["num_ent"], s["ent_emb_size"], s["rel_emb_size"]
    H = s["H"]
    F = (H - 2) * (d // H - 2) * 32
    return int((3 * N * d * 4 + 3 * dr * F * d * 4 + B * N * 4 + 4 * B * F * 4) / 1e6)


DUMP_MAX_ELEMS = 1 << 19       # per array: larger outputs are dumped as a fixed, seeded sample of this many elements


def host_output(t):
    """A device output as float32 (float64 stays float64; integers become exact float64), sampled if large."""
    import torch
    t = t.detach()
    if t.numel() > DUMP_MAX_ELEMS:
        idx = np.unique(np.random.default_rng(0).integers(0, t.numel(), DUMP_MAX_ELEMS))
        t = t.reshape(-1)[torch.as_tensor(idx, device=t.device)]
    a = t.cpu().numpy()
    return a.astype(np.float64 if a.dtype in (np.float64, np.int64, np.int32) else np.float32)


def write_outputs(out_dir, outputs):
    total = sum(a.nbytes for a in outputs.values())
    if total > 64 << 20:
        raise RuntimeError("--dump-outputs: %d bytes exceed the 64 MB cap" % total)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measure(ctx, shape, prec, K, W, peaks, *, sharded=False, dp=False, e2e=True, breakdown=True, graphs_multi=True,
            overlap=True, outputs=None):
    """One workload: device-resident train / eval throughput, end-to-end numbers and the per-stage rooflines.
    sharded=False builds a single-GPU model on this rank (no collectives) even inside a multi-rank job.
    outputs (a dict) receives, as host arrays, what the last timed train step and eval batch returned: the loss, the
    model state after the update (variables, optimizer slots, batch-norm statistics) and the filtered ranks."""
    torch = ctx.torch
    from coper_b200 import synthetic
    from coper_b200.models import ConvE, EntityShard
    s = synthetic.SHAPES[shape]
    world = ctx.world if sharded else 1
    rank = ctx.rank if sharded else 0
    dp = dp and world > 1
    B = s["batch"] * (world if dp else 1)
    md = synthetic.descriptors(shape, dropout=True)
    shard = EntityShard(s["num_ent"], rank, world)
    model = ConvE(md, seed=0, prec=prec, shard=shard, conv_in_height=s["H"], init_fast=s["num_ent"] > 1_000_000,
                  graphs_multi_gpu=graphs_multi, data_parallel=dp, overlap_grad_allreduce=overlap)
    n_batches = 8
    host = synthetic.make_batches(s["num_ent"], s["num_rel"], B, n_batches, seed=1)
    devb = [{k: torch.as_tensor(v).cuda() for k, v in hb.items()} for hb in host]
    coll = world > 1
    last = {}

    def train(i):
        last["loss"] = model.train_step(devb[i % n_batches])

    def evaluate(i):
        last["rank"], last["n_equal"] = model.filtered_ranks(devb[i % n_batches])
    train_ms, train_launches = ctx.timed(model, train, K, W, coll)
    if outputs is not None:
        outputs["train_loss"] = host_output(last["loss"])
        for k, t in model.state_dict().items():
            if k != "seed_dev":                  # a uint64 hash seed, not a computed value
                outputs["state__" + k.replace("/", "__")] = host_output(t)
    eval_ms, eval_launches = ctx.timed(model, evaluate, K, W, coll)
    if outputs is not None:
        outputs["eval_rank"], outputs["eval_n_equal"] = host_output(last["rank"]), host_output(last["n_equal"])
    nnz = float(np.mean([hb["e2_multi_col"].shape[0] for hb in host]))
    h2d = int(B * 8 * 2 + (B + 1) * 4 + nnz * 4)
    out = {
        "workload": workload_name(shape, s, B), "precision": prec, "dtype": DTYPE_NAME[prec],
        "value": B / train_ms * 1e3, "unit": "train rows/s", "ms_per_step": train_ms,
        "eval": {"value": B / eval_ms * 1e3, "unit": "eval queries/s", "ms_per_batch": eval_ms,
                 "gpu_launches_per_batch": eval_launches / K},
        "gpu_launches": int(train_launches), "gpu_launches_per_step": train_launches / K,
        "l2": "no flush: per-step working set ~%d MB > 126 MB L2; %d distinct input batches cycled" % (
            working_set_mb(s, B), n_batches),
        "cuda_graph": bool(model.use_graphs and (world == 1 or model.graphs_multi_gpu)),
        "parallelism": "single GPU" if world == 1 else "entity-sharded 1-N scorer x%d (rows/GPU=%d), %s" % (
            world, shard.rows,
            "data-parallel front end: global batch %d = %d rows/GPU, sync batch norm, one bucketed gradient "
            "all-reduce" % (B, B // world) if dp else "replicated front end (fixed batch %d)" % B),
        "_B": B,
    }
    if e2e:
        # end-to-end through the public API: pinned host batches in, loss / ranks read back every step
        def e2e_train(i):
            return float(model.train_step(host[i % n_batches]).item())

        def e2e_eval(i):
            r, _ = model.filtered_ranks(host[i % n_batches])
            return r.cpu()
        e2e_train_ms, _ = ctx.timed(model, e2e_train, K, W, coll)
        e2e_eval_ms, _ = ctx.timed(model, e2e_eval, K, W, coll)
        out["e2e"] = {"value": B / e2e_train_ms * 1e3, "unit": "train rows/s", "h2d_bytes_per_step": h2d,
                      "d2h_bytes_per_step": 8, "ms_per_step": e2e_train_ms, "eval_value": B / e2e_eval_ms * 1e3,
                      "eval_unit": "eval queries/s", "eval_ms_per_batch": e2e_eval_ms,
                      "eval_d2h_bytes_per_batch": B * 4}
    if breakdown and world == 1:
        out["kernel_ms"], out["rooflines"], out["roofline"] = kernel_breakdown(model, devb[0], peaks, prec, shape)
    model_ref = model
    del model, devb
    return out, model_ref, host


def kernel_breakdown(model, batch, peaks, prec, shape="wn18rr", reps=10):
    """CUDA-event time of each C-ABI stage in isolation (same stream, warm) and its roofline: algorithmic FLOPs or
    bytes (DESIGN.md §4) / time / measured peak.  Returns (kernel_ms, rooflines of every stage, dominant train stage)."""
    import torch
    from coper_b200._lib import call, ptr
    b = model.stage_batch(batch)
    model._train_device(b)                 # populate every buffer
    torch.cuda.synchronize()
    B, d, F = b.B, model.ent_emb_size, model.F
    Ns = model.shard.rows
    g = model.grads
    Pw, Pb = model.fc_weights.projections[-1], model.fc_bias.projections[-1]
    dc = Pw.shape[0]
    pos, neg = 0.9 + 1.0 / model.num_ent, 1.0 / model.num_ent
    bits_q = b.bits                      # query-major filter rows for the standalone (two-pass) rank kernel
    if bits_q is None:
        bits_q = torch.zeros(B, b.words, dtype=torch.int32, device=model.dev)
        call("coper_csr_to_bits", ptr(b.rowptr), ptr(b.col), B, model.shard.lo, model.shard.hi, ptr(bits_q))
    n_params = sum(p.numel() for _, p, _ in model.trainables)
    scatter_dst = torch.zeros_like(model.ent_emb) if Ns * d * 4 < (2 << 30) else None
    rows_touched = int(torch.unique(b.e1).numel())
    stages = {
        "cpg_fc_fwd": (lambda: call("coper_cpg_fc_fwd", ptr(b.cw), ptr(b.f), ptr(Pw), ptr(model.P_prep), ptr(b.cb), ptr(Pb), B, dc, F, d,
                                    Pb.shape[0], 1.0, None, 0, ptr(b.y), ptr(b.ws_cpg), b.ws_cpg_bytes, model.prec),
                       2.0 * B * dc * F * d, "tensor", True),
        "cpg_fc_bwd": (lambda: call("coper_cpg_fc_bwd", ptr(b.cw), ptr(b.f), ptr(Pw), ptr(model.P_prep), ptr(b.cb), ptr(Pb), ptr(b.dy),
                                    B, dc, F, d, Pb.shape[0], ptr(g["fc_weights/CPG/Projection0"]),
                                    ptr(g["fc_bias/CPG/Projection0"]), ptr(b.df), ptr(b.dcw), ptr(b.dcb), ptr(b.ws_cpg),
                                    b.ws_cpg_bytes, model.prec, 0), 4.0 * B * dc * F * d, "tensor", True),
        "score1n_bce_fwd_bwd": (lambda: call("coper_score1n_bce_fwd_bwd", ptr(b.q), ptr(model.ent_emb), ptr(model.E_prep),
                                             ptr(model.pred_bias), ptr(b.bits if model.prec == 0 else b.bitsT), B, Ns, d, pos, neg,
                                             1.0 / (B * model.num_ent), ptr(b.loss_sum), ptr(model._grad_buf(b)), b.ld, ptr(b.dq),
                                             ptr(g["ent_emb"]), ptr(g["pred_bias"]), ptr(b.ws), b.ws_bytes,
                                             model.prec), 6.0 * B * d * Ns, "tensor", True),
        "clip_and_amsgrad": (lambda: model._clip_and_apply(), n_params * 4.0 * 5, "hbm", True),
        "score1n_fwd": (lambda: model._score(b), 2.0 * B * d * Ns, "tensor", False),
        "score1n_rank_fused": (lambda: model._rank_device(b), 2.0 * B * d * Ns, "tensor", False),
        "filtered_rank": (lambda: call("coper_filtered_rank", ptr(model._scores_buf(b)), b.ld, B, Ns, ptr(b.e2), model.shard.lo,
                                       ptr(b.gold), ptr(bits_q), ptr(b.n_greater), ptr(b.n_equal)),
                          B * (4.0 * Ns + Ns / 8.0), "hbm", False),
        "gather_rows": (lambda: call("coper_gather_rows", ptr(model.ent_emb), model.shard.lo, model.shard.hi, d, ptr(b.e1), B,
                                     ptr(b.x0)), 2.0 * B * d * 4 + 8.0 * B, "hbm", True),
    }
    if scatter_dst is not None:
        stages["segscatter_add"] = (
            lambda: call("coper_segscatter_add_sq", ptr(b.e1), B, ptr(b.dx0), d, ptr(scatter_dst), None, model.shard.lo,
                         model.shard.hi), B * d * 4.0 + 2.0 * rows_touched * d * 4 + 8.0 * B, "hbm", True)
    traffic_all, traffic_src = load_traffic()
    out, roofs, best = {}, {}, None
    for name, (fn, work, bound, in_train) in stages.items():
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        out[name] = ms
        if bound == "tensor":
            peak, achieved, unit = peaks["bf16_tflops"], work / (ms * 1e-3) / 1e12, "TFLOP/s"
        else:
            peak, achieved, unit = peaks["hbm_gbs"], work / (ms * 1e-3) / 1e9, "GB/s"
        roofs[name] = {"bound": bound, "achieved": achieved, "peak": peak, "unit": unit, "frac": achieved / peak,
                       "traffic": traffic_all.get(shape, {}).get(prec, {}).get(name), "ms": ms,
                       "algorithmic_work": work, "in_train_step": in_train}
        if in_train and name not in ("gather_rows", "segscatter_add") and (best is None or ms > best[1]):
            best = (name, ms)
    name = best[0]
    roof = dict(roofs[name])
    roof.pop("in_train_step")
    roof = {"kernel": name, **roof,
            "peak_source": peaks["_source"] + (", bf16 dense burst" if roof["bound"] == "tensor" else ", copy bandwidth"),
            "note": "isolated launches of the C-ABI stage (its tcgen05 kernels + reductions), CUDA events on the launching "
                    "stream; prec=%s%s; traffic = DRAM bytes of the stage from the committed ncu capture (%s)" % (
                        prec, " (3 tf32 MMAs per product: tensor-pipe time = 6x the bf16-equivalent of the algorithmic "
                              "FLOPs)" if prec == "tf32x3" else
                        " (3 fp16 MMAs per product: tensor-pipe time = 3x the bf16-equivalent of the algorithmic FLOPs)"
                        if prec == "fp16x3" else "", traffic_src)}
    return out, roofs, roof


def hbm_kernels(ctx, peaks, reps=10):
    """gather / segmented scatter / standalone filtered rank at sizes where the HBM stream, not the launch, is timed
    (north_star: 'achieved HBM GB/s ... for gather and rank'); algorithmic bytes as in BASELINE.md §2."""
    torch = ctx.torch
    from coper_b200._lib import call, ptr
    dev = "cuda"
    out = {}

    def t(fn):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    def entry(ms, work, what):
        a = work / (ms * 1e-3) / 1e9
        return {"bound": "hbm", "achieved": a, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": a / peaks["hbm_gbs"],
                "ms": ms, "algorithmic_work": work, "workload": what}
    rows, d, M = 1_250_000, 256, 1 << 20
    E = torch.rand(rows, d, device=dev)
    idx = torch.randint(0, rows, (M,), device=dev, dtype=torch.int64)
    x = torch.empty(M, d, device=dev)
    ms = t(lambda: call("coper_gather_rows", ptr(E), 0, rows, d, ptr(idx), M, ptr(x)))
    out["gather_rows"] = entry(ms, 2.0 * M * d * 4 + 8.0 * M, "M=%d random rows of a [%d, %d] fp32 table" % (M, rows, d))
    dst = torch.zeros(rows, d, device=dev)
    ws_bytes = ctx.lib.coper_segscatter_workspace_bytes(M) if hasattr(ctx.lib, "coper_segscatter_workspace_bytes") else 0
    if ws_bytes:
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        touched = int(torch.unique(idx).numel())
        ms = t(lambda: call("coper_segscatter_add", ptr(idx), M, ptr(x), d, ptr(dst), 0, rows, ptr(ws), ws_bytes))
        out["segscatter_add"] = entry(ms, M * d * 4.0 + 2.0 * touched * d * 4 + 8.0 * M,
                                      "M=%d slices of width %d into %d distinct rows (radix sort + segmented sum)" % (
                                          M, d, touched))
    del E, x, dst
    B, N = 512, 1_250_000
    ld = -(-N // 32) * 32
    S = torch.randn(B, ld, device=dev)
    bits = torch.zeros(B, ld // 32, dtype=torch.int32, device=dev)
    e2 = torch.randint(0, N, (B,), device=dev, dtype=torch.int64)
    gold = torch.zeros(B, device=dev)
    ng, ne = torch.zeros(B, dtype=torch.int32, device=dev), torch.zeros(B, dtype=torch.int32, device=dev)
    call("coper_gold_scores", ptr(S), ld, B, N, ptr(e2), 0, ptr(gold))
    ms = t(lambda: call("coper_filtered_rank", ptr(S), ld, B, N, ptr(e2), 0, ptr(gold), ptr(bits), ptr(ng), ptr(ne)))
    out["filtered_rank"] = entry(ms, B * (4.0 * N + N / 8.0), "B=%d queries x N=%d fp32 logits + 1-bit filter rows" % (B, N))
    return out


def _free(ctx, *objs):
    for o in objs:
        del o
    gc.collect()
    ctx.torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--shape", default=os.environ.get("COPER_BENCH_SHAPE"),
                    help="default: wn18rr at N = 1, synth-10m at N > 1")
    ap.add_argument("--prec", default=os.environ.get("COPER_BENCH_PREC"),
                    help="default: fp16x3 (fp32-class) for the named datasets, bf16 for synth-10m")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-budget", type=float, default=20.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-breakdown", action="store_true")
    ap.add_argument("--no-alt", action="store_true", help="skip the extra bf16-engine measurement")
    ap.add_argument("--no-extra", action="store_true",
                    help="skip the blocks beside the headline (other configs, hbm_kernels, scaling base, wn18rr_weak)")
    ap.add_argument("--num-labels", type=int, default=1000,
                    help="also time the sampled-label training step (SURVEY §8f-2) with this many labels; 0 = skip")
    ap.add_argument("--no-graph-multi", action="store_true",
                    help="N > 1: do not capture the step (with its NCCL collectives) in a CUDA graph")
    ap.add_argument("--front-end", default=os.environ.get("COPER_BENCH_FRONT_END"),
                    choices=["data-parallel", "replicated"],
                    help="N > 1: data-parallel = every rank owns B rows of a global batch of N*B (weak scaling, "
                         "synchronised batch norm, bucketed gradient all-reduce); replicated = all ranks run the "
                         "front end of the same B rows, only the scorer is sharded (strong scaling).  Default: "
                         "replicated for synth-10m, data-parallel otherwise")
    ap.add_argument("--no-overlap", action="store_true",
                    help="data-parallel: all-reduce the whole gradient bucket at the end of the backward pass instead "
                         "of overlapping the generator-weight gradient with the conv backward")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps of the headline workload, write what its last train step and eval "
                         "batch computed as DIR/<name>.npy (float32 / float64; arrays above %d elements as a fixed "
                         "seeded sample; N > 1: rank 0's entity rows) so that two builds can be compared on the same "
                         "inputs" % DUMP_MAX_ELEMS)
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    multi = max(world, args.gpus) > 1
    explicit = args.shape is not None
    shape = args.shape or ("synth-10m" if multi else "wn18rr")
    prec = args.prec or ("bf16" if shape == "synth-10m" else "fp16x3")
    front = args.front_end or ("replicated" if shape == "synth-10m" else "data-parallel")
    dp = multi and front == "data-parallel"
    from coper_b200 import synthetic
    s = synthetic.SHAPES[shape]
    B = s["batch"] * (max(world, args.gpus) if dp else 1)
    scaling = "weak" if (dp or not multi) else "strong"
    workload = workload_name(shape, s, B)

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, shape, B, scaling, workload)
        return

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    # stdout carries exactly ONE JSON line: everything libraries print while we run (e.g. NCCL's version banner)
    # is diverted to stderr at the file-descriptor level
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = Ctx(rank, world, local_rank)
    peaks = load_peaks()
    K, W = args.steps, args.warmup
    extra = not args.no_extra and not explicit
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    outputs = {} if args.dump_outputs and rank == 0 else None
    head, model, host = measure(ctx, shape, prec, K, W, peaks, sharded=True, dp=dp, e2e=True,
                                breakdown=not args.no_breakdown, graphs_multi=not args.no_graph_multi,
                                overlap=not args.no_overlap, outputs=outputs)
    clocks = sampler.stop() if rank == 0 else None
    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)
    n_batches = len(host)

    alt = sampled = cpu = None
    configs, hbm, base, weak = {}, None, None, None
    if world == 1:
        md = synthetic.descriptors(shape, dropout=True)
        from coper_b200.models import ConvE, EntityShard
        shard = EntityShard(s["num_ent"], 0, 1)
        devb = [{k: torch.as_tensor(v).cuda() for k, v in hb.items()} for hb in host]
        # the same workload on the bf16 tensor-pipe engine (north_star's throughput path), beside the headline
        if prec != "bf16" and not args.no_alt:
            _free(ctx, model)
            model = None
            m16 = ConvE(md, seed=0, prec="bf16", shard=shard, conv_in_height=s["H"], init_fast=s["num_ent"] > 1_000_000)
            t_ms, _ = ctx.timed(m16, lambda i: m16.train_step(devb[i % n_batches]), K, W)
            e_ms, _ = ctx.timed(m16, lambda i: m16.filtered_ranks(devb[i % n_batches]), K, W)
            alt = {"precision": "bf16 (tcgen05 kind::f16, fp32 accumulate)", "value": B / t_ms * 1e3,
                   "unit": "train rows/s", "ms_per_step": t_ms, "eval_value": B / e_ms * 1e3,
                   "eval_unit": "eval queries/s", "eval_ms_per_batch": e_ms}
            if not args.no_breakdown:
                alt["kernel_ms"], alt["rooflines"], _ = kernel_breakdown(m16, devb[0], peaks, "bf16", shape)
            _free(ctx, m16)
        # SURVEY §8f-2: the sampled-label training step the shipped big-dataset configs use (num_labels = 1000)
        if args.num_labels > 0 and s["num_ent"] <= 1_000_000:
            md_s = copy.deepcopy(md)
            md_s["use_negative_sampling"] = True
            _free(ctx, model)
            model = None
            ms = ConvE(md_s, seed=0, prec=prec, shard=shard, conv_in_height=s["H"])
            sb_host = [synthetic.to_sampled(hb, s["num_ent"], args.num_labels, seed=7 + i) for i, hb in enumerate(host)]
            sb_dev = [{k: torch.as_tensor(v).cuda() for k, v in hb.items()} for hb in sb_host]
            t_ms, n_l = ctx.timed(ms, lambda i: ms.train_step(sb_dev[i % n_batches]), K, W)
            e2e_ms, _ = ctx.timed(ms, lambda i: float(ms.train_step(sb_host[i % n_batches]).item()), K, W)
            # labels drawn on the device (coper_sample_labels) from host CSR batches: only ids + id lists cross PCIe
            dev_host = [dict(hb, sample_on_device=(args.num_labels, 10.0)) for hb in host]
            ds_ms, _ = ctx.timed(ms, lambda i: float(ms.train_step(dev_host[i % n_batches]).item()), K, W)
            gather_bytes = float(B * args.num_labels * s["ent_emb_size"] * 4)
            sampled = {"num_labels": args.num_labels, "value": B / t_ms * 1e3, "unit": "train rows/s", "ms_per_step": t_ms,
                       "e2e_value": B / e2e_ms * 1e3, "e2e_ms_per_step": e2e_ms,
                       "device_sampling_e2e_value": B / ds_ms * 1e3, "device_sampling_e2e_ms_per_step": ds_ms,
                       "device_sampling_h2d_bytes_per_step": head["e2e"]["h2d_bytes_per_step"],
                       "h2d_bytes_per_step": int(B * 16 + B * args.num_labels * 8), "gpu_launches_per_step": n_l / K,
                       "gather_bytes_per_step": int(gather_bytes),
                       # the step streams the [B, L, d] gathered rows twice (scores + dq, then the dE scatter): HBM-bound
                       "roofline": {"bound": "hbm", "achieved": 2 * gather_bytes / (t_ms * 1e-3) / 1e9,
                                    "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                    "frac": 2 * gather_bytes / (t_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                    "algorithmic_work": 2 * gather_bytes,
                                    "note": "whole sampled-label step; algorithmic bytes = 2 passes over the gathered "
                                            "[B, L, d] fp32 rows"}}
            _free(ctx, ms, sb_dev)
        _free(ctx, model, devb)
        model = None
        if extra:
            # ---- every other named configuration of BASELINE.json on one GPU (parity-tested at full size in tests/)
            for other in ("fb15k-237", "nell-995", "yago3-10", "synth-10m"):
                if other == shape:
                    continue
                try:
                    blk, m_o, _ = measure(ctx, other, "bf16" if other == "synth-10m" else "fp16x3", K, W, peaks,
                                          e2e=True, breakdown=not args.no_breakdown)
                    blk.pop("_B")
                    blk["steps"], blk["warmup"] = K, W
                    configs[other] = blk
                    _free(ctx, m_o)
                except Exception as exc:           # one failing extra block must not take the headline down
                    configs[other] = {"error": repr(exc)}
                    _free(ctx)
            try:
                hbm = hbm_kernels(ctx, peaks)
            except Exception as exc:
                hbm = {"error": repr(exc)}
            _free(ctx)
        if rank == 0 and not args.no_cpu_baseline:
            try:
                cpu = run_cpu_baseline(shape, args.cpu_budget)
            except Exception as exc:  # the CPU leg must never take the GPU numbers down with it
                cpu = {"value": None, "unit": "train rows/s", "cores": os.cpu_count(), "kind": "port",
                       "sample": "failed: %r" % (exc,)}
    else:
        _free(ctx, model)
        model = None
        if extra:
            # ---- the data-parallel WN18RR weak-scaling numbers (global batch N * 512), all ranks
            try:
                weak, m_w, _ = measure(ctx, "wn18rr", "fp16x3", K, W, peaks, sharded=True, dp=True, e2e=True,
                                       breakdown=False, graphs_multi=not args.no_graph_multi, overlap=not args.no_overlap)
                weak.pop("_B")
                weak["scaling"] = "weak"
                _free(ctx, m_w)
            except Exception as exc:
                weak = {"error": repr(exc)}
            # ---- strong-scaling base: the headline workload on ONE GPU, measured by rank 0 while the others wait
            dist.barrier()
            torch.cuda.synchronize()
            if rank == 0:
                try:
                    base, m_b, _ = measure(ctx, shape, prec, K, W, peaks, sharded=False, e2e=False, breakdown=False)
                    base = {"n_gpus": 1, "value": base["value"], "unit": base["unit"], "ms_per_step": base["ms_per_step"],
                            "eval_value": base["eval"]["value"], "eval_ms_per_batch": base["eval"]["ms_per_batch"],
                            "steps": K, "warmup": W,
                            "note": "same workload, single GPU, measured by rank 0 in this run; strong-scaling ratio = "
                                    "value / (n_gpus * strong_scaling_base.value)"}
                    _free(ctx, m_b)
                except Exception as exc:
                    base = {"error": repr(exc)}
            dist.barrier()
    if world > 1:
        dist.barrier()
    if rank != 0:
        _finish(world, torch, dist)
        return
    line = {
        "metric": "train_rows_per_s", "value": head["value"], "unit": "train rows/s", "n_gpus": world,
        "steps": K, "warmup": W, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
        "scaling": scaling, "vs_baseline": None, "dtype": DTYPE_NAME[prec], "data": "synthetic",
        "config": {"workload": workload, "precision": prec, "parallelism": head["parallelism"], "l2": head["l2"],
                   "dropout": "on (feature-map 0.3, output 0.2)", "batch_norm": "batch statistics (train)",
                   "cuda_graph": head["cuda_graph"]},
        "eval": head["eval"], "e2e": head.get("e2e"),
        "gpu_launches": head["gpu_launches"], "gpu_launches_per_step": head["gpu_launches_per_step"],
        "clocks": clocks, "roofline": head.get("roofline"), "rooflines": head.get("rooflines"),
        "kernel_ms": head.get("kernel_ms"), "bf16": alt, "sampled_labels": sampled, "cpu_baseline": cpu,
        "configs": configs or None, "hbm_kernels": hbm, "strong_scaling_base": base, "wn18rr_weak": weak,
        "peaks": {k: peaks.get(k) for k in ("hbm_gbs", "bf16_tflops", "bf16_tflops_sustained", "_source")},
    }
    sys.stdout.flush()
    os.dup2(real_stdout, 1)
    print(json.dumps(line), flush=True)
    _finish(world, torch, dist)


def _finish(world, torch, dist):
    """N > 1: leave without tearing NCCL down — destroy_process_group() blocks forever once collectives have been
    captured into CUDA graphs (observed on the 2-GPU box); everything is flushed and synchronised first."""
    if world > 1:
        sys.stdout.flush()
        sys.stderr.flush()
        torch.cuda.synchronize()
        os._exit(0)


if __name__ == "__main__":
    main()
