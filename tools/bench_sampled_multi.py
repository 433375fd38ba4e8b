"""Sampled-label training step (num_labels = L) at the WN18RR shape, on one GPU and entity-sharded over P GPUs.

    python tools/bench_sampled_multi.py --out sampled.json                                  # one process, one GPU
    torchrun --nproc-per-node P tools/bench_sampled_multi.py --out sampled_P.json           # P processes, NCCL

One process times today's single-GPU step (``coper_score_sampled_bce_fwd_bwd``) on device-resident host-sampled
batches and with the labels drawn on the device.  Under torchrun every rank holds N/P entity rows and both multi-GPU
schedules are timed with the step captured as a CUDA graph (collectives included):
  replicated     every rank runs the front end on the same B = 512 queries; fixed batch (strong scaling)
  data-parallel  global batch Bg = P * 512, each rank runs the front end on its 512 rows (weak scaling)
Times are CUDA-event times over --steps steps after --warmup steps, read on rank 0.  The JSON also carries, from the
cost model (not measured), the bytes of gathered entity rows each rank's scorer reads per step.  The card's name and
power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                                   # the numbers are still reported, without the card
        return {"error": str(e)}


def time_step(model, batches, steps, warmup):
    """ms per train step: CUDA events around `steps` steps after `warmup` (the first two calls run eagerly and
    capture the graph)."""
    import torch
    for i in range(warmup):
        model.train_step(batches[i % len(batches)])
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(steps):
        loss = model.train_step(batches[i % len(batches)])
    b.record()
    b.synchronize()
    assert torch.isfinite(loss).item()
    return a.elapsed_time(b) / steps


def device_batches(shape, B, L, n, sampling, seed=11):
    """n batches of B queries on the GPU: host-sampled [B, L] ids / labels, or the CSR lists for device sampling."""
    import torch
    from coper_b200 import synthetic
    s = synthetic.SHAPES[shape]
    host = synthetic.make_batches(s["num_ent"], s["num_rel"], B, n, seed=seed)
    out = []
    for i, hb in enumerate(host):
        b = hb if sampling else synthetic.to_sampled(hb, s["num_ent"], L, seed=7 + i)
        b = {k: torch.as_tensor(v).cuda() for k, v in b.items()}
        if sampling:
            b["sample_on_device"] = (L, 10.0)
        out.append(b)
    return out


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True, help="JSON file to write (rank 0)")
    ap.add_argument("--num-labels", type=int, default=1000)
    ap.add_argument("--prec", default="fp16x3", choices=["fp32", "tf32x3", "fp16x3", "bf16"])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args(argv)
    import torch
    import torch.distributed as dist
    from coper_b200 import synthetic
    from coper_b200.models import ConvE
    from coper_b200.sharding import EntityShard
    if not torch.cuda.is_available():
        raise SystemExit("bench_sampled_multi needs a CUDA device")
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > torch.cuda.device_count():
        raise SystemExit("%d ranks need %d GPUs, %d visible" % (world, world, torch.cuda.device_count()))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    shape, L = "wn18rr", args.num_labels
    s = synthetic.SHAPES[shape]
    B, d = s["batch"], s["ent_emb_size"]
    md = synthetic.descriptors(shape, dropout=True, use_negative_sampling=True)
    res = {"workload": "sampled-label train step, WN18RR shape (N=%d, d=%d), B=%d per front end, L=%d"
                       % (s["num_ent"], d, B, L),
           "precision": args.prec, "gpus": world, "steps": args.steps, "warmup": args.warmup,
           "card": card() if rank == 0 else None}
    if world == 1:
        m = ConvE(md, seed=0, prec=args.prec, conv_in_height=s["H"])
        for key, sampling in (("host_sampled", False), ("device_sampling", True)):
            t = time_step(m, device_batches(shape, B, L, 8, sampling), args.steps, args.warmup)
            res[key] = {"ms_per_step": t, "rows_per_s": B / t * 1e3}
        res["multi_gpu"] = "run under torchrun --nproc-per-node P for the sharded schedules"
    else:
        for sched, dp in (("replicated", False), ("data_parallel", True)):
            Bg = B * world if dp else B
            m = ConvE(md, seed=0, prec=args.prec, conv_in_height=s["H"], shard=EntityShard(s["num_ent"], rank, world),
                      data_parallel=dp, graphs_multi_gpu=True)
            t = time_step(m, device_batches(shape, Bg, L, 8, False), args.steps, args.warmup)
            res[sched] = {"batch": Bg, "ms_per_step": t, "rows_per_s": Bg / t * 1e3,
                          "scaling": "weak" if dp else "strong"}
            del m
            torch.cuda.empty_cache()
    # cost model (not measured): bytes of fp32 entity rows the scorer reads per rank and step; with uniform ids each
    # rank owns 1/P of the Bg * L positions -> flat in P for data-parallel (Bg = P * B), 1/P for replicated
    res["cost_model_scorer_row_bytes_per_rank"] = {
        sched: 4 * d * L * (B * world if sched == "data_parallel" else B) // world
        for sched in (("replicated", "data_parallel") if world > 1 else ("single",))}
    if rank == 0:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)
        print(json.dumps(res))
    if world > 1:
        # (collectives captured into CUDA graphs: leave without tearing NCCL down, as run_cpg does)
        torch.cuda.synchronize()
        sys.stdout.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
