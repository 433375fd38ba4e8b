"""Top-k link prediction on one GPU: the fused call against what a user would otherwise run.

For each (shape, precision, k) it times, with CUDA events after warm-up and on the same staged batch:
  predict_topk   ConvE.predict_topk(batch, k)              (front end + fused scorer / top-k + merge)
  ranks          ConvE.filtered_ranks(batch)              (front end + gold + fused rank counts: the evaluation path)
  all_topk       ConvE.predict_all(batch) + torch.topk    (front end + [B, N] fp32 logits in HBM + torch's selection)
and writes one JSON file with the card's name and power limit read in the same run.

    python tools/bench_topk.py --out profiles/r03_topk_bench.json [--shapes wn18rr,1m,synth-10m] [--iters 20]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"wn18rr": ("wn18rr", None), "1m": ("wn18rr", 1_000_000), "synth-10m": ("synth-10m", None)}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                                   # the numbers are still reported, without the card
        return {"error": str(e)}


def time_ms(fn, iters, warmup):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "topk_bench.json"))
    ap.add_argument("--shapes", default="wn18rr,1m,synth-10m")
    ap.add_argument("--precs", default="fp16x3,bf16")
    ap.add_argument("--ks", default="1,10,100")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_topk needs a CUDA device")
    from coper_b200 import synthetic
    from coper_b200.models import ConvE
    rows = []
    for shape in args.shapes.split(","):
        base, n_override = SHAPES[shape]
        s = dict(synthetic.SHAPES[base])
        if n_override:
            s["num_ent"] = n_override
        B, N, d = s["batch"], s["num_ent"], s["ent_emb_size"]
        batch = synthetic.make_batches(N, s["num_rel"], B, 1, seed=11)[0]
        for prec in args.precs.split(","):
            t0 = time.time()
            md = synthetic.descriptors(base, dropout=False, num_ent=N)
            m = ConvE(md, seed=0, prec=prec, conv_in_height=s["H"], init_fast=N > 1_000_000)
            setup_s = time.time() - t0
            t_rank = time_ms(lambda: m.filtered_ranks(batch), args.iters, args.warmup)

            def all_topk(k):
                S = m.predict_all(batch)
                return torch.topk(S, k, dim=1)
            for k in (int(x) for x in args.ks.split(",")):
                t_topk = time_ms(lambda: m.predict_topk(batch, k=k), args.iters, args.warmup)
                t_all = time_ms(lambda: all_topk(k), max(3, args.iters // 4), 1)
                row = {"shape": shape, "B": B, "num_ent": N, "d": d, "prec": prec, "k": k,
                       "predict_topk_ms": round(t_topk, 4), "filtered_ranks_ms": round(t_rank, 4),
                       "predict_all_torch_topk_ms": round(t_all, 4),
                       "topk_over_ranks": round(t_topk / t_rank, 3), "all_topk_over_topk": round(t_all / t_topk, 3),
                       "scorer_tflop": round(2.0 * B * d * N / 1e12, 4), "model_setup_s": round(setup_s, 1)}
                rows.append(row)
                print(json.dumps(row), flush=True)
            del m
            torch.cuda.empty_cache()
    out = {"card": card(), "iters": args.iters, "warmup": args.warmup,
           "note": "predict_all + torch.topk is unfiltered; predict_topk is filtered by e2_multi", "rows": rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
