"""Scores and ranks of given candidates on one GPU: whole calls and the two kernels, against the gather bound.

For each (shape, C) it times, with CUDA events after warm-up and on the same staged batch:
  score_candidates   ConvE.score_candidates(batch, cand)      (front end + coper_score_candidates + padding mask)
  candidate_ranks    ConvE.candidate_ranks(batch, cand)       (front end + gold + coper_candidate_rank, filtered)
  filtered_ranks     ConvE.filtered_ranks(batch)              (front end + rank against all N entities, for comparison)
  score_kernel       coper_score_candidates alone on the model's q
  rank_kernel        coper_candidate_rank alone (filtered, the engine's bit layout)
Bytes of a kernel = B*C*(4d + 4 + 4) + 4*B*d (rows, bias, ids; q), + 4*B*C for the scores coper_score_candidates
writes; the bound is bytes / 7.7 TB/s (HBM3e of one B200).  A table that fits the 126 MB L2 (WN18RR: 33 MB) is read
from L2 after the first pass, so its kernel time is compared with that bound only as a ratio, not as an HBM fraction.
Candidates are uniform over all entities.  Writes one JSON file with the card's name and power limit read in the same
run.

    python tools/bench_candidates.py --out profiles/r05_candidates.json
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_topk import card, time_ms  # noqa: E402

HBM_BPS = 7.7e12
L2_BYTES = 126 << 20
# (shape, engine, candidate counts): the WN18RR shape with the fp16x3 model, synth-10m with the bf16 model
CASES = [("wn18rr", "fp16x3", (1, 100, 1000)), ("synth-10m", "bf16", (1000,))]


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "candidates_bench.json"))
    ap.add_argument("--shapes", default="wn18rr,synth-10m")
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args(argv)
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_candidates needs a CUDA device")
    from coper_b200 import synthetic
    from coper_b200._lib import call, ptr
    from coper_b200.models import ConvE
    rows = []
    for shape, prec, cs in CASES:
        if shape not in args.shapes.split(","):
            continue
        s = synthetic.SHAPES[shape]
        B, N, d = s["batch"], s["num_ent"], s["ent_emb_size"]
        batch = synthetic.make_batches(N, s["num_rel"], B, 1, seed=11)[0]
        t0 = time.time()
        m = ConvE(synthetic.descriptors(shape, dropout=False), seed=0, prec=prec, conv_in_height=s["H"],
                  init_fast=N > 1_000_000)
        setup_s = time.time() - t0
        t_full = time_ms(lambda: m.filtered_ranks(batch), args.iters, args.warmup)
        rng = np.random.default_rng(0)
        for C in cs:
            cand = rng.integers(0, N, (B, C)).astype(np.int32)
            t_score = time_ms(lambda: m.score_candidates(batch, cand), args.iters, args.warmup)
            t_rank = time_ms(lambda: m.candidate_ranks(batch, cand), args.iters, args.warmup)
            b = m._buffers(B)
            c = b.cand[C]
            sh = m.shard
            bits = b.bits if m.prec == 0 else b.bitsT
            k_score = time_ms(lambda: call("coper_score_candidates", ptr(b.q), ptr(m.ent_emb), ptr(m.pred_bias),
                                           ptr(c.cand), B, C, d, sh.lo, sh.hi, ptr(c.scores)),
                              args.iters, args.warmup)
            k_rank = time_ms(lambda: call("coper_candidate_rank", ptr(b.q), ptr(m.ent_emb), ptr(m.pred_bias),
                                          ptr(c.cand), ptr(c.e2), B, C, d, sh.lo, sh.hi, ptr(c.gold), ptr(bits),
                                          int(m.prec != 0), ptr(c.n_greater), ptr(c.n_equal)),
                             args.iters, args.warmup)
            rank_bytes = B * C * (4 * d + 4 + 4) + 4 * B * d
            score_bytes = rank_bytes + 4 * B * C
            table = N * d * 4
            row = {"shape": shape, "prec": prec, "B": B, "C": C, "num_ent": N, "d": d,
                   "table_MB": round(table / 1e6, 1), "table_in_l2": table < L2_BYTES,
                   "score_candidates_ms": round(t_score, 4), "candidate_ranks_ms": round(t_rank, 4),
                   "filtered_ranks_ms": round(t_full, 4),
                   "score_kernel_us": round(k_score * 1e3, 2), "rank_kernel_us": round(k_rank * 1e3, 2),
                   "score_kernel_MB": round(score_bytes / 1e6, 3), "rank_kernel_MB": round(rank_bytes / 1e6, 3),
                   "score_kernel_TBps": round(score_bytes / (k_score * 1e-3) / 1e12, 3),
                   "rank_kernel_TBps": round(rank_bytes / (k_rank * 1e-3) / 1e12, 3),
                   "score_kernel_over_hbm_bound": round(score_bytes / HBM_BPS / (k_score * 1e-3), 3),
                   "rank_kernel_over_hbm_bound": round(rank_bytes / HBM_BPS / (k_rank * 1e-3), 3),
                   "model_setup_s": round(setup_s, 1)}
            rows.append(row)
            print(json.dumps(row), flush=True)
        del m
        torch.cuda.empty_cache()
    out = {"card": card(), "iters": args.iters, "warmup": args.warmup, "hbm_TBps_datasheet": HBM_BPS / 1e12,
           "note": "kernel times: CUDA events around back-to-back launches of one kernel (the table of the WN18RR shape "
                   "stays in L2 between them); *_over_hbm_bound = (bytes / 7.7 TB/s) / kernel time",
           "rows": rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
