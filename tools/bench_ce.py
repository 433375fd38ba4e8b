"""Train-step time of the softmax cross-entropy objective against the BCE objective on one GPU, and the log-sum-exp
pass against the fused rank kernel (both read E once and write nothing of size [B, N]).

    python tools/bench_ce.py --out profiles/ce.json [--steps 50]

Per case the BCE and CE models are timed in the same run, alternating in rounds: device-resident steps (the staged
batch replayed, CUDA events) and end-to-end steps (host batch staged every step, host clock to a synchronise).
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

import torch  # noqa: E402

from coper_b200 import _lib as L  # noqa: E402
from coper_b200 import synthetic  # noqa: E402
from coper_b200.models import ConvE  # noqa: E402

CASES = [("wn18rr", "fp16x3"), ("wn18rr", "bf16"), ("synth-10m", "bf16")]


def _card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split("\n")[0]
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as exc:                      # the card is part of the number: refuse to report without it
        raise SystemExit("cannot read the card name / power limit: %s" % exc)


def _events_ms(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def bench_steps(shape, prec, steps, rounds):
    s = synthetic.SHAPES[shape]
    batches = synthetic.make_batches(s["num_ent"], s["num_rel"], s["batch"], 4, seed=1)
    models = {}
    for loss in ("bce", "softmax_ce"):
        md = synthetic.descriptors(shape, loss=loss)
        m = ConvE(md, device="cuda:0", prec=prec, conv_in_height=s["H"], init_fast=True)
        for _ in range(3):                         # eager, capture, replay
            m.train_step(batches[0])
        models[loss] = m
    res = {k: {"device_ms": [], "e2e_ms": []} for k in models}
    for _ in range(rounds):
        for loss, m in models.items():
            b = m.stage_batch(batches[0])
            res[loss]["device_ms"].append(_events_ms(lambda: m._run_train(("train", b.B), b, True), steps))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(steps):
                m.train_step(batches[i % len(batches)])
            torch.cuda.synchronize()
            res[loss]["e2e_ms"].append((time.perf_counter() - t0) * 1e3 / steps)
    out = {}
    for loss, r in res.items():
        out[loss] = {k: min(v) for k, v in r.items()}
        out[loss]["loss_after"] = float(models[loss].train_step(batches[1]).item())
    del models
    torch.cuda.empty_cache()
    return out


def bench_lse_vs_rank(shape, prec, reps):
    """coper_score1n_lse against coper_score1n_rank_prepared on the same prepared operands and shape."""
    s = synthetic.SHAPES[shape]
    B, N, d = s["batch"], s["num_ent"], s["ent_emb_size"]
    p = L.PREC[prec]
    lib = L.load()
    g = torch.Generator(device="cuda").manual_seed(0)
    q = torch.rand(B, d, device="cuda", generator=g) - 0.5
    E = (torch.rand(N, d, device="cuda", generator=g) - 0.5) * 0.1
    bias = torch.zeros(N, device="cuda")
    qp = torch.empty(lib.coper_prepared_bytes(B, d, p), dtype=torch.uint8, device="cuda")
    Ep = torch.empty(lib.coper_prepared_bytes(N, d, p), dtype=torch.uint8, device="cuda")
    L.call("coper_prepare_operand", L.ptr(q), B, d, d, p, L.ptr(qp))
    L.call("coper_prepare_operand", L.ptr(E), N, d, d, p, L.ptr(Ep))
    ws = torch.empty(lib.coper_score1n_lse_workspace_bytes(B, N, d, p), dtype=torch.uint8, device="cuda")
    ml = torch.empty(B, 2, device="cuda")
    gold = torch.zeros(B, device="cuda")
    filt = torch.zeros(N, -(-B // 32), dtype=torch.int32, device="cuda")
    cnt = torch.zeros(2, B, dtype=torch.int32, device="cuda")
    lse = lambda: L.call("coper_score1n_lse", L.ptr(q), L.ptr(E), L.ptr(Ep), L.ptr(bias), B, N, d, L.ptr(ml), L.ptr(ws),
                         ws.numel(), p)
    rank = lambda: L.call("coper_score1n_rank_prepared", L.ptr(qp), L.ptr(Ep), L.ptr(bias), B, N, d, L.ptr(gold),
                          L.ptr(filt), L.ptr(cnt[0]), L.ptr(cnt[1]), p)
    for f in (lse, rank):
        f()
    torch.cuda.synchronize()
    t = {"lse_ms": [], "rank_ms": []}
    for _ in range(5):
        t["lse_ms"].append(_events_ms(lse, reps))
        t["rank_ms"].append(_events_ms(rank, reps))
    return {k: min(v) for k, v in t.items()}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ce.py measures the GPU: no CUDA device")
    name, power = _card()
    result = {"card": name, "power_limit": power, "steps": args.steps, "rounds": args.rounds,
              "note": "min over rounds; BCE and CE alternate within each round", "cases": []}
    for shape, prec in CASES:
        steps = args.steps if shape != "synth-10m" else max(5, args.steps // 10)
        case = {"shape": shape, "prec": prec, "train": bench_steps(shape, prec, steps, args.rounds),
                "lse_vs_rank": bench_lse_vs_rank(shape, prec, 20 if shape != "synth-10m" else 5)}
        print(json.dumps(case), flush=True)
        result["cases"].append(case)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
