"""Sampled-label training on an entity-sharded table: the sharded scorer (coper_score_sampled_bce_fwd_bwd_sharded)
against the unsharded one, the two multi-GPU schedules of ConvE against the single-GPU model and the oracle, and the
entry point under torchrun.  The world-2 tests use the harness of test_gpu_multi.py (NCCL with >= 2 GPUs, else two
processes sharing cuda:0 over gloo)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import yaml

from oracle import conve_oracle as O
from oracle import dropout_hash as DH
from test_gpu_multi import DP_CFG, _free_port, _init_dist

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------------ kernel, one GPU
def _kernel_inputs(N, d, L, B, seed):
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(B, d, generator=g) * 0.3
    E = torch.randn(N, d, generator=g) * 0.3
    bias = torch.randn(N, generator=g) * 0.1
    lookup = torch.randint(0, N, (B, L), generator=g, dtype=torch.int32)
    lookup[:, -1] = lookup[:, 0]                        # duplicates within a row
    lookup[B // 2:] = lookup[:B - B // 2]               # ... and across rows
    lookup[1] = torch.randint(0, 100, (L,), generator=g, dtype=torch.int32)   # a query only the first shard scores
    labels = (torch.rand(B, L, generator=g) < 0.2).float()
    return [t.cuda() for t in (q, E, bias, lookup, labels)]


def _run_scorer(q, E, bias, lookup, labels, N, shard=None):
    """One call of the unsharded (shard None) or sharded scorer.  scores / g are pre-filled with a sentinel."""
    from coper_b200._lib import call, load, ptr
    B, L = lookup.shape
    d = q.shape[1]
    rows = E.shape[0]
    f = dict(dtype=torch.float32, device="cuda")
    out = {"loss": torch.zeros(1, dtype=torch.float64, device="cuda"), "scores": torch.full((B, L), -7.25, **f),
           "g": torch.full((B, L), -7.25, **f), "dq": torch.full((B, d), 3.5, **f),
           "dE_sum": torch.zeros(rows, d, **f), "dE_sq": torch.zeros(rows, d, **f),
           "db_sum": torch.zeros(rows, **f), "db_sq": torch.zeros(rows, **f)}
    lib = load()
    args = (ptr(q), ptr(E), ptr(bias), ptr(lookup), ptr(labels), B, L, N, d, 0.9, 1.0 / N, 1.0 / (B * L),
            ptr(out["loss"]), ptr(out["scores"]), ptr(out["g"]), ptr(out["dq"]), ptr(out["dE_sum"]),
            ptr(out["dE_sq"]), ptr(out["db_sum"]), ptr(out["db_sq"]))
    if shard is None:
        ws = torch.empty(lib.coper_score_sampled_workspace_bytes(B, L), dtype=torch.uint8, device="cuda")
        call("coper_score_sampled_bce_fwd_bwd", *args, ptr(ws), ws.numel())
    else:
        ws = torch.empty(lib.coper_score_sampled_sharded_workspace_bytes(B, L), dtype=torch.uint8, device="cuda")
        call("coper_score_sampled_bce_fwd_bwd_sharded", *args, shard.lo, shard.hi, ptr(ws), ws.numel())
    torch.cuda.synchronize()
    return {k: v.cpu() for k, v in out.items()}


def _bits(t):
    return t.contiguous().view(torch.int32)


@pytest.mark.parametrize("d", [200, 256])
@pytest.mark.parametrize("L", [12, 100])
def test_sharded_scorer_matches_unsharded(d, L):
    from coper_b200.sharding import EntityShard
    N, B = 1003, 130
    q, E, bias, lookup, labels = _kernel_inputs(N, d, L, B, seed=d + L)
    ref = _run_scorer(q, E, bias, lookup, labels, N)
    lk = lookup.cpu()
    for P in (1, 2, 3):
        parts = []
        for r in range(P):
            sh = EntityShard(N, r, P)
            assert ((lk >= sh.lo) & (lk < sh.hi)).any()                     # ids in every shard
            o = _run_scorer(q, E[sh.lo:sh.hi].contiguous(), bias[sh.lo:sh.hi].contiguous(), lookup, labels, N, sh)
            own = (lk >= sh.lo) & (lk < sh.hi)
            for k in ("scores", "g"):
                assert torch.equal(_bits(o[k])[own], _bits(ref[k])[own]), (P, r, k)
                assert (o[k][~own] == -7.25).all(), (P, r, k)              # non-owned entries untouched
            for k in ("dE_sum", "dE_sq", "db_sum", "db_sq"):
                assert torch.equal(_bits(o[k]), _bits(ref[k][sh.lo:sh.hi])), (P, r, k)
            none = ~own.any(1)
            assert (o["dq"][none] == 0).all()
            if P > 1 and r > 0:
                assert bool(none[1])                                         # query 1 has no lookup here
            parts.append(o)
        if P == 1:                                                          # every output bit-identical
            for k in ref:
                assert torch.equal(parts[0][k], ref[k]), k
        loss = sum(float(o["loss"]) for o in parts)
        assert abs(loss - float(ref["loss"])) <= 1e-6 * abs(float(ref["loss"]))
        dq = sum(o["dq"].double() for o in parts)
        assert (dq - ref["dq"].double()).abs().max() <= 1e-5 * ref["dq"].abs().max()


# ------------------------------------------------------------------------------------------------ world 2
REP_CFG = dict(num_ent=1003, num_rel=22, ent_emb_size=200, rel_emb_size=8, context_rel_out=[],
               batch_norm_train_stats=True, batch_norm_momentum=0.1, hidden_dropout=0.3, output_dropout=0.2)
B_REP, L_SAMP = 130, 100


def _sampled_batch(cfg, B, seed=5):
    """Host-sampled batch: [B, L] ids with positives first, duplicates within and across rows, labels = membership."""
    e1, rel, e2, rowptr, col = O.synthetic_batch(cfg, B, seed=seed, mean_pos=5.0)
    dense = O.csr_to_dense(rowptr, col, cfg.num_ent)
    rng = np.random.default_rng(seed + 1)
    lookup = rng.integers(0, cfg.num_ent, (B, L_SAMP)).astype(np.int32)
    for i in range(B):
        pos = col[rowptr[i]:rowptr[i + 1]][:3]
        lookup[i, :len(pos)] = pos
    lookup[:, -1] = lookup[:, 0]
    labels = dense[np.arange(B)[:, None], lookup].astype(np.float32)
    return {"e1": e1, "rel": rel, "e2": e2, "e2_multi": labels, "lookup_values": lookup}


def _descr(cfg):
    from test_gpu_model import descriptors
    md = descriptors(cfg, 1e-2)
    md["use_negative_sampling"] = True
    return md


def _snapshot(m, loss):
    return dict(loss=loss, norm=float(m.clip_out[1].item()), dE=m.grads["ent_emb"].cpu().numpy(),
                dE_sq=m.grad_sq["ent_emb"].cpu().numpy(), db=m.grads["pred_bias"].cpu().numpy(),
                ent=m.ent_emb.cpu().numpy(), rel_emb=m.rel_emb.cpu().numpy(),
                P=m.fc_weights.projections[0].cpu().numpy(), conv=m.conv1_weights.cpu().numpy(),
                lo=m.shard.lo, hi=m.shard.hi)


def _rep_worker(rank, world, port, out_dir, prec):
    import torch.distributed as dist
    from coper_b200.models import ConvE
    from coper_b200.sharding import EntityShard
    dev = _init_dist(rank, world, port)
    try:
        cfg = O.OracleConfig(**REP_CFG)
        m = ConvE(_descr(cfg), device="cuda:%d" % dev, seed=0, shard=EntityShard(cfg.num_ent, rank, world), prec=prec)
        m.load_variables(O.init_params(cfg, seed=3, bias_noise=0.05))
        loss = float(m.train_step(_sampled_batch(cfg, B_REP)).item())
        torch.cuda.synchronize()
        np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **_snapshot(m, loss))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("prec", ["fp32", "fp16x3"])
def test_replicated_front_end_sampled_matches_single_gpu(prec, tmp_path):
    import torch.multiprocessing as mp
    from coper_b200.models import ConvE
    world = 2
    mp.spawn(_rep_worker, args=(world, _free_port(), str(tmp_path), prec), nprocs=world, join=True)
    cfg = O.OracleConfig(**REP_CFG)
    m = ConvE(_descr(cfg), device="cuda:0", seed=0, prec=prec)
    m.load_variables(O.init_params(cfg, seed=3, bias_noise=0.05))
    ref = _snapshot(m, float(m.train_step(_sampled_batch(cfg, B_REP)).item()))
    outs = [np.load(os.path.join(str(tmp_path), "rank%d.npz" % r)) for r in range(world)]

    def close(a, b, tol):
        return np.abs(a - b).max() <= tol * np.abs(b).max()
    for o in outs:
        lo, hi = int(o["lo"]), int(o["hi"])
        assert abs(float(o["loss"]) - ref["loss"]) < 2e-6 * abs(ref["loss"])
        assert abs(float(o["norm"]) - ref["norm"]) < 1e-5 * ref["norm"]
        assert close(o["dE"], ref["dE"][lo:hi], 1e-5) and close(o["dE_sq"], ref["dE_sq"][lo:hi], 1e-5)
        assert close(o["db"], ref["db"][lo:hi], 1e-5)
        # updated variables: 5e-4, as in test_gpu_multi (AMSGrad amplifies fp32 order noise on near-zero gradients)
        assert close(o["ent"], ref["ent"][lo:hi], 5e-4)
        for k in ("rel_emb", "P", "conv"):
            assert close(o[k], ref[k], 5e-4), k
    for k in ("rel_emb", "P", "conv"):
        assert np.array_equal(outs[0][k], outs[1][k]), k


def _dp_batch(cfg, device_sampling):
    B = 132
    e1, rel, e2, rowptr, col = O.synthetic_batch(cfg, B, seed=5, mean_pos=5.0)
    e1[B // 2:] = e1[:B - B // 2]                       # heads shared ACROSS the two ranks' slices
    if device_sampling:
        return {"e1": e1, "rel": rel, "e2": e2, "e2_multi_rowptr": rowptr, "e2_multi_col": col,
                "sample_on_device": (L_SAMP, 4.0)}
    b = _sampled_batch(cfg, B)
    b.update(e1=e1, rel=rel, e2=e2)
    return b


def _dp_worker(rank, world, port, out_dir, prec, device_sampling):
    import torch.distributed as dist
    from coper_b200.models import ConvE
    from coper_b200.sharding import EntityShard
    from test_gpu_model import export_masks
    dev = _init_dist(rank, world, port)
    try:
        cfg = O.OracleConfig(**DP_CFG)
        batch = _dp_batch(cfg, device_sampling)
        Bg = len(batch["e1"])
        sh = EntityShard(cfg.num_ent, rank, world)
        m = ConvE(_descr(cfg), device="cuda:%d" % dev, seed=0, shard=sh, prec=prec, data_parallel=True,
                  graphs_multi_gpu=dist.get_backend() == "nccl")
        m.load_variables(O.init_params(cfg, seed=3, bias_noise=0.05))
        loss = float(m.train_step(batch, apply_update=False).item())
        masks = export_masks(m, cfg, Bg // world)
        sb = m._bufs[Bg].samp[L_SAMP]
        res = {"loss": loss, "lo": sh.lo, "hi": sh.hi, "q": m._bufs[("dp", Bg)].q.cpu().numpy(),
               "lookup": sb.lookup.cpu().numpy(), "labels": sb.labels.cpu().numpy(),
               "seed": int(m.seed_dev.item()) - (rank << 32)}
        res.update({k.replace("/", "__"): v.cpu().numpy() for k, v in m.grads.items()})
        res.update({"mask_" + k: (np.stack(v) if isinstance(v, list) else v) for k, v in masks.items()})
        m._clip_and_apply()
        draws = []
        for _ in range(3):                              # eager, then (NCCL) capture and replay
            loss2 = float(m.train_step(batch).item())
            assert np.isfinite(loss2)
            draws.append((int(m.seed_dev.item()) - (rank << 32), sb.lookup.cpu().numpy(), sb.labels.cpu().numpy()))
        res["draw_seed"] = np.array([s for s, _, _ in draws])
        res["draw_lookup"] = np.stack([lk for _, lk, _ in draws])
        res["draw_labels"] = np.stack([lb for _, _, lb in draws])
        res["rel_emb_new"] = m.rel_emb.cpu().numpy()
        res["P_new"] = m.fc_weights.projections[-1].cpu().numpy()
        torch.cuda.synchronize()
        np.savez(os.path.join(out_dir, "dp%d.npz" % rank), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("device_sampling", [False, True])
@pytest.mark.parametrize("prec", ["fp32", "fp16x3"])
def test_data_parallel_front_end_sampled_matches_oracle(prec, device_sampling, tmp_path):
    import torch.multiprocessing as mp
    world = 2
    mp.spawn(_dp_worker, args=(world, _free_port(), str(tmp_path), prec, device_sampling), nprocs=world, join=True)
    outs = [np.load(os.path.join(str(tmp_path), "dp%d.npz" % r)) for r in range(world)]
    cfg = O.OracleConfig(**DP_CFG)
    batch = _dp_batch(cfg, device_sampling)
    e1, rel = batch["e1"], batch["rel"]
    lookup, labels = outs[0]["lookup"], outs[0]["labels"]
    for o in outs:                                      # every rank scores the same global [Bg, L]
        assert np.array_equal(o["lookup"], lookup) and np.array_equal(o["labels"], labels)
    if device_sampling:
        rowptr, col = batch["e2_multi_rowptr"], batch["e2_multi_col"]
        need = int(1.0 / (1.0 + 4.0) * L_SAMP)
        # the rank-free seed is the single-GPU model's seed of the same step
        assert int(outs[0]["seed"]) == DH.model_seed0(0) + 1
        seeds = [int(x) for x in [outs[0]["seed"]] + list(outs[0]["draw_seed"])]
        lks = [lookup] + list(outs[0]["draw_lookup"])
        lbs = [labels] + list(outs[0]["draw_labels"])
        for o in outs:
            assert [int(x) for x in o["draw_seed"]] == seeds[1:]
            assert np.array_equal(o["draw_lookup"], outs[0]["draw_lookup"])
            assert np.array_equal(o["draw_labels"], outs[0]["draw_labels"])
        for s, lk, lb in zip(seeds, lks, lbs):
            lk_ref, lb_ref = DH.sample_labels(rowptr, col, cfg.num_ent, L_SAMP, need, s)
            assert np.array_equal(lk, lk_ref) and np.array_equal(lb, lb_ref), s
        assert not np.array_equal(lks[1], lks[2])
    else:
        assert np.array_equal(lookup, batch["lookup_values"]) and np.array_equal(labels, batch["e2_multi"])
    params = O.init_params(cfg, seed=3, bias_noise=0.05)
    masks = {"feature_map": np.concatenate([o["mask_feature_map"] for o in outs], 0),
             "output": np.concatenate([o["mask_output"] for o in outs], 0)}
    for key in ("ctx_w", "ctx_b"):
        masks[key] = list(np.concatenate([o["mask_" + key] for o in outs], 1))
    out = O.forward(params, cfg, e1, rel, True, masks, labels, np.float64, lookup=lookup)
    g = O.backward(out, cfg)

    def rel_err(a, b, floor=0.0):
        return np.abs(a - b).max() / max(np.abs(b).max(), floor, 1e-30)
    assert rel_err(np.concatenate([o["q"] for o in outs], 0), out["q"]) < 1e-5
    scale = max(np.abs(g[k]).max() for k in ("ent_emb", "rel_emb", "conv1_weights"))
    for o in outs:
        lo, hi = int(o["lo"]), int(o["hi"])
        assert abs(float(o["loss"]) - out["loss"]) < 1e-6 * abs(out["loss"])
        assert rel_err(o["ent_emb"], g["ent_emb"][lo:hi]) < 2e-4
        assert rel_err(o["pred_bias"], g["pred_bias"][lo:hi]) < 2e-4
        assert rel_err(o["rel_emb"].reshape(g["rel_emb"].shape), g["rel_emb"]) < 2e-4
        assert rel_err(o["conv1_weights"].reshape(g["conv1_weights"].shape), g["conv1_weights"]) < 2e-4
        for nm in ("FCBN", "Conv1BN"):
            for k in ("gamma", "beta"):
                assert rel_err(o["%s__%s" % (nm, k)], g[nm][k], 1e-4 * scale) < 2e-4, (nm, k)
        for i in range(len(g["fc_weights_proj"])):
            assert rel_err(o["fc_weights__CPG__Projection%d" % i].reshape(g["fc_weights_proj"][i].shape),
                           g["fc_weights_proj"][i], 1e-4 * scale) < 2e-4
    assert np.array_equal(outs[0]["rel_emb_new"], outs[1]["rel_emb_new"])
    assert np.array_equal(outs[0]["P_new"], outs[1]["P_new"])


# ------------------------------------------------------------------------------------------------ entry point
def _write_dataset(path, n_ent=400, n_trip=3000, seed=0):
    rng = np.random.default_rng(seed)
    rows = sorted({("e%d" % rng.integers(n_ent), "r%d" % rng.integers(4), "e%d" % rng.integers(n_ent))
                   for _ in range(n_trip)})
    os.makedirs(path, exist_ok=True)
    for fn, part in (("train.txt", rows[:-80]), ("dev.txt", rows[-80:-40]), ("test.txt", rows[-40:])):
        with open(os.path.join(path, fn), "w") as fh:
            for r in part:
                fh.write("\t".join(r) + "\n")


@pytest.mark.parametrize("mode", ["device_sampling", "one_positive"])
def test_run_cpg_sampled_under_torchrun(mode, tmp_path):
    """The shipped default (num_labels set) trains and evaluates on two ranks without --full-1n."""
    from coper_b200 import configs
    data_dir = os.path.join(str(tmp_path), "data")
    _write_dataset(data_dir)
    cfg = configs.load_config("WN18RR", "cpg")
    cfg.model.entity_embedding_size, cfg.model.relation_embedding_size = 40, 8
    cfg.training.update(batch_size=16, num_labels=24, prop_negatives=3.0, max_steps=6,
                        one_positive_label_per_sample=mode == "one_positive")
    cfg.eval.update(log_steps=2, eval_steps=5)
    cfg_path = os.path.join(str(tmp_path), "cfg.yaml")
    with open(cfg_path, "w") as fh:
        yaml.safe_dump(_plain(cfg), fh)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), "-m", "coper_b200.run_cpg",
           "--dataset", "countries_S1", "--data-dir", data_dir, "--config", cfg_path,
           "--working-dir", os.path.join(str(tmp_path), "work"), "--eval-batches", "2", "--prec", "fp16x3"]
    if mode == "device_sampling":
        cmd.append("--device-sampling")
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, _first_traceback(out.stderr)
    assert "num_labels_24" in out.stderr and "MRR" in out.stderr
    losses = [float(line.split("Loss:")[1]) for line in out.stderr.splitlines() if "| Loss:" in line]
    assert len(losses) == 3 and all(np.isfinite(losses))


def _first_traceback(err):
    lines = err.splitlines()
    i = next((k for k, line in enumerate(lines) if "Traceback" in line), max(0, len(lines) - 60))
    return "\n".join(lines[i:i + 60])


def _plain(d):
    return {k: _plain(v) if isinstance(v, dict) else v for k, v in d.items()}
