"""Softmax cross-entropy over all entities on the GPU: the C entry points (log-sum-exp pass, finalize, CE scorer
gradient) against fp64 for every engine, sharded row ranges, and ConvE(loss="softmax_ce") training steps."""
import numpy as np
import pytest
import torch


pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _release_models():
    """Free this test's models (and their captured CUDA graphs) before the next test runs: a graph destroyed by a later
    garbage collection in the middle of another test's stream capture would invalidate that capture."""
    yield
    import gc
    gc.collect()
    torch.cuda.synchronize()

PREC = {"fp32": 0, "bf16": 1, "tf32x3": 2, "fp16x3": 3}


def _bf16(x):
    return x.to(torch.bfloat16).to(torch.float64)


def _relerr(a, b):
    return ((a.double() - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


class _Case:
    """q, E, bias and CSR positives (rows of 0, 1 and several positives) on the device, and the fp64 reference."""

    def __init__(self, B, N, d, prec, scale=1.0, seed=0, eps=0.1):
        g = torch.Generator(device="cuda").manual_seed(seed + B + N + d)
        self.B, self.N, self.d, self.prec, self.eps = B, N, d, prec, eps
        self.q = (torch.rand(B, d, device="cuda", generator=g) * 2 - 1) * (scale / d ** 0.5)
        self.E = torch.rand(N, d, device="cuda", generator=g) * 2 - 1
        self.bias = torch.randn(N, device="cuda", generator=g) * 0.1
        k = torch.tensor([(1, 0, 1, 5)[b % 4] for b in range(B)])
        self.rowptr = torch.zeros(B + 1, dtype=torch.int32)
        self.rowptr[1:] = torch.cumsum(k, 0)
        self.col = torch.cat([torch.randperm(N)[:int(n)] for n in k]).to(torch.int32)
        self.rowptr, self.col = self.rowptr.cuda(), self.col.cuda()
        cast = _bf16 if prec == "bf16" else (lambda x: x.double())
        S = cast(self.q) @ cast(self.E).T + self.bias.double()
        self.lse_ref = torch.logsumexp(S, 1)
        T = torch.full((B, N), eps / N, dtype=torch.float64, device="cuda")
        rp = self.rowptr.cpu().numpy()
        for b in range(B):
            ids = self.col[rp[b]:rp[b + 1]].long()
            T[b, ids] += (1 - eps) / max(rp[b + 1] - rp[b], 1)
        tau = T.sum(1)
        self.loss_ref = ((T * (self.lse_ref[:, None] - S)).sum() / B).item()
        G = (tau[:, None] * torch.exp(S - self.lse_ref[:, None]) - T) / B
        self.G_ref = G
        self.dq_ref, self.dE_ref, self.db_ref = G @ cast(self.E), G.T @ cast(self.q), G.sum(0)


def _bits(L, c, lo, hi):
    if PREC[c.prec] == 0:
        bits = torch.zeros(c.B, -(-(hi - lo) // 32), dtype=torch.int32, device="cuda")
        L.call("coper_csr_to_bits", L.ptr(c.rowptr), L.ptr(c.col), c.B, lo, hi, L.ptr(bits))
    else:
        bits = torch.zeros(max(hi - lo, 1), -(-c.B // 32), dtype=torch.int32, device="cuda")
        L.call("coper_csr_to_bits_t", L.ptr(c.rowptr), L.ptr(c.col), c.B, lo, hi, L.ptr(bits))
    return bits


def _lse_ml(L, c, lo, hi):
    lib, p = L.load(), PREC[c.prec]
    Ns = hi - lo
    ws = torch.empty(lib.coper_score1n_lse_workspace_bytes(c.B, Ns, c.d, p), dtype=torch.uint8, device="cuda")
    ml = torch.full((c.B, 2), float("nan"), device="cuda")
    L.call("coper_score1n_lse", L.ptr(c.q), L.ptr(c.E[lo:hi]), None, L.ptr(c.bias[lo:hi]), c.B, Ns, c.d, L.ptr(ml),
           L.ptr(ws), ws.numel(), p)
    return ml


def _finalize(L, parts):
    lse = torch.full((parts.shape[1],), float("nan"), device="cuda")
    L.call("coper_lse_finalize", L.ptr(parts.contiguous()), parts.shape[0], parts.shape[1], L.ptr(lse))
    return lse


def _ce(L, c, lse, lo, hi, mode="full"):
    """mode: full | norm | split (dE == NULL, then coper_score1n_bce_dE)."""
    lib, p = L.load(), PREC[c.prec]
    B, Ns, d = c.B, hi - lo, c.d
    ws = torch.empty(lib.coper_score1n_bce_workspace_bytes(B, Ns, d, p), dtype=torch.uint8, device="cuda")
    G = torch.empty(lib.coper_score1n_bce_G_bytes(B, Ns, p), dtype=torch.uint8, device="cuda")
    ld = -(-Ns // 32) * 32
    loss = torch.zeros(1, dtype=torch.float64, device="cuda")
    ss = torch.zeros(1, dtype=torch.float64, device="cuda")
    nan = float("nan")
    dq, dE, db = (torch.full(s, nan, device="cuda") for s in ((B, d), (Ns, d), (Ns,)))
    args = (L.ptr(c.q), L.ptr(c.E[lo:hi]), None, L.ptr(c.bias[lo:hi]), L.ptr(_bits(L, c, lo, hi)), L.ptr(c.rowptr),
            L.ptr(lse), B, Ns, d, c.N, c.eps, 1.0 / B, L.ptr(loss), L.ptr(G), ld, L.ptr(dq))
    if mode == "full":
        L.call("coper_score1n_ce_fwd_bwd", *args, L.ptr(dE), L.ptr(db), L.ptr(ws), ws.numel(), p)
    elif mode == "norm":
        L.call("coper_score1n_ce_fwd_bwd_norm", *args, L.ptr(dE), L.ptr(db), L.ptr(ss), L.ptr(ws), ws.numel(), p)
    else:
        L.call("coper_score1n_ce_fwd_bwd_norm", *args, None, L.ptr(db), L.ptr(ss), L.ptr(ws), ws.numel(), p)
        L.call("coper_score1n_bce_dE", L.ptr(G), B, Ns, d, lib.coper_score1n_ce_dE_inv_count(1.0 / B, c.N, p), L.ptr(dE),
               L.ptr(ss), L.ptr(db), L.ptr(ws), ws.numel(), p)
    torch.cuda.synchronize()
    return loss.item(), dq, dE, db, ss.item()


SHAPES = [(1, 1, 8), (7, 97, 40), (33, 1000, 200), (512, 40943, 200), (4096, 100003, 256)]


@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "fp16x3", "bf16"])
@pytest.mark.parametrize("B,N,d", SHAPES)
def test_ce_entry_points_match_fp64(prec, B, N, d):
    from coper_b200 import _lib as L
    if prec == "fp32" and B * N > 1 << 27:
        pytest.skip("fp32 engine: [B, N] G of this shape is covered by the tensor-pipe engines")
    c = _Case(B, N, d, prec, scale=3.0)
    ml = _lse_ml(L, c, 0, N)
    lse = _finalize(L, ml.unsqueeze(0))
    fp32_class = prec != "bf16"
    assert _relerr(lse, c.lse_ref) < (1e-6 if fp32_class else 1e-5)
    loss, dq, dE, db, _ = _ce(L, c, lse, 0, N)
    assert abs(loss / B - c.loss_ref) <= (1e-5 if fp32_class else 1e-4) * abs(c.loss_ref)
    gt = 1e-5 if fp32_class else 2e-2
    assert _relerr(dq, c.dq_ref) < gt
    assert _relerr(dE, c.dE_ref) < (2e-4 if fp32_class else 2e-2)
    assert _relerr(db, c.db_ref) < gt
    # determinism: a second call is bit-identical
    ml2 = _lse_ml(L, c, 0, N)
    assert torch.equal(ml, ml2)
    loss2, dq2, dE2, db2, _ = _ce(L, c, lse, 0, N)
    assert loss2 == loss and torch.equal(dq, dq2) and torch.equal(dE, dE2) and torch.equal(db, db2)
    if prec != "fp32":              # the _norm form and the split form equal the unsplit call bitwise
        for mode in ("norm", "split"):
            l3, dq3, dE3, db3, ss = _ce(L, c, lse, 0, N, mode)
            assert l3 == loss and torch.equal(dq, dq3) and torch.equal(dE, dE3) and torch.equal(db, db3), mode
            assert abs(ss - (dE.double() ** 2).sum().item()) <= 1e-6 * ss


@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "fp16x3", "bf16"])
def test_ce_large_logits(prec):
    """|s| ~ 80: exp(s) overflows fp32, the two-pass normaliser does not."""
    from coper_b200 import _lib as L
    c = _Case(64, 3001, 64, prec, scale=240.0)          # logits of standard deviation ~80
    lse = _finalize(L, _lse_ml(L, c, 0, c.N).unsqueeze(0))
    assert c.lse_ref.abs().max() > 40
    assert _relerr(lse, c.lse_ref) < (1e-6 if prec != "bf16" else 1e-5)
    loss, dq, dE, db, _ = _ce(L, c, lse, 0, c.N)
    assert np.isfinite(loss) and torch.isfinite(dq).all() and torch.isfinite(dE).all()
    assert abs(loss / c.B - c.loss_ref) <= (1e-5 if prec != "bf16" else 1e-3) * abs(c.loss_ref)
    assert _relerr(dq, c.dq_ref) < (1e-5 if prec != "bf16" else 2e-2)


def test_ce_fp16x3_gradient_scale_at_a_million_entities():
    """Most CE gradient entries are ~1/N: the fp16x3 planes carry them scaled by a power of two chosen from N."""
    from coper_b200 import _lib as L
    N = (1 << 20) + 77
    c = _Case(33, N, 64, "fp16x3")
    lse = _finalize(L, _lse_ml(L, c, 0, N).unsqueeze(0))
    assert _relerr(lse, c.lse_ref) < 1e-6
    loss, dq, dE, db, _ = _ce(L, c, lse, 0, N)
    assert abs(loss / c.B - c.loss_ref) <= 1e-5 * abs(c.loss_ref)
    assert _relerr(dq, c.dq_ref) < 1e-5
    assert _relerr(dE, c.dE_ref) < 2e-4
    assert _relerr(db, c.db_ref) < 1e-5


@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "fp16x3", "bf16"])
@pytest.mark.parametrize("ways", [2, 3])
def test_ce_row_ranges_reproduce_unsharded(prec, ways):
    from coper_b200 import _lib as L
    from coper_b200.sharding import EntityShard
    B, N, d = 97, 5003, 72
    c = _Case(B, N, d, prec)
    lse_full = _finalize(L, _lse_ml(L, c, 0, N).unsqueeze(0))
    loss_full, dq_full, dE_full, _, _ = _ce(L, c, lse_full, 0, N)
    shards = [EntityShard(N, r, ways) for r in range(ways)]
    parts = torch.stack([_lse_ml(L, c, s.lo, s.hi) for s in shards])
    lse = _finalize(L, parts)
    assert _relerr(lse, lse_full.double()) < 1e-6
    loss, dq = 0.0, torch.zeros(B, d, dtype=torch.float64, device="cuda")
    for s in shards:
        l, dqs, dEs, _, _ = _ce(L, c, lse, s.lo, s.hi)
        loss += l
        dq += dqs.double()
        assert _relerr(dEs, dE_full[s.lo:s.hi].double()) < (1e-5 if prec != "bf16" else 1e-2)
    assert abs(loss - loss_full) <= 1e-6 * abs(loss_full)
    assert _relerr(dq, dq_full.double()) < (1e-5 if prec != "bf16" else 1e-2)


# ---------------------------------------------------------------------------------------------------------- ConvE
def _md(cfg, B, **kw):
    md = {"use_negative_sampling": False, "label_smoothing_epsilon": cfg.label_smoothing_epsilon,
          "num_ent": cfg.num_ent, "num_rel": cfg.num_rel, "ent_emb_size": cfg.ent_emb_size,
          "rel_emb_size": cfg.rel_emb_size, "concat_rel": False, "context_rel_conv": cfg.context_rel_conv,
          "context_rel_out": cfg.context_rel_out, "context_rel_dropout": 0.0, "context_rel_use_batch_norm": False,
          "input_dropout": 0.0, "hidden_dropout": 0.0, "output_dropout": 0.0, "learning_rate": 1e-3,
          "batch_size": B, "batch_norm_momentum": 0.9, "batch_norm_train_stats": True,
          "do_parameter_lookup": False, "loss": "softmax_ce"}
    md.update(kw)
    return md


def _one_positive_batch(O, cfg, B, seed):
    e1, rel, e2, _, _ = O.synthetic_batch(cfg, B, seed)
    rowptr = np.arange(B + 1, dtype=np.int64)
    return e1, rel, e2, rowptr, np.asarray(e2, np.int64)


@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "fp16x3", "bf16"])
@pytest.mark.parametrize("variant", ["g_linear", "g_mlp", "gen_conv"])
@pytest.mark.parametrize("B", [4096, 4097])
def test_conve_ce_step_matches_oracle(prec, variant, B):
    """One CE training step (gradients only, one positive per row) against the oracle's CE step: the loss, dbias and
    the relation gradient (which depends on dq through the whole front-end backward).  The entity gradient is the
    scorer's dE plus the scatter of the front end's d x0; the scorer's share is checked against fp64 on the model's own
    q (the front end's fp32 d x0 differs from the fp64 oracle's by ~1e-6 absolute at this batch size, independent of
    the loss)."""
    from oracle import conve_oracle as O
    from softmax_ce_reference import ce_loss_grad, oracle_ce_step
    from coper_b200.models import ConvE
    ctx = {"g_linear": dict(context_rel_out=[]), "g_mlp": dict(context_rel_out=[8]),
           "gen_conv": dict(context_rel_out=[8], context_rel_conv=[4])}[variant]
    cfg = O.OracleConfig(num_ent=3001, num_rel=7, ent_emb_size=40, rel_emb_size=5, batch_norm_train_stats=True,
                         batch_norm_momentum=0.9, label_smoothing_epsilon=0.1, **ctx)
    params = O.init_params(cfg, seed=2, bias_noise=0.05)
    e1, rel, e2, rowptr, col = _one_positive_batch(O, cfg, B, 5)
    loss_ref, g_ref, _ = oracle_ce_step(O, params, cfg, e1, rel, rowptr, col)
    m = ConvE(_md(cfg, B), device="cuda:0", prec=prec)
    m.load_variables(params)
    batch = {"e1": e1, "rel": rel, "e2": e2, "e2_multi_rowptr": rowptr, "e2_multi_col": col}
    loss = float(m.train_step(batch, apply_update=False).item())
    fp32_class = prec != "bf16"
    assert abs(loss - loss_ref) <= (1e-5 if fp32_class else 2e-3) * abs(loss_ref)
    assert _relerr(m.grads["pred_bias"], torch.as_tensor(g_ref["pred_bias"]).cuda()) < (1e-4 if fp32_class else 3e-2)
    g_rel = torch.as_tensor(g_ref["rel_emb"]).cuda()
    if fp32_class:
        assert _relerr(m.grads["rel_emb"], g_rel) < 1e-4
    else:
        # bf16: the rounded forward flips the few FC ReLU units whose pre-activation lies within rounding of zero, and
        # batch-stat BN amplifies those elements in the backward (test_gpu_model.py): a direction check, as there
        cos = torch.nn.functional.cosine_similarity(m.grads["rel_emb"].double().flatten(), g_rel.flatten(), dim=0)
        assert cos.item() > 0.99
    slot = m._bufs[B]
    q = slot.q.double()
    E = torch.as_tensor(params["ent_emb"], dtype=torch.float64).cuda()
    bias = torch.as_tensor(params["pred_bias"], dtype=torch.float64).cuda()
    if not fp32_class:
        q, E = _bf16(q), _bf16(E)
    _, G, _ = ce_loss_grad((q @ E.T + bias).cpu().numpy(), rowptr, col, cfg.label_smoothing_epsilon)
    ref = torch.as_tensor(G).cuda().T @ q
    ref.index_add_(0, torch.as_tensor(np.asarray(e1)).cuda(), slot.dx0.double())
    assert _relerr(m.grads["ent_emb"], ref) < (1e-4 if fp32_class else 3e-2)


@pytest.mark.parametrize("prec", ["tf32x3", "bf16"])
def test_conve_ce_graph_replay_equals_eager(prec):
    """Captured and replayed CE steps follow the eager model step for step, and the loss falls."""
    from oracle import conve_oracle as O
    from coper_b200.models import ConvE
    cfg = O.OracleConfig(num_ent=997, num_rel=6, ent_emb_size=40, rel_emb_size=5, context_rel_out=[],
                         batch_norm_train_stats=True, batch_norm_momentum=0.9, label_smoothing_epsilon=0.1)
    params = O.init_params(cfg, seed=1, bias_noise=0.05)
    B = 64
    e1, rel, e2, rowptr, col = O.synthetic_batch(cfg, B, seed=2)
    batch = {"e1": e1, "rel": rel, "e2": e2, "e2_multi_rowptr": rowptr, "e2_multi_col": col}
    runs = []
    for graphs in (False, True):
        m = ConvE(_md(cfg, B), device="cuda:0", prec=prec, use_graphs=graphs)
        m.load_variables(params)
        runs.append(([float(m.train_step(batch).item()) for _ in range(6)], m.ent_emb.clone()))
    (l0, E0), (l1, E1) = runs
    assert l0 == l1 and torch.equal(E0, E1)
    assert l0[-1] < l0[0]


def test_conve_ce_rejects_sampled_labels():
    from oracle import conve_oracle as O
    from coper_b200.models import ConvE
    cfg = O.OracleConfig(num_ent=97, num_rel=6, ent_emb_size=40, rel_emb_size=5, context_rel_out=[])
    with pytest.raises(NotImplementedError, match="full-1n"):
        ConvE(_md(cfg, 8, use_negative_sampling=True), device="cuda:0")


# ---------------------------------------------------------------------------------------------------------------
# Whole training steps with the update, every model type: gradients and clip norm against the oracle's CE step at the
# pre-step parameters and dropout masks, theta against fp64 AMSGrad of the model's own gradients and clip factor (the
# bars of test_gpu_model.py / test_gpu_update.py).  Step 0 runs eager, step 1 is captured and replayed.
CE_UPDATE_CASES = ["toy_glinear_dropout", "toy_gmlp_bn_dropout", "cpgconv_glinear", "plain_toy", "lookup_toy"]


@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "fp16x3", "bf16"])
@pytest.mark.parametrize("name", CE_UPDATE_CASES)
def test_conve_ce_update_matches_oracle(name, prec):
    import coper_b200.models as M
    from oracle import conve_oracle as O
    from softmax_ce_reference import oracle_ce_step
    from test_gpu_model import CASES, batch_of, compare_grads, descriptors, export_masks
    from test_gpu_update import amsgrad_ref, close_to_max, host, oracle_clip, params_of
    kw, B = CASES[name]
    cfg = O.OracleConfig(label_smoothing_epsilon=0.1, **kw)
    params = O.init_params(cfg, seed=3, bias_noise=0.05)
    model = M.ConvE(dict(descriptors(cfg, 1e-3), loss="softmax_ce"), conv_in_height=cfg.conv_in_height, prec=prec)
    model.load_variables(params)
    fp32_class = prec != "bf16"
    for step in range(2):
        e1, rel, e2, rowptr, col = O.synthetic_batch(cfg, B, seed=60 + step)
        e1[B // 2:] = e1[:B - B // 2]                   # duplicate heads: the scatter's segments
        pre = {n: {"theta": host(p), "vhat": host(model.vhat[n]),
                   "m": host(model.m[n]) if n in model.m else None, "v": host(model.v[n]) if n in model.v else None}
               for n, p, _ in model.trainables}
        pre_params = params_of(model, params)
        loss = float(model.train_step(batch_of(e1, rel, e2, rowptr, col)).item())
        torch.cuda.synchronize()
        cs, norm_dev = (float(x) for x in model.clip_out.cpu().numpy())
        lr_t = float(model.step_state[0].item())
        masks = export_masks(model, cfg, B)
        loss_ref, g, _ = oracle_ce_step(O, pre_params, cfg, e1, rel, rowptr, col, masks)
        assert abs(loss - loss_ref) <= (1e-5 if fp32_class else 2e-3) * abs(loss_ref), (step, loss, loss_ref)
        norm_ref = oracle_clip(model, g, M.CLIP_NORM)[2]
        assert abs(norm_dev - norm_ref) <= (1e-4 if fp32_class else 5e-2) * norm_ref, (step, norm_dev, norm_ref)
        if fp32_class:
            compare_grads(model, g, cfg)
        else:
            assert _relerr(model.grads["pred_bias"], torch.as_tensor(g["pred_bias"]).cuda()) < 5e-2
        for n, p, _ in model.trainables:
            gsq = host(model.grad_sq[n]) if n in model.sparse_vars else None
            th, m, v, vhat = amsgrad_ref(pre[n], host(model.grads[n]), gsq, cs, lr_t, model.bug_compat)
            assert np.abs(host(p) - th).max() <= 2.0 ** -21 * np.abs(th).max() + 1e-5 * lr_t, (step, n)
            assert close_to_max(host(model.vhat[n]), vhat, 1e-6), (step, n)


# ---------------------------------------------------------------------------------------------------------------
# Entity-sharded CE steps in two processes (tests/test_gpu_multi.py: NCCL with one GPU per rank, else two processes on
# cuda:0 over gloo), under the replicated and the data-parallel front end: the per-rank log-sum-exp pairs are exchanged
# (sharding.combine_lse) and every rank finalises the same lse.  A CE step must equal the single-GPU CE step and the
# replicated variables must stay bit-identical across ranks.  No dropout: every run draws the same (no) masks.
CE_MULTI_CFG = dict(num_ent=1003, num_rel=22, ent_emb_size=200, rel_emb_size=8, context_rel_out=[12],
                    context_rel_use_batch_norm=True, batch_norm_train_stats=True, batch_norm_momentum=0.1,
                    label_smoothing_epsilon=0.1)
CE_MULTI_B = 132


def _ce_multi_run(model, rank_rows):
    """One gradient-only step and its update, then three full steps (eager, capture + replay, replay when graphed)."""
    from oracle import conve_oracle as O
    cfg = O.OracleConfig(**CE_MULTI_CFG)
    e1, rel, e2, rowptr, col = O.synthetic_batch(cfg, CE_MULTI_B, seed=5, mean_pos=5.0)
    e1[CE_MULTI_B // 2:] = e1[:CE_MULTI_B - CE_MULTI_B // 2]
    batch = {"e1": e1, "rel": rel, "e2": e2, "e2_multi_rowptr": rowptr, "e2_multi_col": col}
    lo, hi = rank_rows
    host = lambda t: t.detach().cpu().numpy().copy()
    last_w = model._last_w_name
    out = {"loss0": float(model.train_step(batch, apply_update=False).item())}
    for n in ("ent_emb", "pred_bias"):
        out["g_" + n] = host(model.grads[n])
    for n in ("rel_emb", last_w, "conv1_weights"):
        out["g_" + n.replace("/", "__")] = host(model.grads[n])
    model._clip_and_apply()
    out["norm"] = float(model.clip_out[1].item())
    # theta after the update of the compared gradients (AMSGrad as written steps every element by ~lr: later steps
    # would turn round-off sign flips of near-zero gradients into full-size differences)
    out["ent_emb"], out["pred_bias"] = host(model.ent_emb), host(model.pred_bias)
    out["rel_emb"], out["P"], out["conv1_weights"] = (host(model.rel_emb), host(model.fc_weights.projections[-1]),
                                                      host(model.conv1_weights))
    out["losses"] = np.array([float(model.train_step(batch).item()) for _ in range(3)])
    torch.cuda.synchronize()
    for n in ("rel_emb", "P", "conv1_weights"):
        out[n + "_end"] = host(model.rel_emb if n == "rel_emb" else model.conv1_weights if n == "conv1_weights"
                               else model.fc_weights.projections[-1])
    out["lo"], out["hi"] = lo, hi
    return out


def _ce_multi_worker(rank, world, port, out_dir, prec, dp, graphs):
    import os
    import torch.distributed as dist
    from oracle import conve_oracle as O
    from coper_b200.models import ConvE
    from coper_b200.sharding import EntityShard
    from test_gpu_model import descriptors
    from test_gpu_multi import _init_dist
    dev = _init_dist(rank, world, port)
    try:
        cfg = O.OracleConfig(**CE_MULTI_CFG)
        params = O.init_params(cfg, seed=3, bias_noise=0.05)
        sh = EntityShard(cfg.num_ent, rank, world)
        m = ConvE(dict(descriptors(cfg, 1e-2), loss="softmax_ce"), device="cuda:%d" % dev, seed=0, shard=sh,
                  prec=prec, data_parallel=dp, use_graphs=graphs, graphs_multi_gpu=graphs)
        m.load_variables(params)
        np.savez(os.path.join(out_dir, "ce%d.npz" % rank), **_ce_multi_run(m, (sh.lo, sh.hi)))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("prec,dp", [("fp32", False), ("fp16x3", False), ("bf16", False), ("fp32", True),
                                     ("fp16x3", True)])
@pytest.mark.parametrize("graphs", [False, True])
def test_ce_sharded_steps_match_single_gpu(prec, dp, graphs, tmp_path):
    import os
    import torch.multiprocessing as mp
    from oracle import conve_oracle as O
    from coper_b200.models import ConvE
    from test_gpu_model import descriptors
    from test_gpu_multi import _free_port
    world = 2
    if graphs and torch.cuda.device_count() < world:
        pytest.skip("captured sharded steps need NCCL, one GPU per rank (the gloo exchange stages through the host)")
    mp.spawn(_ce_multi_worker, args=(world, _free_port(), str(tmp_path), prec, dp, graphs), nprocs=world, join=True)
    cfg = O.OracleConfig(**CE_MULTI_CFG)
    params = O.init_params(cfg, seed=3, bias_noise=0.05)
    m = ConvE(dict(descriptors(cfg, 1e-2), loss="softmax_ce"), device="cuda:0", seed=0, prec=prec)
    m.load_variables(params)
    ref = _ce_multi_run(m, (0, cfg.num_ent))
    outs = [dict(np.load(os.path.join(str(tmp_path), "ce%d.npz" % r))) for r in range(world)]
    fp32_class = prec != "bf16"
    close = lambda a, b, tol: np.abs(a - b).max() <= tol * np.abs(b).max()
    for o in outs:
        lo, hi = int(o["lo"]), int(o["hi"])
        assert abs(float(o["loss0"]) - ref["loss0"]) <= (1e-5 if fp32_class else 2e-3) * abs(ref["loss0"])
        assert np.all(np.abs(o["losses"] - ref["losses"]) <= (1e-4 if fp32_class else 5e-3) * np.abs(ref["losses"]))
        assert abs(float(o["norm"]) - ref["norm"]) <= (1e-5 if fp32_class else 1e-2) * ref["norm"]
        gt = (1e-4 if dp else 1e-5) if fp32_class else 1e-2
        for n in ("ent_emb", "pred_bias"):
            assert close(o["g_" + n], ref["g_" + n][lo:hi], gt), n
        for n in [k for k in ref if k.startswith("g_") and k not in ("g_ent_emb", "g_pred_bias")]:
            assert close(o[n], ref[n], gt), n
        if fp32_class:
            # AMSGrad as written steps every element by ~lr g / |g|: an element whose gradient is round-off (its sign
            # set by summation order) moves by a full step either way, so theta is compared where the gradient is
            # not (|g| >= 1e-4 max|g|: at least 90 % of the elements), at 5e-4 as in test_gpu_multi.py
            for n, gn, rows in (("ent_emb", "g_ent_emb", slice(lo, hi)), ("rel_emb", "g_rel_emb", slice(None)),
                                ("P", next(k for k in ref if k.startswith("g_fc_weights")), slice(None)),
                                ("conv1_weights", "g_conv1_weights", slice(None))):
                gref = ref[gn][rows].reshape(ref[n][rows].shape)
                sure = np.abs(gref) >= 1e-4 * np.abs(gref).max()
                assert sure.mean() >= 0.9, n
                assert np.abs(o[n] - ref[n][rows])[sure].max() <= 5e-4 * np.abs(ref[n][rows]).max(), n
    for n in ("rel_emb", "P", "conv1_weights"):     # replicated variables: bit-identical on every rank, every step
        assert np.array_equal(outs[0][n], outs[1][n]) and np.array_equal(outs[0][n + "_end"], outs[1][n + "_end"]), n
    assert np.array_equal(outs[0]["losses"], outs[1]["losses"])
