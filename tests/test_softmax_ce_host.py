"""CPU tests of the softmax cross-entropy objective: the fp64 reference against torch autograd, the full oracle backward
with this loss, the sharded log-sum-exp exchange over gloo and run_cpg's argument handling.  (No GPU.)"""
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import conve_oracle as O
from oracle.torch_port import TorchPort
from softmax_ce_reference import ce_loss_grad, oracle_ce_step, targets


def _rows(B, N, rng):
    """CSR positives with rows of 0, 1 and many positives."""
    rowptr, col = [0], []
    for b in range(B):
        k = (0, 1, 7)[b % 3]
        col += list(rng.choice(N, size=k, replace=False))
        rowptr.append(len(col))
    return np.asarray(rowptr, np.int64), np.asarray(col, np.int64)


@pytest.mark.parametrize("eps", [0.0, 0.1])
@pytest.mark.parametrize("scale", [1.0, 1e3])
def test_reference_equals_autograd(eps, scale):
    rng = np.random.default_rng(3)
    B, N = 9, 37
    S = rng.normal(size=(B, N)) * scale
    rowptr, col = _rows(B, N, rng)
    loss, G, lse = ce_loss_grad(S, rowptr, col, eps)
    St = torch.tensor(S, dtype=torch.float64, requires_grad=True)
    T = torch.tensor(targets(rowptr, col, N, eps))
    L = -(T * torch.log_softmax(St, dim=1)).sum() / B
    L.backward()
    assert np.isfinite(loss) and np.isfinite(G).all()
    assert abs(loss - L.item()) <= 1e-12 * max(1.0, abs(L.item()))
    assert np.abs(G - St.grad.numpy()).max() <= 1e-12
    assert np.allclose(lse, torch.logsumexp(St.detach(), 1).numpy(), rtol=1e-14, atol=0)
    # a row without positives and eps = 0 contributes nothing; with eps > 0 its target is uniform eps / N
    assert np.all(G[0] == 0) if eps == 0.0 else abs(G[0].sum()) < 1e-14


class _CePort(TorchPort):
    """The literal torch port with the softmax cross-entropy in place of the BCE (labels = target matrix)."""

    def loss(self, S, T):
        return -(torch.as_tensor(T, dtype=self.dtype) * torch.log_softmax(S, dim=1)).sum() / S.shape[0]


@pytest.mark.parametrize("ctx,conv", [([], None), ([6], None)])      # (the torch port has no generated conv)
def test_oracle_backward_with_ce_matches_autograd(ctx, conv):
    cfg = O.OracleConfig(num_ent=97, num_rel=6, ent_emb_size=40, rel_emb_size=5, context_rel_out=ctx,
                         context_rel_conv=conv, label_smoothing_epsilon=0.1, batch_norm_train_stats=True,
                         batch_norm_momentum=0.9)
    p = O.init_params(cfg, 1, bias_noise=0.1)
    B = 7
    e1, rel, e2, rowptr, col = O.synthetic_batch(cfg, B, 3)
    loss, g, _ = oracle_ce_step(O, p, cfg, e1, rel, rowptr, col)
    L, tg = _CePort(p, cfg, torch.float64).loss_and_grads(e1, rel, targets(rowptr, col, cfg.num_ent, 0.1), True, None)
    rel_err = lambda a, b: np.abs(a - b).max() / (np.abs(b).max() + 1e-6)
    assert abs(loss - L) < 1e-12
    for nm in ("ent_emb", "rel_emb", "pred_bias"):
        assert rel_err(g[nm], tg[nm]) < 1e-9, nm
    for i, a in enumerate(g["fc_weights_proj"]):
        assert rel_err(a, tg["fc_weights_proj.%d" % i]) < 1e-9
    for nm in ("FCBN", "Conv1BN"):
        assert rel_err(g[nm]["gamma"], tg[nm + ".gamma"]) < 1e-9


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _combine_worker(rank, world, port, S, bounds, q):
    import torch.distributed as dist
    from coper_b200 import sharding
    dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    lo, hi = bounds[rank], bounds[rank + 1]
    s = torch.tensor(S[:, lo:hi], dtype=torch.float32)
    m = s.max(1).values
    ml = torch.stack([m, torch.exp(s - m[:, None]).sum(1)], 1)
    parts = sharding.combine_lse(ml, world, None)
    # coper_lse_finalize's fixed-order combine, restated on the host
    p64 = parts.double()
    M = p64[:, :, 0].max(0).values
    lse = (M + torch.log((p64[:, :, 1] * torch.exp(p64[:, :, 0] - M)).sum(0))).float()
    q.put((rank, parts.numpy().tobytes(), lse.numpy()))
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_combine_lse_gloo(world):
    rng = np.random.default_rng(world)
    B, N = 5, 301
    S = rng.normal(size=(B, N)) * 4
    bounds = [0, 128, 256, N] if world == 3 else [0, 256, N]          # uneven shards
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_combine_worker, args=(r, world, port, S, bounds, q)) for r in range(world)]
    for pr in procs:
        pr.start()
    res = sorted(q.get(timeout=120) for _ in range(world))
    for pr in procs:
        pr.join(60)
        assert pr.exitcode == 0
    ref = torch.logsumexp(torch.tensor(S), 1).numpy()
    for _, raw, lse in res:
        assert raw == res[0][1]                                         # every rank holds the same pairs
        assert np.array_equal(lse, res[0][2])
        assert np.abs(lse - ref).max() <= 1e-6 * np.abs(ref).max()


def test_run_cpg_rejects_ce_on_sampled_config(capsys):
    from coper_b200 import run_cpg
    with pytest.raises(SystemExit):
        run_cpg.main(["--dataset", "FB15k-237", "--loss", "softmax_ce"])
    assert "--full-1n" in capsys.readouterr().err


def test_model_name_unchanged_for_bce():
    from coper_b200 import configs
    from coper_b200.run_cpg import model_name_of
    cfg = configs.load_config("WN18RR", "cpg")
    name = model_name_of(cfg, "cpg", "WN18RR", True, False)
    assert "loss" not in name
    cfg.model.loss = "softmax_ce"
    assert model_name_of(cfg, "cpg", "WN18RR", True, False) == name + "-loss_softmax_ce"
    md = configs.model_descriptors(configs.load_config("WN18RR", "cpg"), 10, 2)
    assert md["loss"] == "bce"
