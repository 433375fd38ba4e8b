"""fp64 reference of the softmax cross-entropy over all entities (include/coper.h):

    t_bn  = (1-eps) [n in P_b] / max(n_b, 1) + eps / N
    lse_b = log sum_n exp(s_bn)
    loss  = (1/B) sum_b sum_n t_bn (lse_b - s_bn)
    G_bn  = (tau_b exp(s_bn - lse_b) - t_bn) / B,   tau_b = sum_n t_bn = eps + (1-eps) [n_b > 0]

written with a stable log-softmax so that logits of magnitude 1e3 do not overflow.  ``oracle_ce_step`` runs the full
oracle backward (FC / CPG / conv layers) with this loss in place of the BCE."""
import numpy as np


def targets(rowptr, col, N, eps):
    B = len(rowptr) - 1
    n = np.diff(np.asarray(rowptr, np.int64))
    T = np.full((B, N), eps / N, dtype=np.float64)
    for b in range(B):
        ids = np.asarray(col[rowptr[b]:rowptr[b + 1]], np.int64)
        T[b, ids] += (1.0 - eps) / max(int(n[b]), 1)
    return T


def ce_loss_grad(S, rowptr, col, eps):
    """(loss, G, lse) of fp64 logits S [B, N]."""
    S = np.asarray(S, np.float64)
    B, N = S.shape
    m = S.max(axis=1, keepdims=True)
    lse = (m + np.log(np.exp(S - m).sum(axis=1, keepdims=True)))[:, 0]
    T = targets(rowptr, col, N, eps)
    tau = T.sum(axis=1)
    loss = (T * (lse[:, None] - S)).sum() / B
    G = (tau[:, None] * np.exp(S - lse[:, None]) - T) / B
    return loss, G, lse


def oracle_ce_step(O, params, cfg, e1, rel, rowptr, col, masks=None):
    """Oracle forward + backward with the CE loss: (loss, gradients, forward outputs).  The oracle's backward forms
    G = (sigmoid(S) - zs) / (B N); its smoothed targets zs are replaced by sigmoid(S) - G_ce B N, exact in fp64 up to
    round-off, so that every layer below the scorer back-propagates the CE gradient."""
    dense = O.csr_to_dense(rowptr, col, cfg.num_ent)
    out = O.forward(params, cfg, e1, rel, True, masks, dense, np.float64)
    S = out["scores"]
    B, N = S.shape
    loss, G, _ = ce_loss_grad(S, rowptr, col, cfg.label_smoothing_epsilon)
    out["_cache"]["zs"] = O.sigmoid(S) - G * float(B * N)
    out["loss"] = loss
    return loss, O.backward(out, cfg), out
