"""Diagnostic (not collected by pytest): how far the bf16 engine's downstream gradients sit from the fp64 oracle,
(a) against the unmodified oracle and (b) against the oracle backward evaluated at the ENGINE's own ReLU activation
pattern (the bf16 forward flips units whose pre-activation lies within rounding of zero; each flip moves that element
of dy by the full common part of dq, which dominates the max-norm error of (a)).
Lives under tests/ because it uses the oracle (only tests/, smoke() and bench.py's CPU legs may)."""
import os, sys
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE)); sys.path.insert(0, HERE)
import numpy as np, torch
from oracle import conve_oracle as O
import test_gpu_model as T
for name in ("toy_glinear_batch_stats", "toy_gmlp_bn_dropout", "ragged_mid", "d256_16x16", "plain_d200", "lookup_d200",
             "lookup_toy", "cpgconv_gmlp_d200"):
    kw, B = T.CASES[name]
    cfg = O.OracleConfig(**kw)
    params = O.init_params(cfg, seed=3, bias_noise=0.05)
    e1, rel, e2, rowptr, col = O.synthetic_batch(cfg, B, seed=5)
    e1[B // 2:] = e1[: B - B // 2]
    dense = O.csr_to_dense(rowptr, col, cfg.num_ent)
    for prec in ("bf16",):
        m = T.make(cfg, params, prec=prec)
        m.train_step(T.batch_of(e1, rel, e2, rowptr, col), apply_update=False)
        masks = T.export_masks(m, cfg, B)
        out = O.forward(params, cfg, e1, rel, True, masks, dense, np.float64)
        g = O.backward(out, cfg)
        b = m._bufs[B]
        mg = T.grads_by_name(m)
        last = g["fc_weights_proj"][-1].reshape(-1)
        def row(tag, g):
            print("%-24s %-6s dq %.2e dy %.2e df %.2e dE %.2e dP %.2e" % (
                name, tag, T.relerr(b.dq.cpu().numpy(), g["_dq"]), T.relerr(b.dy.cpu().numpy(), g["_dy"]),
                T.relerr(b.df.cpu().numpy(), g["_df"]), T.relerr(mg["ent_emb"], g["ent_emb"]),
                T.relerr(mg[m._last_w_name].reshape(-1), g["fc_weights_proj"][-1].reshape(-1))))
        row("plain", g)
        flips = int(((b.q.cpu().numpy() > 0) != (out["_cache"]["relu2"] > 0)).sum())
        out["_cache"]["relu2"] = (b.q.cpu().numpy() > 0).astype(np.float64)
        row("mask", O.backward(out, cfg))
        print("   relu units flipped by the bf16 forward: %d of %d" % (flips, b.q.numel()))
