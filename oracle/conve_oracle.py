"""CPU ORACLE (test infrastructure, NOT product code) for the CoPER-ConvE hot path.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this module; the product package
``coper_b200`` never does (it fails loudly when its CUDA library is missing).

What this restates (all citations relative to /root/reference/CoPER_ConvE/qa_cpg/):

* ``models.py:176-180``  embedding lookups                      -> :func:`forward`
* ``models.py:32-76``    ContextualParameterGenerator.generate  -> :func:`cpg_context`, :func:`forward`
* ``models.py:354-426``  ConvE._create_predictions              -> :func:`forward`
* ``models.py:428-446``  ConvE._compute_likelihoods (1-N)       -> :func:`forward`
* ``models.py:448-457``  ConvE._create_loss                     -> :func:`forward`
* ``models.py:196-200``  gradients + clip_by_global_norm(5.0)   -> :func:`backward`, :func:`clip_by_global_norm`
* ``metrics.py:40-76``   ranking_and_hits numerical core        -> :func:`rank_literal`, :func:`rank_count`, :func:`summarize_ranks`
* ``utils/amsgrad.py:130-159,230-241`` AMSGrad dense rule        -> :class:`AMSGradOracle`

PARITY PINNING STATUS.  The reference ships no tests / golden vectors and its
arithmetic lives in TensorFlow 1.14 (requirements.txt:6, README.md:116), which is
not installable here.  Two pins exist and are committed under ``tests/golden``:

1. ``metrics.py`` is executed UNMODIFIED (real NumPy, a 10-line fake ``tensorflow``
   module that only supplies ``tf.errors.OutOfRangeError``) by
   ``oracle/gen_golden.py``; :func:`rank_literal` / :func:`rank_count` are checked
   against its ranks, MR, MRR and Hits.
2. ``models.py`` is executed UNMODIFIED on ``oracle/tf1_shim`` — a torch-CPU
   emulation of the TF-1 API surface that file touches — so the *graph wiring*
   (op order, shapes, reshape/flatten order, loss reduction, clip) is the
   reference's own code, while each TF op's numerical semantics is restated from
   TF's documented behaviour (ASSUMED, listed below).  This is weaker than
   running real TensorFlow: for the model part parity is "pinned to the
   reference's graph code, TF op semantics assumed".

TF-1.14 semantics hard-coded here (assumed from TF documentation):
  * ``tf.nn.conv2d`` NHWC/HWIO, stride 1, VALID, cross-correlation.
  * ``tf.layers.batch_normalization``: axis=-1, epsilon=1e-3, gamma=1/beta=0 and
    moving mean 0 / variance 1 at init; ``momentum`` is the DECAY of the moving
    average; training-mode normalisation uses the biased batch variance; the
    moving-variance update is Bessel-corrected only on the fused (4-D) path.
  * ``tf.nn.dropout(x, keep)`` = x * mask / keep.
  * ``tf.losses.sigmoid_cross_entropy`` = mean over all elements of
    max(s,0) - s*z + log1p(exp(-|s|)).
  * ``tf.clip_by_global_norm``: g * clip / max(||g||, clip).
  * xavier_initializer = U(+-sqrt(6/(fan_in+fan_out))).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import numpy as np

BN_EPS = 1e-3  # tf.layers.batch_normalization default epsilon


# --------------------------------------------------------------------------------------
# configuration
# --------------------------------------------------------------------------------------
@dataclass
class OracleConfig:
    """Shape/behaviour knobs; names follow ``model_descriptors`` (run_cpg.py:115-137)."""
    num_ent: int
    num_rel: int
    ent_emb_size: int
    rel_emb_size: int
    context_rel_out: Optional[List[int]] = field(default_factory=list)  # [] = g_linear, [64] = g_MLP
    # not None: the conv filter [KH,KW,1,C] and bias [C] are generated per query as well (models.py:216-241) and the
    # convolution runs per example (tf.map_fn, models.py:375-380); restated for the cpg model type only
    context_rel_conv: Optional[List[int]] = None
    conv_in_height: int = 10           # models.py:261 hard-codes 10; parametrised for d=256 (16x16)
    conv_filter_height: int = 3
    conv_filter_width: int = 3
    conv_num_channels: int = 32
    label_smoothing_epsilon: float = 0.1
    hidden_dropout: float = 0.0        # == cfg.model.feature_map_dropout (run_cpg.py:128)
    output_dropout: float = 0.0
    context_rel_dropout: float = 0.0
    context_rel_use_batch_norm: bool = False
    batch_norm_momentum: float = 0.1
    batch_norm_train_stats: bool = False
    # "cpg"          context_rel_out = [...] (every *_cpg.yaml): FC weights / bias generated from the relation embedding
    # "plain"        context_rel_out = context_rel_conv = None (*_plain.yaml): the relation embedding is reshaped and
    #                stacked under the entity image (models.py:360-362), shared FC weights (models.py:334-340, 410)
    # "param_lookup" do_parameter_lookup (*_param_lookup.yaml): FC weights / bias are rows of per-relation tables
    #                (ParameterLookup, models.py:79-94, 279-287); there is no relation embedding (models.py:210, 180)
    variant: str = "cpg"
    # models.py:270-271, 406-407: the relation embedding is concatenated to the flattened conv features before the FC
    # layer (fc_input_size grows by rel_emb_size); not used by a shipped configuration
    concat_rel: bool = False

    @property
    def conv_in_width(self) -> int:
        assert self.ent_emb_size % self.conv_in_height == 0
        return self.ent_emb_size // self.conv_in_height

    @property
    def conv_total_height(self) -> int:  # models.py:261-265: plain ConvE convolves the stacked [e1; rel] image
        if self.variant == "plain":
            assert self.rel_emb_size == self.ent_emb_size, "tf.concat(axis=1) needs equal image widths (models.py:361)"
            return 2 * self.conv_in_height
        return self.conv_in_height

    @property
    def conv_out_hw(self):
        return (self.conv_total_height - self.conv_filter_height + 1,
                self.conv_in_width - self.conv_filter_width + 1)

    @property
    def conv_feature_size(self) -> int:  # models.py:266-269
        oh, ow = self.conv_out_hw
        return oh * ow * self.conv_num_channels

    @property
    def fc_input_size(self) -> int:  # models.py:266-271
        return self.conv_feature_size + (self.rel_emb_size if self.concat_rel else 0)

    @property
    def context_sizes(self) -> List[int]:  # models.py:294: [rel_emb_size] + context_rel_out
        if self.variant == "plain":          # shared weights == a generator with the constant context [1]
            return [1]
        if self.variant == "param_lookup":   # table rows == a linear generator applied to one-hot(rel)
            return [self.num_rel]
        return [self.rel_emb_size] + list(self.context_rel_out or [])


def xavier_uniform(rng: np.random.Generator, shape: Sequence[int], dtype=np.float32) -> np.ndarray:
    """tf.contrib.layers.xavier_initializer (models.py:208,213,49-54)."""
    shape = tuple(int(s) for s in shape)
    if len(shape) == 1:
        fan_in = fan_out = shape[0]
    else:
        rec = int(np.prod(shape[:-2])) if len(shape) > 2 else 1
        fan_in, fan_out = shape[-2] * rec, shape[-1] * rec
    lim = math.sqrt(6.0 / (fan_in + fan_out))
    return rng.uniform(-lim, lim, size=shape).astype(dtype)


def _bn_init(n, dtype=np.float32):
    return {"gamma": np.ones(n, dtype), "beta": np.zeros(n, dtype),
            "moving_mean": np.zeros(n, dtype), "moving_var": np.ones(n, dtype)}


def init_params(cfg: OracleConfig, seed: int = 0, bias_noise: float = 0.0) -> Dict[str, object]:
    """Random-init variables with the reference's shapes and initialisers (models.py:203-336).

    ``bias_noise`` > 0 perturbs the zero-initialised tensors (pred_bias, conv1_bias,
    CPG bias projections, BN beta/gamma/moving stats) so that tests exercise those paths.
    """
    rng = np.random.default_rng(seed)
    KH, KW, C = cfg.conv_filter_height, cfg.conv_filter_width, cfg.conv_num_channels
    F, d = cfg.fc_input_size, cfg.ent_emb_size
    ctx = cfg.context_sizes
    p: Dict[str, object] = {}
    p["ent_emb"] = xavier_uniform(rng, (cfg.num_ent, d))
    if cfg.variant != "param_lookup":                                   # models.py:210
        p["rel_emb"] = xavier_uniform(rng, (cfg.num_rel, cfg.rel_emb_size))
    p["conv1_weights"] = xavier_uniform(rng, (KH, KW, 1, C))
    p["conv1_bias"] = np.zeros(C, np.float32)
    if cfg.context_rel_conv is not None:                                # models.py:216-241
        assert cfg.variant == "cpg"
        cs = [cfg.rel_emb_size] + list(cfg.context_rel_conv)
        sw, sb = cs + [KH * KW * C], cs + [C]
        p["conv1_weights_proj"] = [xavier_uniform(rng, (sw[i], sw[i + 1])) for i in range(len(sw) - 1)]
        p["conv1_bias_proj"] = [np.zeros((sb[i], sb[i + 1]), np.float32) for i in range(len(sb) - 1)]
        p["conv1_weights_bn"] = [_bn_init(n) for n in cs[1:]]
        p["conv1_bias_bn"] = [_bn_init(n) for n in cs[1:]]
        del p["conv1_weights"], p["conv1_bias"]
    sizes_w = ctx + [F * d]
    sizes_b = ctx + [d]
    p["fc_weights_proj"] = [xavier_uniform(rng, (sizes_w[i], sizes_w[i + 1])) for i in range(len(sizes_w) - 1)]
    p["fc_bias_proj"] = [np.zeros((sizes_b[i], sizes_b[i + 1]), np.float32) for i in range(len(sizes_b) - 1)]
    if cfg.variant == "plain":          # the variable is [F, d] (models.py:334-337): Xavier limits of THAT shape
        p["fc_weights_proj"] = [xavier_uniform(rng, (F, d)).reshape(1, F * d)]
    if cfg.variant == "param_lookup":   # ParameterLookup initialises BOTH tables Xavier (models.py:86-89)
        p["fc_bias_proj"] = [xavier_uniform(rng, (cfg.num_rel, d))]
    p["fc_weights_bn"] = [_bn_init(n) for n in ctx[1:]]
    p["fc_bias_bn"] = [_bn_init(n) for n in ctx[1:]]
    p["Conv1BN"] = _bn_init(C)
    p["FCBN"] = _bn_init(d)
    p["pred_bias"] = np.zeros(cfg.num_ent, np.float32)
    if bias_noise > 0:
        def noise(a, scale=bias_noise):
            return (a + rng.normal(0, scale, a.shape)).astype(np.float32)
        p["pred_bias"] = noise(p["pred_bias"])
        if "conv1_bias" in p:
            p["conv1_bias"] = noise(p["conv1_bias"])
        p["fc_bias_proj"] = [noise(a) for a in p["fc_bias_proj"]]
        if "conv1_bias_proj" in p:
            p["conv1_bias_proj"] = [noise(a) for a in p["conv1_bias_proj"]]
        for bn in [p["Conv1BN"], p["FCBN"]] + p["fc_weights_bn"] + p["fc_bias_bn"] + p.get("conv1_weights_bn", []) \
                + p.get("conv1_bias_bn", []):
            bn["gamma"] = noise(bn["gamma"])
            bn["beta"] = noise(bn["beta"])
            bn["moving_mean"] = noise(bn["moving_mean"])
            bn["moving_var"] = (bn["moving_var"] * np.exp(rng.normal(0, bias_noise, bn["moving_var"].shape))).astype(np.float32)
    return p


def cast_params(p, dtype):
    def c(x):
        if isinstance(x, np.ndarray):
            return x.astype(dtype)
        if isinstance(x, list):
            return [c(y) for y in x]
        if isinstance(x, dict):
            return {k: c(v) for k, v in x.items()}
        return x
    return {k: c(v) for k, v in p.items()}


# --------------------------------------------------------------------------------------
# building blocks
# --------------------------------------------------------------------------------------
def _bn_forward(x2, bn, use_batch_stats, bessel_for_moving, momentum):
    """x2: [R, C].  Returns (out, cache, new_moving_mean, new_moving_var)."""
    R = x2.shape[0]
    if use_batch_stats:
        mean = x2.mean(axis=0)
        var = ((x2 - mean) ** 2).mean(axis=0)                    # biased (population) variance
        var_mov = var * (R / max(R - 1, 1)) if bessel_for_moving else var
        new_mm = bn["moving_mean"] * momentum + mean * (1 - momentum)
        new_mv = bn["moving_var"] * momentum + var_mov * (1 - momentum)
    else:
        mean, var = bn["moving_mean"], bn["moving_var"]
        new_mm, new_mv = bn["moving_mean"], bn["moving_var"]
    inv = 1.0 / np.sqrt(var + x2.dtype.type(BN_EPS))
    xhat = (x2 - mean) * inv
    out = xhat * bn["gamma"] + bn["beta"]
    return out, {"xhat": xhat, "inv": inv, "batch": use_batch_stats, "gamma": bn["gamma"]}, new_mm, new_mv


def _bn_backward(dout, cache):
    """Returns (dx, dgamma, dbeta) for x2 [R, C]."""
    xhat, inv, gamma = cache["xhat"], cache["inv"], cache["gamma"]
    dgamma = (dout * xhat).sum(axis=0)
    dbeta = dout.sum(axis=0)
    if cache["batch"]:
        R = dout.shape[0]
        dx = gamma * inv * (dout - dbeta / R - xhat * dgamma / R)
    else:
        dx = dout * gamma * inv
    return dx, dgamma, dbeta


def _conv_valid(X, Wc):
    """X: [B,H,W], Wc: [KH,KW,C] -> [B,OH,OW,C]; cross-correlation, VALID (models.py:382-385)."""
    B, H, W = X.shape
    KH, KW, C = Wc.shape
    OH, OW = H - KH + 1, W - KW + 1
    Z = np.zeros((B, OH, OW, C), X.dtype)
    for i in range(KH):
        for j in range(KW):
            Z += X[:, i:i + OH, j:j + OW, None] * Wc[i, j][None, None, None, :]
    return Z


def _conv_valid_per_query(X, Wq):
    """X: [B,H,W], Wq: [B,KH,KW,C] -> [B,OH,OW,C]: one filter per example (tf.map_fn of conv2d, models.py:375-380)."""
    B, H, W = X.shape
    _, KH, KW, C = Wq.shape
    OH, OW = H - KH + 1, W - KW + 1
    Z = np.zeros((B, OH, OW, C), X.dtype)
    for i in range(KH):
        for j in range(KW):
            Z += X[:, i:i + OH, j:j + OW, None] * Wq[:, i, j][:, None, None, :]
    return Z


def cpg_context(r, projs, bns, cfg: OracleConfig, is_train, masks, dtype):
    """Hidden layers of ContextualParameterGenerator.generate (models.py:56-68).

    Returns (context, caches, moving_updates).  With ``context_rel_out == []`` (g_linear)
    the context is the relation embedding itself.
    """
    h = r
    caches, updates = [], []
    keep = 1.0 - (cfg.context_rel_dropout if is_train else 0.0)
    for i, P in enumerate(projs[:-1]):
        a = h @ P
        c = {"in": h, "P": P}
        if cfg.context_rel_use_batch_norm:
            use_batch = bool(cfg.batch_norm_train_stats and is_train)
            a_bn, bc, mm, mv = _bn_forward(a, bns[i], use_batch, False, cfg.batch_norm_momentum)
            c["bn"] = bc
            updates.append((mm, mv))
        else:
            a_bn = a
            updates.append(None)
        act = np.maximum(a_bn, 0)
        c["relu"] = a_bn > 0
        m = masks[i] if (masks is not None and keep < 1.0) else None
        if m is not None:
            act = act * m.astype(dtype) / dtype(keep)
        c["mask"], c["keep"] = m, keep
        caches.append(c)
        h = act
    return h, caches, updates


def _cpg_context_backward(dh, caches, use_bn):
    """Back through the hidden layers; returns (dr, [dP_i], [(dgamma, dbeta) or None])."""
    dPs, dbns = [], []
    for c in reversed(caches):
        if c["mask"] is not None:
            dh = dh * c["mask"].astype(dh.dtype) / dh.dtype.type(c["keep"])
        dh = dh * c["relu"]
        if use_bn:
            dh, dg, db = _bn_backward(dh, c["bn"])
            dbns.append((dg, db))
        else:
            dbns.append(None)
        dPs.append(c["in"].T @ dh)
        dh = dh @ c["P"].T
    return dh, dPs[::-1], dbns[::-1]


# --------------------------------------------------------------------------------------
# forward / backward
# --------------------------------------------------------------------------------------
def forward(params, cfg: OracleConfig, e1, rel, is_train=False, masks=None, labels=None,
            dtype=np.float64, want_scores=True, lookup=None):
    """Restates models.py:176-192 for the CPG (``context_rel_out`` not None,
    ``context_rel_conv`` None) configuration every shipped ``*_cpg.yaml`` uses.

    masks: optional dict of Bernoulli keep-masks (bool/0-1 arrays) with keys
      'feature_map' [B,OH,OW,C], 'output' [B,d], 'ctx_w'/'ctx_b' lists per hidden layer.
    labels: dense multi-hot [B,N] (e2_multi) or None.
    lookup: sampled-label mode (models.py:438-443; ``use_negative_sampling``): int [B,L] entity ids, ``labels`` is then
      the [B,L] label matrix of those ids; the loss is the mean over B*L (same ``+ 1/num_ent`` smoothing, :450).
    Returns a dict of tensors (and caches for :func:`backward`).
    """
    dt = np.dtype(dtype).type
    p = cast_params(params, dtype)
    masks = masks or {}
    e1 = np.asarray(e1, np.int64)
    rel = np.asarray(rel, np.int64)
    B = e1.shape[0]
    H, W = cfg.conv_in_height, cfg.conv_in_width
    C = cfg.conv_num_channels
    OH, OW = cfg.conv_out_hw
    F, d = cfg.fc_input_size, cfg.ent_emb_size

    variant = cfg.variant
    x0 = p["ent_emb"][e1]                                     # models.py:176
    r = p["rel_emb"][rel] if variant != "param_lookup" else None   # models.py:178 / 180
    X = x0.reshape(B, H, W)                                   # models.py:355
    if variant == "plain":                                    # models.py:360-362: [e1 image; rel image] along height
        X = np.concatenate([X, r.reshape(B, H, W)], axis=1)
    conv_cpg = cfg.context_rel_conv is not None
    if conv_cpg:
        # models.py:367 (_get_conv_params) generates weights then bias: their hidden-layer dropouts are drawn first
        KH, KW = cfg.conv_filter_height, cfg.conv_filter_width
        ccw, ccw_caches, ccw_upd = cpg_context(r, p["conv1_weights_proj"], p["conv1_weights_bn"], cfg, is_train,
                                               masks.get("ctx_cw"), dt)
        ccb, ccb_caches, ccb_upd = cpg_context(r, p["conv1_bias_proj"], p["conv1_bias_bn"], cfg, is_train,
                                               masks.get("ctx_cb"), dt)
        Wq = (ccw @ p["conv1_weights_proj"][-1]).reshape(B, KH, KW, C)       # [-1] + [KH, KW, 1, C]
        bq = ccb @ p["conv1_bias_proj"][-1]                                  # [B, C]
        Z = _conv_valid_per_query(X, Wq) + bq[:, None, None, :]               # models.py:375-381
    else:
        Z = _conv_valid(X, p["conv1_weights"][:, :, 0, :]) + p["conv1_bias"]     # models.py:382-385
    use_batch = bool(cfg.batch_norm_train_stats and is_train)  # models.py:358
    Zbn, bn1c, mm1, mv1 = _bn_forward(Z.reshape(-1, C), p["Conv1BN"], use_batch, True, cfg.batch_norm_momentum)
    A1 = np.maximum(Zbn, 0)                                   # models.py:389
    relu1 = Zbn > 0
    keep1 = 1.0 - (cfg.hidden_dropout if is_train else 0.0)   # models.py:390-391
    m1 = masks.get("feature_map") if keep1 < 1.0 else None
    if m1 is not None:
        A1 = A1 * m1.reshape(-1, C).astype(dtype) / dt(keep1)
    f = A1.reshape(B, cfg.conv_feature_size)                  # models.py:404  (h,w,c) order
    if cfg.concat_rel:                                        # models.py:406-407
        f = np.concatenate([f, r], axis=1)

    # CPG (models.py:338-352, 56-76): weights and bias generators own separate hidden nets.
    if variant == "cpg":
        cw, cw_caches, cw_upd = cpg_context(r, p["fc_weights_proj"], p["fc_weights_bn"], cfg, is_train,
                                            masks.get("ctx_w"), dt)
        cb, cb_caches, cb_upd = cpg_context(r, p["fc_bias_proj"], p["fc_bias_bn"], cfg, is_train,
                                            masks.get("ctx_b"), dt)
    else:
        # plain: y = f.W + b (models.py:410) == the contraction below with the constant context [1];
        # param_lookup: y_b = f_b . table[rel_b] + bias_table[rel_b] (models.py:90-94, 412) == the same contraction
        # with the one-hot context (adding exact zeros)
        if variant == "plain":
            cw = np.ones((B, 1), dtype)
        else:
            cw = np.zeros((B, cfg.num_rel), dtype)
            cw[np.arange(B), rel] = 1
        cb, cw_caches, cb_caches, cw_upd, cb_upd = cw, [], [], [], []
    Pw = p["fc_weights_proj"][-1]                             # [dc, F*d]
    Pb = p["fc_bias_proj"][-1]                                # [dc, d]
    dc = Pw.shape[0]
    # y_b = f_b . reshape(c_b . P, [F, d]) + c_b . P_b  (models.py:70-73, 412), evaluated in the
    # algebraically identical fused form y = (c (x) f) . P^  (P^ = P viewed [dc*F, d]).
    kr = (cw[:, :, None] * f[:, None, :]).reshape(B, dc * F)
    y = kr @ Pw.reshape(dc * F, d) + cb @ Pb
    keep2 = 1.0 - (cfg.output_dropout if is_train else 0.0)   # models.py:414-415
    m2 = masks.get("output") if keep2 < 1.0 else None
    yd = y * m2.astype(dtype) / dt(keep2) if m2 is not None else y
    ybn, bn2c, mm2, mv2 = _bn_forward(yd, p["FCBN"], use_batch, False, cfg.batch_norm_momentum)  # :416-418
    q = np.maximum(ybn, 0)                                    # models.py:419
    relu2 = ybn > 0

    out = {"x0": x0, "r": r, "Z": Z, "f": f, "cw": cw, "cb": cb, "y": y, "q": q,
           "moving": {"Conv1BN": (mm1, mv1), "FCBN": (mm2, mv2), "ctx_w": cw_upd, "ctx_b": cb_upd},
           "_cache": dict(e1=e1, rel=rel, X=X, bn1=bn1c, relu1=relu1, m1=m1, keep1=keep1, m2=m2, keep2=keep2,
                          bn2=bn2c, relu2=relu2, cw_caches=cw_caches, cb_caches=cb_caches, p=p, B=B)}
    if conv_cpg:
        out["ccw"], out["ccb"] = ccw, ccb
        out["moving"]["ctx_cw"], out["moving"]["ctx_cb"] = ccw_upd, ccb_upd
        out["_cache"].update(Wq=Wq, ccw_caches=ccw_caches, ccb_caches=ccb_caches)
    if lookup is not None:
        lk = np.asarray(lookup, np.int64)
        Eg = p["ent_emb"][lk]                                  # tf.gather -> [B, L, d]   (models.py:438)
        SL = np.einsum("bd,bld->bl", q, Eg) + p["pred_bias"][lk]   # models.py:439-442
        out["scores_lookup"] = SL
        if want_scores:
            out["scores"] = q @ p["ent_emb"].T + p["pred_bias"]
        z = np.asarray(labels).astype(dtype)
        zs = dt(1.0 - cfg.label_smoothing_epsilon) * z + dt(1.0 / cfg.num_ent)       # models.py:450
        el = np.maximum(SL, 0) - SL * zs + np.log1p(np.exp(-np.abs(SL)))
        out["loss"] = el.mean()                                # mean over B*L
        out["_cache"]["zs"] = zs
        out["_cache"]["lookup"] = lk
        return out
    if want_scores or labels is not None:
        S = q @ p["ent_emb"].T + p["pred_bias"]              # models.py:434-437
        out["scores"] = S
        if labels is not None:
            z = np.asarray(labels).astype(dtype)
            zs = dt(1.0 - cfg.label_smoothing_epsilon) * z + dt(1.0 / cfg.num_ent)   # models.py:450
            el = np.maximum(S, 0) - S * zs + np.log1p(np.exp(-np.abs(S)))            # stable BCE-with-logits
            out["loss"] = el.mean()                            # models.py:451-453 (mean over B*N)
            out["_cache"]["zs"] = zs
    return out


def sigmoid(x):
    return np.where(x >= 0, 1.0 / (1.0 + np.exp(-np.abs(x))), np.exp(-np.abs(x)) / (1.0 + np.exp(-np.abs(x))))


def backward(out, cfg: OracleConfig):
    """Analytic gradients of ``out['loss']`` w.r.t. every trainable variable
    (what ``optimizer.compute_gradients`` returns at models.py:198), un-clipped.
    Entity-table gradient = dense scorer term + scatter of the e1 gather gradient.
    """
    c = out["_cache"]
    p, B = c["p"], c["B"]
    q, f = out["q"], out["f"]
    N, d = p["ent_emb"].shape
    C = cfg.conv_num_channels
    F = cfg.fc_input_size
    OH, OW = cfg.conv_out_hw
    KH, KW = cfg.conv_filter_height, cfg.conv_filter_width
    g: Dict[str, object] = {}

    if "lookup" in c:
        # sampled labels (models.py:438-443): the gradients of the two tf.gather calls are IndexedSlices; the dense
        # sums are returned under the usual names, the slices under "_sparse" (values [M, ...], indices [M]) in the
        # form tf.clip_by_global_norm / the sparse AMSGrad rule consume them.
        lk = c["lookup"]
        L = lk.shape[1]
        SL = out["scores_lookup"]
        G = (sigmoid(SL) - c["zs"]) / SL.dtype.type(B * L)
        dq = np.einsum("bl,bld->bd", G, p["ent_emb"][lk])
        dE = np.zeros_like(p["ent_emb"])
        sl_vals = (G[:, :, None] * q[:, None, :]).reshape(B * L, d)
        np.add.at(dE, lk.reshape(-1), sl_vals)
        db = np.zeros_like(p["pred_bias"])
        np.add.at(db, lk.reshape(-1), G.reshape(-1))
        g["pred_bias"] = db
        g["_sparse"] = {"ent_emb": [(sl_vals, lk.reshape(-1))], "pred_bias": [(G.reshape(-1), lk.reshape(-1))]}
    else:
        S = out["scores"]
        G = (sigmoid(S) - c["zs"]) / S.dtype.type(B * N)       # dL/dS
        g["pred_bias"] = G.sum(axis=0)
        dE = G.T @ q
        dq = G @ p["ent_emb"]
    # FC block backward: relu -> FCBN -> output dropout
    dybn = dq * c["relu2"]
    dyd, dg2, db2 = _bn_backward(dybn, c["bn2"])
    g["FCBN"] = {"gamma": dg2, "beta": db2}
    dy = dyd * c["m2"].astype(dyd.dtype) / dyd.dtype.type(c["keep2"]) if c["m2"] is not None else dyd
    # CPG contraction backward
    cw, cb = out["cw"], out["cb"]
    Pw = p["fc_weights_proj"][-1]
    Pb = p["fc_bias_proj"][-1]
    dc = Pw.shape[0]
    P3 = Pw.reshape(dc, F, d)
    kr = (cw[:, :, None] * f[:, None, :]).reshape(B, dc * F)
    dPw = (kr.T @ dy).reshape(dc, F * d)
    dPb = cb.T @ dy
    T = np.einsum("bj,kij->bki", dy, P3, optimize=True)         # T[b,k,i] = sum_j P[k,i,j] dy[b,j] (as a GEMM)
    df = np.einsum("bk,bki->bi", cw, T)
    dcw = np.einsum("bi,bki->bk", f, T)
    dcb = dy @ Pb.T
    use_bn = cfg.context_rel_use_batch_norm
    variant = cfg.variant
    if variant == "cpg":
        dr_w, dPs_w, dbn_w = _cpg_context_backward(dcw, c["cw_caches"], use_bn)
        dr_b, dPs_b, dbn_b = _cpg_context_backward(dcb, c["cb_caches"], use_bn)
        dr = dr_w + dr_b
    else:                                                       # constant / one-hot context: nothing flows into it
        dPs_w, dPs_b, dbn_w, dbn_b, dr = [], [], [], [], None
    g["fc_weights_proj"] = dPs_w + [dPw]
    g["fc_bias_proj"] = dPs_b + [dPb]
    g["fc_weights_bn"] = [None if t is None else {"gamma": t[0], "beta": t[1]} for t in dbn_w]
    g["fc_bias_bn"] = [None if t is None else {"gamma": t[0], "beta": t[1]} for t in dbn_b]
    # conv block backward: feature-map dropout -> relu -> Conv1BN -> bias -> conv
    if cfg.concat_rel:                                         # tf.concat backward (models.py:407): the tail is d rel_emb
        Fc = cfg.conv_feature_size
        dr = df[:, Fc:] if dr is None else dr + df[:, Fc:]
        df_full, df = df, df[:, :Fc]
    dA1 = df.reshape(-1, C)
    if c["m1"] is not None:
        dA1 = dA1 * c["m1"].reshape(-1, C).astype(dA1.dtype) / dA1.dtype.type(c["keep1"])
    dZbn = dA1 * c["relu1"]
    dZ2, dg1, db1 = _bn_backward(dZbn, c["bn1"])
    g["Conv1BN"] = {"gamma": dg1, "beta": db1}
    dZ = dZ2.reshape(B, OH, OW, C)
    X = c["X"]
    dX = np.zeros_like(X)
    if "Wq" in c:                                              # per-query filters: back through the two generators
        Wq = c["Wq"]
        dWq = np.zeros_like(Wq)
        for i in range(KH):
            for j in range(KW):
                dWq[:, i, j] = np.einsum("bhw,bhwc->bc", X[:, i:i + OH, j:j + OW], dZ)
                dX[:, i:i + OH, j:j + OW] += np.einsum("bhwc,bc->bhw", dZ, Wq[:, i, j])
        dbq = dZ.sum(axis=(1, 2))
        Pc, Pcb = p["conv1_weights_proj"][-1], p["conv1_bias_proj"][-1]
        dWq2 = dWq.reshape(B, -1)
        dr_cw, dPs_cw, dbn_cw = _cpg_context_backward(dWq2 @ Pc.T, c["ccw_caches"], use_bn)
        dr_cb, dPs_cb, dbn_cb = _cpg_context_backward(dbq @ Pcb.T, c["ccb_caches"], use_bn)
        g["conv1_weights_proj"] = dPs_cw + [out["ccw"].T @ dWq2]
        g["conv1_bias_proj"] = dPs_cb + [out["ccb"].T @ dbq]
        g["conv1_weights_bn"] = [None if t is None else {"gamma": t[0], "beta": t[1]} for t in dbn_cw]
        g["conv1_bias_bn"] = [None if t is None else {"gamma": t[0], "beta": t[1]} for t in dbn_cb]
        dr = dr + dr_cw + dr_cb
    else:
        g["conv1_bias"] = dZ.sum(axis=(0, 1, 2))
        Wc = p["conv1_weights"][:, :, 0, :]
        dWc = np.zeros_like(Wc)
        for i in range(KH):
            for j in range(KW):
                dWc[i, j] = np.einsum("bhw,bhwc->c", X[:, i:i + OH, j:j + OW], dZ)
                dX[:, i:i + OH, j:j + OW] += dZ @ Wc[i, j]
        g["conv1_weights"] = dWc[:, :, None, :]
    H = cfg.conv_in_height
    if variant == "plain":                                     # tf.concat backward: the two halves of the image
        dx0 = dX[:, :H].reshape(B, d)
        dr = dX[:, H:].reshape(B, d) + (dr if cfg.concat_rel else 0)
    else:
        dx0 = dX.reshape(B, d)
    np.add.at(dE, c["e1"], dx0)                               # gather gradient (IndexedSlices -> dense)
    g["ent_emb"] = dE
    g["_dq"], g["_dy"], g["_df"], g["_dr"], g["_dx0"], g["_G"] = dq, dy, (df_full if cfg.concat_rel else df), dr, dx0, G
    if "_sparse" in g:
        g["_sparse"]["ent_emb"].append((dx0, c["e1"]))         # the e1 gather (models.py:176)
    if variant == "param_lookup":
        # ParameterLookup.generate is an embedding_lookup of the tables (models.py:91): their gradients are
        # IndexedSlices with one [F*d] / [d] slice per query
        sp = g.setdefault("_sparse", {})
        sp["fc_weights"] = [((f[:, :, None] * dy[:, None, :]).reshape(B, F * d), c["rel"])]
        sp["fc_bias"] = [(dy, c["rel"])]
        return g
    dRel = np.zeros_like(p["rel_emb"])
    np.add.at(dRel, c["rel"], dr)
    g["rel_emb"] = dRel
    g.setdefault("_sparse", {})["rel_emb"] = [(dr, c["rel"])]  # models.py:178: always an IndexedSlices
    return g


def flatten_grads(g) -> List[np.ndarray]:
    """All trainable-variable gradients as a flat list (order irrelevant for the norm)."""
    outl = []
    for k, v in g.items():
        if k.startswith("_"):
            continue
        if isinstance(v, np.ndarray):
            outl.append(v)
        elif isinstance(v, dict):
            outl.extend(v.values())
        elif isinstance(v, list):
            for t in v:
                if t is None:
                    continue
                outl.extend(t.values() if isinstance(t, dict) else [t])
    return outl


def clip_by_global_norm(grads: List[np.ndarray], clip_norm: float = 5.0, sparse_values: Sequence[np.ndarray] = ()):
    """tf.clip_by_global_norm (models.py:199): scale = clip / max(norm, clip).

    ``sparse_values``: the ``values`` of gradients TF represents as ``tf.IndexedSlices`` (a variable read only through
    ``tf.nn.embedding_lookup`` — ``rel_emb`` on this path, models.py:178).  ``clip_ops.global_norm`` takes
    ``l2_loss(t.values)`` for those, i.e. slices that share an index are NOT summed before squaring.  Returns
    (clipped dense grads, norm) or, when sparse values are given, (clipped dense, clipped sparse values, norm)."""
    sq = sum(float((x.astype(np.float64) ** 2).sum()) for x in grads)
    sq += sum(float((x.astype(np.float64) ** 2).sum()) for x in sparse_values)
    norm = math.sqrt(sq)
    scale = clip_norm / max(norm, clip_norm)
    dense = [x * x.dtype.type(scale) for x in grads]
    if len(sparse_values):
        return dense, [x * x.dtype.type(scale) for x in sparse_values], norm
    return dense, norm


# --------------------------------------------------------------------------------------
# AMSGrad (utils/amsgrad.py)
# --------------------------------------------------------------------------------------
class AMSGradOracle:
    """Dense update rule of utils/amsgrad.py:130-159 with beta powers from :230-241.

    ``reference_bug_compat=True`` reproduces the dense path as written: the ``m`` and
    ``v`` slots are only decayed (amsgrad.py:142,149) and ``m + (1-b1) g`` / ``v + (1-b2) g^2``
    are never assigned back, so m == v == 0 forever and
        v_hat <- max(v_hat, (1-b2) g^2);  theta <- theta - lr_t (1-b1) g / (sqrt(v_hat) + eps).
    ``False`` gives textbook AMSGrad (m, v accumulated).
    """

    def __init__(self, lr, beta1=0.9, beta2=0.999, eps=1e-8, reference_bug_compat=True):
        self.lr, self.b1, self.b2, self.eps = lr, beta1, beta2, eps
        self.b1p, self.b2p = beta1, beta2                      # amsgrad.py:109-114 (powers start at beta)
        self.compat = reference_bug_compat
        self.state = {}

    def lr_t(self):
        return self.lr * math.sqrt(1 - self.b2p) / (1 - self.b1p)   # amsgrad.py:137

    def apply(self, named, sparse=None):
        """named: dict name -> (theta, grad) ndarrays, dense rule; sparse: dict name -> (theta, values [M, ...],
        indices [M]) for IndexedSlices gradients, which TF routes to ``_apply_sparse_shared`` (amsgrad.py:161-189):
        there the slots ARE accumulated (``scatter_add`` mutates them): m <- b1 m; m[idx] += (1-b1) g_i (duplicates
        add); v <- b2 v; v[idx] += (1-b2) g_i^2 (each slice squared on its own); v_hat <- max(v_hat, v);
        theta <- theta - lr_t m / (sqrt(v_hat) + eps) over the WHOLE variable.  Updates theta in place."""
        lr_t = self.lr_t()
        for k, (th, vals, idx) in (sparse or {}).items():
            st = self.state.setdefault(k, {"m": np.zeros_like(th), "v": np.zeros_like(th),
                                           "vhat": np.zeros_like(th)})
            dt = th.dtype.type
            st["m"] *= dt(self.b1)
            np.add.at(st["m"], idx, vals * dt(1 - self.b1))
            st["v"] *= dt(self.b2)
            np.add.at(st["v"], idx, vals * vals * dt(1 - self.b2))
            st["vhat"] = np.maximum(st["vhat"], st["v"])
            th -= dt(lr_t) * st["m"] / (np.sqrt(st["vhat"]) + dt(self.eps))
        for k, (th, g) in named.items():
            st = self.state.setdefault(k, {"m": np.zeros_like(th), "v": np.zeros_like(th),
                                           "vhat": np.zeros_like(th)})
            dt = th.dtype.type
            if self.compat:
                m_t = st["m"] * dt(self.b1) + g * dt(1 - self.b1)     # slot m stays 0
                v_t = st["v"] * dt(self.b2) + g * g * dt(1 - self.b2)
                st["m"] *= dt(self.b1)
                st["v"] *= dt(self.b2)
            else:
                st["m"] = m_t = st["m"] * dt(self.b1) + g * dt(1 - self.b1)
                st["v"] = v_t = st["v"] * dt(self.b2) + g * g * dt(1 - self.b2)
            st["vhat"] = np.maximum(st["vhat"], v_t)
            th -= dt(lr_t) * m_t / (np.sqrt(st["vhat"]) + dt(self.eps))
        self.b1p *= self.b1
        self.b2p *= self.b2


# --------------------------------------------------------------------------------------
# filtered ranking (metrics.py)
# --------------------------------------------------------------------------------------
def rank_literal(pred, e2, e2_multi):
    """metrics.py:44-51 literally (mask, restore gold, full argsort, where).

    pred: [B,N] float32 logits (copied), e2: [B] int, e2_multi: [B,N] multi-hot.
    """
    pred = np.array(pred, dtype=np.float32, copy=True)
    e2 = np.asarray(e2, np.int64)
    target_values = pred[np.arange(0, len(pred)), e2]            # metrics.py:44
    pred[np.asarray(e2_multi) == 1] = -np.inf                    # metrics.py:45
    pred[np.arange(0, len(pred)), e2] = target_values            # metrics.py:46
    ranks = []
    for i in range(len(e2)):
        pred1_args = np.argsort(-pred[i])                        # metrics.py:49
        ranks.append(int(np.where(pred1_args == e2[i])[0][0]) + 1)   # metrics.py:50 (Q16: [0][0])
    return np.asarray(ranks, np.int64)


def rank_count(pred, e2, e2_multi):
    """Count formulation: rank = 1 + #{n != e2 : not filtered, s_n > s_gold}; also returns the
    tie count #{n != e2 : not filtered, s_n == s_gold}.  Equal to :func:`rank_literal` whenever
    n_equal == 0 (np.argsort's tie order is unspecified, SURVEY Q9)."""
    pred = np.asarray(pred, np.float32)
    e2 = np.asarray(e2, np.int64)
    B, N = pred.shape
    filt = np.asarray(e2_multi) == 1
    gold = pred[np.arange(B), e2][:, None]
    valid = ~filt
    valid[np.arange(B), e2] = False
    n_greater = ((pred > gold) & valid).sum(axis=1)
    n_equal = ((pred == gold) & valid).sum(axis=1)
    return (1 + n_greater).astype(np.int64), n_equal.astype(np.int64)


def summarize_ranks(ranks, hits_to_compute=(1, 3, 5, 10, 20)):
    """metrics.py:53-57,65-76: Hits@k = mean(rank <= k), MR, MRR in float64."""
    ranks = np.asarray(ranks)
    hits = {k: float(np.mean([1.0 if r <= k else 0.0 for r in ranks])) for k in hits_to_compute}
    mr = float(np.mean(ranks))
    mrr = float(np.mean(1.0 / np.array(ranks)))
    return mr, mrr, hits


# --------------------------------------------------------------------------------------
# synthetic batches (SURVEY 8d)
# --------------------------------------------------------------------------------------
def synthetic_batch(cfg: OracleConfig, B: int, seed: int = 0, mean_pos: float = 3.0, max_pos: int = 64):
    """Seeded synthetic (e1, rel, positives) rows; positives per row ~ 1 + Geometric, drawn
    without replacement.  Returns e1, rel, e2 (gold = first positive), CSR (rowptr, col) and the
    dense multi-hot ``e2_multi`` the reference's pipeline would ship (data.py:182-186)."""
    rng = np.random.default_rng(seed)
    e1 = rng.integers(0, cfg.num_ent, B, dtype=np.int64)
    rel = rng.integers(0, cfg.num_rel, B, dtype=np.int64)
    k = np.minimum(rng.geometric(1.0 / mean_pos, B), min(max_pos, cfg.num_ent))
    rowptr = np.zeros(B + 1, np.int32)
    cols = []
    for b in range(B):
        c = rng.choice(cfg.num_ent, size=int(k[b]), replace=False)
        cols.append(c.astype(np.int32))
        rowptr[b + 1] = rowptr[b] + len(c)
    col = np.concatenate(cols).astype(np.int32)
    e2 = np.array([cols[b][0] for b in range(B)], np.int64)
    return e1, rel, e2, rowptr, col


def csr_to_dense(rowptr, col, N, dtype=np.float32):
    B = len(rowptr) - 1
    z = np.zeros((B, N), dtype)
    for b in range(B):
        z[b, col[rowptr[b]:rowptr[b + 1]]] = 1
    return z
