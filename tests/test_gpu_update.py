"""The part of the training step that runs after the gradients are formed, against fp64 references: the fused squared
norm of the entity gradient (dE GEMM epilogue + head-entity scatter corrections), the finishing clip launch with an
external norm, the multi-tensor AMSGrad update with an ACTIVE global-norm clip, and the tensor-pipe operand copies the
update re-emits for the next step.

Tolerances:
  * dE_sumsq vs the fp64 sum of squares of the dE the call stored: 1e-6 relative (the epilogue sums 32 squares in fp32
    before it moves to fp64).
  * squared-norm corrections of the scatter: per writer row 1e-12 (both sides fp64 of the same fp32 values); their sum
    1e-6 of the sum of squares after the scatter.
  * global norm rebuilt in fp64 from the model's own gradient buffers: 1e-6 relative, every engine.
  * global norm vs the oracle's gradients at the device's pre-step parameters: 1e-4 (fp32-class engines), 5e-2 (bf16,
    the bar its parameter gradients are held to in test_gpu_model.py).
  * the update vs fp64 AMSGrad of the model's own gradients and clip factor: theta within 4 fp32 ulps of max|theta|
    plus 1e-5 * lr_t; m, v, vhat within 1e-6 of their max.
"""
import math

import numpy as np
import pytest
import torch

from oracle import conve_oracle as O
from test_gpu_model import CASES, batch_of, descriptors, export_masks, relerr

pytestmark = pytest.mark.gpu

PREC = {"fp32": 0, "bf16": 1, "tf32x3": 2, "fp16x3": 3}
FP32_CLASS = ("fp32", "tf32x3", "fp16x3")
NAN = float("nan")


@pytest.fixture(scope="module")
def L():
    from coper_b200 import _lib
    _lib.load()
    return _lib


def same_bits(a, b):
    """Bitwise equality of two device tensors of the same dtype (NaN-safe)."""
    it = {4: torch.int32, 8: torch.int64}[a.element_size()]
    return a.shape == b.shape and torch.equal(a.contiguous().view(it), b.contiguous().view(it))


def bf16_round(x):
    return torch.as_tensor(x, dtype=torch.float32).to(torch.bfloat16).to(torch.float64).numpy()


def csr_labels(rng, B, N):
    """1..5 distinct positives per query, as CSR."""
    counts = np.minimum(rng.integers(1, 6, B), N)
    rowptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    col = np.concatenate([rng.choice(N, size=int(k), replace=False) for k in counts]).astype(np.int32)
    return rowptr, col


# ------------------------------------------------------------------------------------------ 1. scorer norm, split form
SCORER_SHAPES = [(1, 1, 8), (7, 97, 40), (130, 1003, 200), (33, 5000, 256), (512, 40943, 200), (4096, 5118, 200),
                 (257, 1111, 40)]      # d = 40 (masked columns of the last 32-wide chunk), N % 128 != 0


@pytest.mark.parametrize("prec", ["bf16", "tf32x3", "fp16x3"])
@pytest.mark.parametrize("B,N,d", SCORER_SHAPES)
def test_scorer_norm_and_split_form(L, prec, B, N, d):
    """coper_score1n_bce_fwd_bwd_norm unsplit and split (dE on a second stream, as ConvE runs it) against the plain call
    and fp64: bf16 takes the fused single-pass scorer, tf32x3 / fp16x3 the three-pass path."""
    lib = L.load()
    p = PREC[prec]
    rng = np.random.default_rng(B * 5 + N + d)
    q = np.maximum(rng.normal(size=(B, d)), 0).astype(np.float32)
    E = rng.uniform(-0.05, 0.05, size=(N, d)).astype(np.float32)
    bias = (rng.normal(size=N) * 0.1).astype(np.float32)
    rowptr, col = csr_labels(rng, B, N)
    bits = torch.full((N, -(-B // 32)), -1, dtype=torch.int32, device="cuda")
    trp, tcol = torch.as_tensor(rowptr).cuda(), torch.as_tensor(col).cuda()
    L.call("coper_csr_to_bits_t", L.ptr(trp), L.ptr(tcol), B, 0, N, L.ptr(bits))
    pos, neg = np.float32(np.float32(0.9) + np.float32(1.0 / N)), np.float32(1.0 / N)
    inv = 1.0 / (B * N)
    ld = -(-N // 32) * 32
    tq, tE, tb = (torch.as_tensor(a).cuda() for a in (q, E, bias))
    ws = torch.empty(lib.coper_score1n_bce_workspace_bytes(B, N, d, p), dtype=torch.uint8, device="cuda")
    G = torch.empty(lib.coper_score1n_bce_G_bytes(B, N, p), dtype=torch.uint8, device="cuda")
    inputs = (L.ptr(tq), L.ptr(tE), None, L.ptr(tb), L.ptr(bits), B, N, d, float(pos), float(neg), inv)

    def outputs():       # dq, dE, dbias, loss, dE_sumsq: NaN sentinels
        f64 = dict(dtype=torch.float64, device="cuda")
        return (torch.full((B, d), NAN, device="cuda"), torch.full((N, d), NAN, device="cuda"),
                torch.full((N,), NAN, device="cuda"), torch.full((1,), NAN, **f64), torch.full((1,), NAN, **f64))

    dq0, dE0, db0, loss0, _ = outputs()
    L.call("coper_score1n_bce_fwd_bwd", *inputs, L.ptr(loss0), L.ptr(G), ld, L.ptr(dq0), L.ptr(dE0), L.ptr(db0),
           L.ptr(ws), ws.numel(), p)
    dq1, dE1, db1, loss1, ss1 = outputs()
    L.call("coper_score1n_bce_fwd_bwd_norm", *inputs, L.ptr(loss1), L.ptr(G), ld, L.ptr(dq1), L.ptr(dE1), L.ptr(db1),
           L.ptr(ss1), L.ptr(ws), ws.numel(), p)
    # split form: scorer + dq on this stream, then dE / dbias / dE_sumsq on a side stream ordered after it
    dq2, dE2, db2, loss2, ss2 = outputs()
    db_between = torch.zeros(N, device="cuda")
    L.call("coper_score1n_bce_fwd_bwd_norm", *inputs, L.ptr(loss2), L.ptr(G), ld, L.ptr(dq2), None, L.ptr(db2),
           L.ptr(ss2), L.ptr(ws), ws.numel(), p)
    side = torch.cuda.Stream()
    ev = torch.cuda.Event()
    ev.record()
    side.wait_event(ev)
    with torch.cuda.stream(side):
        db_between.copy_(db2)                        # what the first call left in dbias
        L.call("coper_score1n_bce_dE", L.ptr(G), B, N, d, inv, L.ptr(dE2), L.ptr(ss2), L.ptr(db2), L.ptr(ws), ws.numel(),
               p)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()

    for a, b in ((loss1, loss0), (dq1, dq0), (dE1, dE0), (db1, db0)):
        assert same_bits(a, b)
    for a, b in ((loss2, loss1), (dq2, dq1), (dE2, dE1), (db2, db1), (ss2, ss1)):
        assert same_bits(a, b)
    assert torch.isnan(db_between).all(), "the split scorer call wrote dbias"
    dE_np = dE1.cpu().numpy().astype(np.float64)
    assert np.isfinite(dE_np).all()
    ss_ref = float((dE_np ** 2).sum())
    assert abs(ss1.item() - ss_ref) <= 1e-6 * ss_ref, (ss1.item(), ss_ref)
    # against fp64 (bf16: on the rounded operands, as test_score1n_bce_fwd_bwd_tensor_pipe)
    qq, EE = (q.astype(np.float64), E.astype(np.float64)) if prec != "bf16" else (bf16_round(q), bf16_round(E))
    z = O.csr_to_dense(rowptr, col, N, np.float64)
    zs = np.where(z > 0, np.float64(pos), np.float64(neg))
    Gr = (O.sigmoid(qq @ EE.T + bias) - zs) * inv
    gtol = 2e-5 if prec != "bf16" else 1e-2
    for got, ref in ((dq1, Gr @ EE), (dE1, Gr.T @ qq), (db1, Gr.sum(0))):
        got = got.cpu().numpy()
        assert np.isfinite(got).all()
        assert relerr(got, ref) < gtol


# ------------------------------------------------------------------------------------------ 2. head-entity scatter
@pytest.mark.parametrize("M", [1, 130, 4096])
@pytest.mark.parametrize("pair", [False, True])
def test_head_scatter_norm_delta(L, M, pair):
    """norm_delta of coper_segscatter_add_norm / the a half of coper_segscatter_add_pair: the change of the squared
    norm of the shard's rows, reported once per destination row by its writer (the first position that holds it)."""
    rng = np.random.default_rng(M * 3 + pair)
    d, lo, hi, R, dr = 200, 100, 500, 22, 8
    if M == 1:
        e1 = np.array([lo + 17], np.int64)
    else:
        e1 = rng.integers(0, 700, M).astype(np.int64)           # many duplicates, rows of other shards on both sides
        e1[:10] = [0, lo - 1, lo, hi - 1, hi, hi + 5, lo, hi - 1, lo - 1, 650]
    src = rng.normal(size=(M, d)).astype(np.float32)
    before = rng.normal(size=(hi - lo, d)).astype(np.float32)
    sq_before = rng.uniform(0, 1, size=(hi - lo, d)).astype(np.float32)
    te1, tsrc, tdst, tsq = (torch.as_tensor(a).cuda() for a in (e1, src, before, sq_before))
    nd = torch.full((M,), NAN, dtype=torch.float64, device="cuda")
    if pair:
        rel = rng.integers(0, R, M).astype(np.int64)
        drr = rng.normal(size=(M, dr)).astype(np.float32)
        trel, tdrr = torch.as_tensor(rel).cuda(), torch.as_tensor(drr).cuda()
        dR, dRsq = torch.zeros(R, dr, device="cuda"), torch.zeros(R, dr, device="cuda")
        L.call("coper_segscatter_add_pair", L.ptr(te1), M, L.ptr(tsrc), d, L.ptr(tdst), L.ptr(tsq), lo, hi, L.ptr(nd),
               L.ptr(trel), M, L.ptr(tdrr), dr, L.ptr(dR), L.ptr(dRsq), 0, R)
    else:
        L.call("coper_segscatter_add_norm", L.ptr(te1), M, L.ptr(tsrc), d, L.ptr(tdst), L.ptr(tsq), lo, hi, L.ptr(nd))
    torch.cuda.synchronize()
    delta = nd.cpu().numpy()
    after = tdst.cpu().numpy().astype(np.float64)
    b64 = before.astype(np.float64)
    owned = (e1 >= lo) & (e1 < hi)
    first = np.zeros(M, bool)
    first[np.unique(e1, return_index=True)[1]] = True
    writer = owned & first
    assert np.isfinite(delta).all()
    assert (delta[~writer] == 0).all(), "norm_delta of a non-writer / another shard's row"
    row_delta = (after ** 2 - b64 ** 2).sum(1)
    row_mag = (after ** 2 + b64 ** 2).sum(1)
    rows = e1[writer] - lo
    assert (np.abs(delta[writer] - row_delta[rows]) <= 1e-12 * row_mag[rows]).all()
    total = float((after ** 2 - b64 ** 2).sum())
    assert abs(delta.sum() - total) <= 1e-6 * float((after ** 2).sum())
    # the scattered values themselves
    ref, ref_sq = b64.copy(), sq_before.astype(np.float64)
    np.add.at(ref, e1[owned] - lo, src[owned].astype(np.float64))
    np.add.at(ref_sq, e1[owned] - lo, src[owned].astype(np.float64) ** 2)
    assert np.abs(after - ref).max() <= 1e-6 * np.abs(ref).max()
    assert np.abs(tsq.cpu().numpy() - ref_sq).max() <= 1e-6 * np.abs(ref_sq).max()
    if pair:
        rr, rsq = np.zeros((R, dr)), np.zeros((R, dr))
        np.add.at(rr, rel, drr.astype(np.float64))
        np.add.at(rsq, rel, drr.astype(np.float64) ** 2)
        assert np.abs(dR.cpu().numpy() - rr).max() <= 1e-6 * np.abs(rr).max()
        assert np.abs(dRsq.cpu().numpy() - rsq).max() <= 1e-6 * np.abs(rsq).max()


# ------------------------------------------------------------------------------------------ 3. finishing launch
def _dense_descs(L, grads, ext):
    """coper_param_desc array + chunk list for dense gradients; tensor `ext` has an external norm and no chunks."""
    desc_dt = np.dtype([("theta", np.uint64), ("grad", np.uint64), ("m", np.uint64), ("v", np.uint64),
                        ("vhat", np.uint64), ("prepared", np.uint64), ("grad_sq", np.uint64), ("n", np.int64),
                        ("prepared_prec", np.int32), ("mode", np.int32)])
    desc = np.zeros(len(grads), desc_dt)
    chunks, offsets = [], [0]
    for t, g in enumerate(grads):
        desc[t]["grad"] = desc[t]["theta"] = desc[t]["vhat"] = g.data_ptr()
        desc[t]["n"] = g.numel()
        desc[t]["mode"] = 2 if t == ext else 0
        if t != ext:
            chunks += [(t, c) for c in range(-(-g.numel() // L.MT_CHUNK))]
        offsets.append(len(chunks))
    return (torch.as_tensor(desc.view(np.uint8)).cuda(), torch.as_tensor(np.array(chunks, np.int32)).cuda(),
            len(chunks), torch.as_tensor(np.array(offsets, np.int32)).cuda())


@pytest.mark.parametrize("case", ["active", "inactive", "zero", "negative_deltas"])
def test_mt_sumsq_clip_external_norm(L, case):
    """coper_mt_sumsq_clip with tensor 0's squared norm supplied as parts + deltas (COPER_GRAD_NORM_EXTERNAL):
    clip_out = {c / max(norm, c), norm} in fp64; the external sum is clamped at 0."""
    rng = np.random.default_rng(11)
    clip = 5.0
    sizes = [1003 * 200, 40943, 288, 32, 17, 65536 * 3 + 5]
    scale = {"active": 0.05, "inactive": 0.001, "zero": 0.0, "negative_deltas": 0.003}[case]
    grads = [(rng.normal(size=n) * scale).astype(np.float32) for n in sizes]
    if case == "zero":
        parts, deltas = np.array([0.3]), np.array([-0.1, -0.2])     # 0.3 - 0.1 - 0.2 < 0 in fp64
        assert parts[0] + deltas[0] + deltas[1] < 0
    elif case == "negative_deltas":
        parts, deltas = rng.uniform(0, 5, 7), -rng.uniform(0, 0.03, 300)
    else:
        parts, deltas = rng.uniform(0, 1, 7), rng.normal(size=300) * 1e-3
    tg = [torch.as_tensor(g).cuda() for g in grads]
    tg[0].fill_(NAN)                                 # an external norm: the gradient is never read
    descs, chunks, nch, offs = _dense_descs(L, tg, 0)
    nt = len(tg)
    tparts, tdeltas = torch.as_tensor(parts).cuda(), torch.as_tensor(deltas).cuda()
    partials = torch.zeros(nch, dtype=torch.float64, device="cuda")
    sums = torch.full((nt,), NAN, dtype=torch.float64, device="cuda")
    clip_out = torch.full((2,), NAN, device="cuda")
    L.call("coper_mt_sumsq_clip", L.ptr(descs), nt, L.ptr(chunks), nch, L.ptr(offs), L.ptr(partials), L.ptr(sums), 0,
           L.ptr(tparts), len(parts), L.ptr(tdeltas), len(deltas), clip, L.ptr(clip_out))
    torch.cuda.synchronize()
    s = sums.cpu().numpy()
    ext = max(math.fsum(list(parts) + list(deltas)), 0.0)
    if case == "negative_deltas":
        assert deltas.sum() < 0 < ext
    assert abs(s[0] - ext) <= 1e-12 * max(ext, 1e-300)
    for t in range(1, nt):
        ref = float((grads[t].astype(np.float64) ** 2).sum())
        assert abs(s[t] - ref) <= 1e-6 * ref if ref > 0 else s[t] == 0.0
    norm = math.sqrt(ext + sum(float((g.astype(np.float64) ** 2).sum()) for g in grads[1:]))
    cs, got_norm = (float(x) for x in clip_out.cpu().numpy())
    assert abs(got_norm - norm) <= 1e-6 * norm if norm > 0 else got_norm == 0.0
    ref_cs = clip / max(norm, clip)
    assert abs(cs - ref_cs) <= 1e-6 * ref_cs
    assert (cs == 1.0) == (norm <= clip)
    if case == "active":
        assert norm > clip
    elif case in ("inactive", "zero"):
        assert norm <= clip


# ------------------------------------------------------------------------------------------ 4. multi-step training
UPDATE_CASES = {
    "ragged_mid": CASES["ragged_mid"],                 # cpg, d = 200: fused norm with the pair scatter
    "lookup_d200": CASES["lookup_d200"],               # per-relation tables: IndexedSlices rule (c^2 grad_sq)
    "big_batch": CASES["big_batch"],                   # B = 4096: the largest batch of the fused norm
    "big_batch_4097": (CASES["big_batch"][0], 4097),   # one more query: coper_mt_sumsq reads dE itself
    # d % 8 == 4: bf16 / fp16x3 re-prepare the operands after the update, tf32x3 still emits them from the update
    "d36_h6": (dict(num_ent=517, num_rel=9, ent_emb_size=36, rel_emb_size=6, context_rel_out=[], conv_in_height=6,
                    batch_norm_train_stats=True, hidden_dropout=0.3, output_dropout=0.2), 67),
}
STEPS = 4              # eager, capture + replay, replay, replay
LR = 1e-3
B1, B2, EPS = np.float32(0.9), np.float32(0.999), np.float32(1e-8)
OMB1, OMB2 = float(np.float32(1) - B1), float(np.float32(1) - B2)     # the kernels' 1 - beta, formed in fp32


def tree_get(tree, name):
    """A trainable of the model by its name, from an oracle params / gradient tree."""
    if name in ("fc_weights", "fc_bias"):                 # plain / param_lookup variables
        return tree[name + "_proj"][0]
    if "/CPG/Projection" in name:
        gen, rest = name.split("/CPG/Projection")
        i, _, bn = rest.partition("/BatchNorm/")
        return tree[gen + "_bn"][int(i)][bn] if bn else tree[gen + "_proj"][int(i)]
    if name.startswith(("Conv1BN/", "FCBN/")):
        nm, k = name.split("/")
        return tree[nm][k]
    return tree[name]


def params_of(model, template):
    """The model's variables and batch-norm statistics in the oracle's naming (fp64)."""
    get = lambda t, like: t.detach().cpu().numpy().astype(np.float64).reshape(np.shape(like))
    bn = lambda b: {k: getattr(b, k).cpu().numpy().astype(np.float64) for k in ("gamma", "beta", "moving_mean",
                                                                               "moving_var")}
    p = {"ent_emb": get(model.ent_emb, template["ent_emb"]), "pred_bias": get(model.pred_bias, template["pred_bias"]),
         "Conv1BN": bn(model.conv1_bn), "FCBN": bn(model.fc_bn)}
    if model.rel_emb is not None:
        p["rel_emb"] = get(model.rel_emb, template["rel_emb"])
    if model.conv_w_gen is None:
        p["conv1_weights"] = get(model.conv1_weights, template["conv1_weights"])
        p["conv1_bias"] = get(model.conv1_bias, template["conv1_bias"])
    for gen in model.generators:
        p[gen.name + "_proj"] = [get(t, a) for t, a in zip(gen.projections, template[gen.name + "_proj"])]
        p[gen.name + "_bn"] = [bn(b) for b in gen.bns]
    return p


def fp16x3_exponent_of(absmax):
    """csrc/common.cuh fp16x3_exponent_of: the power of two that puts max |x| into [2^10, 2^11)."""
    a = np.float32(absmax)
    if not (a > 0) or not (a < np.float32(3.0e38)):
        return 0
    ex = math.frexp(float(a))[1]
    return max(-100, min(100, 10 - (ex - 1)))


def oracle_grads(params, cfg, e1, rel, masks, dense):
    out = O.forward(params, cfg, e1, rel, True, masks, dense, np.float64)
    return out, O.backward(out, cfg)


def oracle_clip(model, g, clip):
    """tf.clip_by_global_norm over the oracle's gradients, split as the model's trainables are (IndexedSlices values for
    the sparse variables).  Returns ({name: clipped dense}, {name: (clipped values, indices)}, norm)."""
    dense = [n for n, _, _ in model.trainables if n not in model.sparse_vars]
    sparse = [n for n, _, _ in model.trainables if n in model.sparse_vars]
    vals = [g["_sparse"][n][0] for n in sparse]
    dc, sc, norm = O.clip_by_global_norm([tree_get(g, n) for n in dense], clip, sparse_values=[v for v, _ in vals])
    return dict(zip(dense, dc)), {n: (c, i) for n, c, (_, i) in zip(sparse, sc, vals)}, norm


def amsgrad_ref(pre, grad, grad_sq, cs, lr_t, bug_compat):
    """fp64 AMSGrad of one variable from its pre-step state (include/coper.h, coper_param_desc)."""
    th, vhat = pre["theta"].copy(), pre["vhat"].copy()
    m = v = None
    if grad_sq is not None:                          # IndexedSlices rule: the slots accumulate (both modes)
        m = B1 * pre["m"] + OMB1 * (grad * cs)
        v = B2 * pre["v"] + OMB2 * (grad_sq * cs * cs)
        vhat = np.maximum(vhat, v)
        th -= lr_t * m / (np.sqrt(vhat) + EPS)
    elif bug_compat:                                 # the reference as written: m, v never accumulate
        g = grad * cs
        vhat = np.maximum(vhat, g * g * OMB2)
        th -= lr_t * (g * OMB1) / (np.sqrt(vhat) + EPS)
    else:
        g = grad * cs
        m = B1 * pre["m"] + OMB1 * g
        v = B2 * pre["v"] + OMB2 * g * g
        vhat = np.maximum(vhat, v)
        th -= lr_t * m / (np.sqrt(vhat) + EPS)
    return th, m, v, vhat


def close_to_max(got, ref, rel):
    scale = np.abs(ref).max()
    return np.abs(got - ref).max() <= rel * scale if scale > 0 else not np.any(got)


def host(t):
    return t.detach().cpu().numpy().astype(np.float64)


def check_operand_copies(L, model, prec, amax_pre):
    """E_prep / P_prep after the step hold the operand form of the UPDATED variables."""
    d = model.ent_emb_size
    Pw = model.fc_weights.projections[-1]
    for name, theta, prep, rows in (("ent_emb", model.ent_emb, model.E_prep, model.shard.rows),
                                    (model._last_w_name, Pw, model.P_prep, Pw.shape[0] * model.F)):
        if prec != "fp16x3" or not model._emit_prepared:
            # bf16: RN copy; tf32x3: cvt.rna hi plane + exact lo plane; both with pitch d (or re-prepared outright)
            fresh = torch.zeros_like(prep)
            L.call("coper_prepare_operand", L.ptr(theta), rows, d, d, PREC[prec], L.ptr(fresh))
            torch.cuda.synchronize()
            assert torch.equal(prep, fresh), name
            continue
        n = rows * d
        raw = prep.cpu().numpy()
        hi, lo = raw[:2 * n].view(np.float16), raw[2 * n:4 * n].view(np.float16)
        trailer = raw[-(-n * 4 // 256) * 256:][:16].view(np.uint32)
        th = theta.detach().cpu().numpy().reshape(-1)
        e = int(trailer[:1].view(np.int32)[0])
        assert e == fp16x3_exponent_of(amax_pre[name]), (name, e, amax_pre[name])     # rolled from max |theta| before
        assert trailer[2] == np.abs(th).max().view(np.uint32), name                    # running max after the step
        a = th * np.float32(2.0 ** e)
        h = a.astype(np.float16)
        lo_ref = (a - h.astype(np.float32)).astype(np.float16)
        assert np.isfinite(hi).all() and np.isfinite(lo).all(), name
        assert np.array_equal(hi.view(np.uint16), h.view(np.uint16)), name
        assert np.array_equal(lo.view(np.uint16), lo_ref.view(np.uint16)), name
        dec = (hi.astype(np.float64) + lo.astype(np.float64)) * 2.0 ** -e
        assert np.abs(dec - th).max() <= 2.0 ** -21 * np.abs(th).max(), name


UPDATE_PARAMS = [(name, prec, bc, True) for name in UPDATE_CASES for prec in PREC for bc in (True, False)] + \
                [("ragged_mid", "tf32x3", True, False)]       # the default clip (5.0, inactive on these gradients)


@pytest.mark.parametrize("name,prec,bug_compat,low_clip", UPDATE_PARAMS)
def test_training_update_matches_fp64(L, monkeypatch, name, prec, bug_compat, low_clip):
    """STEPS full training steps on every engine; per step: the global norm (self-consistent and vs the oracle), the
    update (vs fp64 AMSGrad of the model's own gradients and clip factor), the operand copies, the scores of the updated
    model; after the last step the oracle's own trajectory."""
    import coper_b200.models as M
    kw, B = UPDATE_CASES[name]
    cfg = O.OracleConfig(**kw)
    params = O.init_params(cfg, seed=3, bias_noise=0.05)
    p64 = O.cast_params(params, np.float64)
    clip = M.CLIP_NORM
    e1, rel, _, rowptr, col = O.synthetic_batch(cfg, B, seed=59)
    if low_clip:         # about half the first step's norm (undropped estimate): the clip is active on every step
        _, g0 = oracle_grads(p64, cfg, e1, rel, None, O.csr_to_dense(rowptr, col, cfg.num_ent))
        clip = 0.5 * oracle_clip(_model_names(cfg), g0, 1.0)[2]
        monkeypatch.setattr(M, "CLIP_NORM", clip)    # baked into the captured step
    model = M.ConvE(descriptors(cfg, LR), conv_in_height=cfg.conv_in_height, prec=prec,
                    reference_bug_compat=bug_compat)
    model.load_variables(params)
    theta0 = {n: host(p) for n, p, _ in model.trainables}
    opt = O.AMSGradOracle(LR, reference_bug_compat=bug_compat)
    prepared = ("ent_emb", model._last_w_name)
    fp32_class = prec in FP32_CLASS
    for step in range(STEPS):
        e1, rel, e2, rowptr, col = O.synthetic_batch(cfg, B, seed=60 + step)
        e1[B // 2:] = e1[:B - B // 2]                   # duplicate heads: the scatter's segments
        dense = O.csr_to_dense(rowptr, col, cfg.num_ent)
        batch = batch_of(e1, rel, e2, rowptr, col)
        pre = {n: {"theta": host(p), "vhat": host(model.vhat[n]),
                   "m": host(model.m[n]) if n in model.m else None, "v": host(model.v[n]) if n in model.v else None}
               for n, p, _ in model.trainables}
        pre_params = params_of(model, params)
        amax_pre = {n: np.abs(pre[n]["theta"]).max() for n in prepared}
        model.train_step(batch)
        torch.cuda.synchronize()
        active = model._bufs[B].q.cpu().numpy() > 0          # the step's FC ReLU pattern (predict_all reuses q)
        cs, norm_dev = (float(x) for x in model.clip_out.cpu().numpy())
        lr_t = float(model.step_state[0].item())
        grads = {n: host(model.grads[n]) for n in pre}
        gsq = {n: host(model.grad_sq[n]) if n in model.sparse_vars else None for n in pre}
        # ---- the norm, from the model's own gradient buffers (any lost / doubled partial or delta shows here)
        sq = sum(float(gsq[n].sum()) if gsq[n] is not None else float((grads[n] ** 2).sum()) for n in pre)
        norm_own = math.sqrt(sq)
        assert abs(norm_dev - norm_own) <= 1e-6 * norm_own, (step, norm_dev, norm_own)
        assert abs(cs - clip / max(norm_own, clip)) <= 1e-6 * cs, (step, cs, clip, norm_own)
        assert cs < 1.0 if low_clip else cs == 1.0, (step, cs)
        # ---- the norm against the oracle's gradients at the same (pre-step) parameters and dropout masks
        masks = export_masks(model, cfg, B)
        out_pre, g_pre = oracle_grads(pre_params, cfg, e1, rel, masks, dense)
        norm_ref = oracle_clip(model, g_pre, clip)[2]
        assert abs(norm_dev - norm_ref) <= (1e-4 if fp32_class else 5e-2) * norm_ref, (step, norm_dev, norm_ref)
        # ---- the update, isolated from gradient error: fp64 AMSGrad of the model's gradients and clip factor
        for n, p, _ in model.trainables:
            th, m, v, vhat = amsgrad_ref(pre[n], grads[n], gsq[n], cs, lr_t, bug_compat)
            got = host(p)
            assert np.abs(got - th).max() <= 2.0 ** -21 * np.abs(th).max() + 1e-5 * lr_t, (step, n)
            assert close_to_max(host(model.vhat[n]), vhat, 1e-6), (step, n)
            if m is not None:
                assert close_to_max(host(model.m[n]), m, 1e-6), (step, n)
                assert close_to_max(host(model.v[n]), v, 1e-6), (step, n)
        if model.E_prep is not None:
            check_operand_copies(L, model, prec, amax_pre)
        # ---- the updated model scores from the updated parameters
        S = model.predict_all(batch).cpu().numpy()
        ref = O.forward(params_of(model, params), cfg, e1, rel, False, None, None, np.float64)["scores"]
        assert relerr(S, ref) < (1e-5 if fp32_class else 2e-2), (step, relerr(S, ref))
        rank, n_equal = model.filtered_ranks(batch)
        cnt, ne = O.rank_count(S, e2, dense)
        assert (rank.cpu().numpy() == cnt).all() and (n_equal.cpu().numpy() == ne).all(), step
        # ---- the oracle's own trajectory under the same clip and masks, and at the engine's FC ReLU pattern: a unit
        # whose pre-activation lies within rounding of 0 flips between fp32 and fp64, and the flip moves that query's
        # whole backward input (test_train_step_parity_tensor_pipe) - over several steps the trajectories would part
        # on the flips alone.  (Before the first update the device's parameters ARE the oracle's.)
        out = out_pre if step == 0 else O.forward(p64, cfg, e1, rel, True, masks, dense, np.float64)
        flips = int((active != (out["_cache"]["relu2"] > 0)).sum()) if fp32_class else 0    # bf16: direction only
        assert flips <= max(2, active.size // 500), (step, flips)
        if flips:
            out["_cache"]["relu2"] = active.astype(np.float64)
        g = g_pre if step == 0 and not flips else O.backward(out, cfg)
        dc, sc, _ = oracle_clip(model, g, clip)
        opt.apply({n: (tree_get(p64, n), c) for n, c in dc.items()},
                  sparse={n: (tree_get(p64, n), c, i) for n, (c, i) in sc.items()})
        for nm in ("Conv1BN", "FCBN"):
            p64[nm]["moving_mean"], p64[nm]["moving_var"] = out["moving"][nm]
    # conv1_bias is left out: its gradient is analytically 0 under batch-statistics BN and moves on rounding noise
    names = ["ent_emb", "pred_bias", model._last_w_name, model._last_b_name] + \
        (["rel_emb"] if model.rel_emb is not None else [])
    for n in names:
        got = host(dict((k, p) for k, p, _ in model.trainables)[n])
        ref = tree_get(p64, n).reshape(got.shape)
        if fp32_class:
            assert relerr(got, ref) < 1e-3, (n, relerr(got, ref))
        else:            # bf16 gradients: the direction of the whole update
            a, b = (got - theta0[n]).ravel(), (ref - theta0[n]).ravel()
            cos = float(a @ b / (np.linalg.norm(a) * np.linalg.norm(b) + 1e-30))
            assert cos > 0.9, (n, cos)


def _model_names(cfg):
    """The trainable split oracle_clip needs, without building a model (for choosing the clip before construction)."""
    names = ["ent_emb", "pred_bias"] + (["rel_emb"] if cfg.variant != "param_lookup" else []) + \
        ["conv1_weights", "conv1_bias"]
    if cfg.variant == "cpg":
        names += ["fc_weights/CPG/Projection%d" % i for i in range(len(cfg.context_rel_out) + 1)]
        names += ["fc_bias/CPG/Projection%d" % i for i in range(len(cfg.context_rel_out) + 1)]
    else:
        names += ["fc_weights", "fc_bias"]
    names += ["Conv1BN/gamma", "Conv1BN/beta", "FCBN/gamma", "FCBN/beta"]
    sparse = {"rel_emb"} if cfg.variant != "param_lookup" else {"fc_weights", "fc_bias"}
    return type("Names", (), {"trainables": [(n, None, None) for n in names], "sparse_vars": sparse})()
