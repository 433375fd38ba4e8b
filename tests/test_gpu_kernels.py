"""Per-kernel GPU parity through the C ABI at BASELINE shapes (WN18RR / FB15k-237 dims) and edge cases.

Checker = numpy fp64 restatements from ``oracle`` (small enough to finish in seconds) plus size-independent
properties (linearity, count identities, permutation invariance) at the larger sizes.
"""
import numpy as np
import pytest
import torch

from oracle import conve_oracle as O

pytestmark = pytest.mark.gpu


_ALIVE = []     # device tensors created inline as call arguments must outlive the (asynchronous) call


@pytest.fixture(autouse=True)
def _release_tensors():
    yield
    torch.cuda.synchronize()
    _ALIVE.clear()


def dev(a, dtype=None):
    t = torch.as_tensor(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    t = t.cuda()
    _ALIVE.append(t)
    return t


def relerr(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return np.abs(a - b).max() / (np.abs(b).max() + 1e-30)


@pytest.fixture(scope="module")
def L():
    from coper_b200 import _lib
    _lib.load()
    return _lib


def ws_buf(nbytes):
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device="cuda")


# ------------------------------------------------------------------------------------------ gather / scatter
def test_gather_rows_full_and_sharded(L):
    rng = np.random.default_rng(0)
    N, w, M = 1000, 200, 77
    tab = rng.normal(size=(N, w)).astype(np.float32)
    idx = rng.integers(0, N, M)
    out = torch.zeros(M, w, device="cuda")
    L.call("coper_gather_rows", L.ptr(dev(tab)), 0, N, w, L.ptr(dev(idx, torch.int64)), M, L.ptr(out))
    assert np.array_equal(out.cpu().numpy(), tab[idx])
    lo, hi = 256, 640
    L.call("coper_gather_rows", L.ptr(dev(tab[lo:hi])), lo, hi, w, L.ptr(dev(idx, torch.int64)), M, L.ptr(out))
    exp = np.where(((idx >= lo) & (idx < hi))[:, None], tab[idx], 0)
    assert np.array_equal(out.cpu().numpy(), exp)


@pytest.mark.parametrize("M,rows,w", [(512, 97, 200), (1, 5, 8), (4096, 11, 37), (300, 100000, 256),
                                      (20000, 5000, 64), (4097, 3, 200)])
def test_segscatter_deterministic_and_exact(L, M, rows, w):
    """M <= 4096 takes the sort-free path, larger M the radix-sort path; both sum in index order."""
    rng = np.random.default_rng(1)
    idx = rng.integers(0, rows, M)
    idx[: M // 3] = idx[0]                                         # a hub row
    src = rng.normal(size=(M, w)).astype(np.float32)
    base = rng.normal(size=(rows, w)).astype(np.float32)
    ws = ws_buf(L.load().coper_segscatter_workspace_bytes(M))
    outs = []
    for _ in range(2):
        dst = dev(base)
        L.call("coper_segscatter_add", L.ptr(dev(idx, torch.int64)), M, L.ptr(dev(src)), w, L.ptr(dst), 0, rows,
               L.ptr(ws), ws.numel())
        outs.append(dst.cpu().numpy())
    assert np.array_equal(outs[0], outs[1])
    exp = base.astype(np.float64)
    np.add.at(exp, idx, src.astype(np.float64))
    assert np.abs(outs[0] - exp).max() < 1e-4 * max(1.0, np.abs(exp).max())
    # sharded: only rows in [lo, hi) are touched
    lo, hi = rows // 4, rows // 4 + max(1, rows // 2)
    dst = dev(base[lo:hi])
    L.call("coper_segscatter_add", L.ptr(dev(idx, torch.int64)), M, L.ptr(dev(src)), w, L.ptr(dst), lo, hi,
           L.ptr(ws), ws.numel())
    assert np.abs(dst.cpu().numpy() - exp[lo:hi]).max() < 1e-4 * max(1.0, np.abs(exp).max())
    if M <= 4096:      # sum + sum of squares in one pass (IndexedSlices bookkeeping)
        d1, d2 = dev(base), torch.zeros(rows, w, device="cuda")
        L.call("coper_segscatter_add_sq", L.ptr(dev(idx, torch.int64)), M, L.ptr(dev(src)), w, L.ptr(d1), L.ptr(d2),
               0, rows)
        assert np.array_equal(d1.cpu().numpy(), outs[0])
        sq = np.zeros((rows, w))
        np.add.at(sq, idx, src.astype(np.float64) ** 2)
        assert np.abs(d2.cpu().numpy() - sq).max() < 1e-4 * max(1.0, np.abs(sq).max())


# ------------------------------------------------------------------------------------------ conv
@pytest.mark.parametrize("B,H,W", [(5, 10, 20), (64, 16, 16), (3, 10, 4)])
def test_conv_fwd_bwd(L, B, H, W):
    rng = np.random.default_rng(2)
    KH = KW = 3
    C = 32
    OH, OW = H - 2, W - 2
    x = rng.normal(size=(B, H, W))
    wc = rng.normal(size=(KH, KW, C))
    bc = rng.normal(size=C)
    z = torch.zeros(B, OH * OW * C, device="cuda")
    L.call("coper_conv_fwd", L.ptr(dev(x, torch.float32)), B, H, W, L.ptr(dev(wc, torch.float32)),
           L.ptr(dev(bc, torch.float32)), KH, KW, C, 0, L.ptr(z))
    Z = O._conv_valid(x, wc) + bc
    assert relerr(z.cpu().numpy().reshape(Z.shape), Z) < 1e-5
    dz = rng.normal(size=Z.shape)
    dx = torch.zeros(B, H * W, device="cuda")
    dwp = torch.zeros(B, KH * KW * C, device="cuda")
    dbp = torch.zeros(B, C, device="cuda")
    L.call("coper_conv_bwd", L.ptr(dev(dz, torch.float32)), L.ptr(dev(x, torch.float32)), B, H, W,
           L.ptr(dev(wc, torch.float32)), KH, KW, C, 0, L.ptr(dx), L.ptr(dwp), L.ptr(dbp))
    dW = np.zeros_like(wc)
    dX = np.zeros_like(x)
    for i in range(KH):
        for j in range(KW):
            dW[i, j] = np.einsum("bhw,bhwc->c", x[:, i:i + OH, j:j + OW], dz)
            dX[:, i:i + OH, j:j + OW] += dz @ wc[i, j]
    assert relerr(dx.cpu().numpy().reshape(dX.shape), dX) < 1e-5
    assert relerr(dwp.cpu().numpy().sum(0).reshape(dW.shape), dW) < 1e-4
    assert relerr(dbp.cpu().numpy().sum(0), dz.sum(axis=(0, 1, 2))) < 1e-4


# ------------------------------------------------------------------------------------------ fused CPG-FC
def _cpg_ref(c, f, P, cb, Pb):
    B, dc = c.shape
    F = f.shape[1]
    d = Pb.shape[1]
    kr = (c[:, :, None] * f[:, None, :]).reshape(B, dc * F)
    return kr @ P.reshape(dc * F, d) + cb @ Pb


def _bf16r(x):
    return torch.as_tensor(np.asarray(x), dtype=torch.float32).to(torch.bfloat16).to(torch.float64).numpy()


@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "fp16x3", "bf16"])
@pytest.mark.parametrize("B,dc,F,d", [(512, 8, 4608, 200), (7, 5, 192, 40), (130, 3, 1000, 72), (64, 32, 512, 200),
                                      (512, 32, 6272, 256)])
def test_cpg_fc_fwd_bwd(L, B, dc, F, d, prec):
    """fused generate-and-apply + backward.  fp32 (CUDA cores) and tf32x3 (tcgen05, 3-term compensated) are held to
    the fp32 bar; bf16 (tcgen05) is compared with fp64 arithmetic on the bf16-rounded operands it actually consumes
    (f, P, dy and c*dy are rounded to bf16; c scales in fp32)."""
    p = L.PREC[prec]
    if prec != "fp32" and F % 32:
        pytest.skip("tensor-pipe CPG kernels need F % 32 == 0 (F = OH*OW*32 in the model)")
    rng = np.random.default_rng(3)
    c = rng.normal(size=(B, dc))
    f = np.maximum(rng.normal(size=(B, F)), 0)
    P = rng.normal(size=(dc, F * d)) * 0.01
    cb = rng.normal(size=(B, dc))
    Pb = rng.normal(size=(dc, d))
    lib = L.load()
    ws = ws_buf(max(lib.coper_cpg_fc_fwd_workspace_bytes(B, dc, F, d, p), lib.coper_cpg_fc_bwd_workspace_bytes(B, dc, F, d, p)))
    c, f, P, cb, Pb = (a.astype(np.float32).astype(np.float64) for a in (c, f, P, cb, Pb))
    tc, tf, tP, tcb, tPb = (dev(a, torch.float32) for a in (c, f, P, cb, Pb))
    y = torch.full((B, d), float("nan"), device="cuda")
    L.call("coper_cpg_fc_fwd", L.ptr(tc), L.ptr(tf), L.ptr(tP), None, L.ptr(tcb), L.ptr(tPb), B, dc, F, d, dc, 1.0, None, 0,
           L.ptr(y), L.ptr(ws), ws.numel(), p)
    dy = rng.normal(size=(B, d)).astype(np.float32).astype(np.float64)
    if prec == "bf16":
        fr, Pr = _bf16r(f), _bf16r(P)
    else:
        fr, Pr = f, P
    yr = _cpg_ref(c, fr, Pr, cb, Pb)
    assert relerr(y.cpu().numpy(), yr) < 1e-5
    if prec == "bf16":
        assert relerr(y.cpu().numpy(), _cpg_ref(c, f, P, cb, Pb)) < 1e-2
    dP = torch.zeros(dc, F * d, device="cuda")
    dPb = torch.zeros(dc, d, device="cuda")
    df = torch.zeros(B, F, device="cuda")
    dcw = torch.zeros(B, dc, device="cuda")
    dcb = torch.zeros(B, dc, device="cuda")
    L.call("coper_cpg_fc_bwd", L.ptr(tc), L.ptr(tf), L.ptr(tP), None, L.ptr(tcb), L.ptr(tPb), L.ptr(dev(dy, torch.float32)),
           B, dc, F, d, dc, L.ptr(dP), L.ptr(dPb), L.ptr(df), L.ptr(dcw), L.ptr(dcb), L.ptr(ws), ws.numel(), p,
           int(prec != "fp32"))
    dyr = _bf16r(dy) if prec == "bf16" else dy
    P3 = Pr.reshape(dc, F, d)
    T = np.einsum("bj,kij->bki", dyr, P3)
    assert relerr(df.cpu().numpy(), np.einsum("bk,bki->bi", c, T)) < 2e-5
    assert relerr(dcw.cpu().numpy(), np.einsum("bi,bki->bk", f, T)) < 2e-5       # f enters the row sums in fp32
    if prec == "bf16":
        dyc = _bf16r((c[:, :, None] * dy[:, None, :]).astype(np.float32))       # [B, dc, d] rounded as consumed
        dPr = np.einsum("bi,bkj->kij", fr, dyc).reshape(dc, F * d)
    else:
        kr = (c[:, :, None] * f[:, None, :]).reshape(B, dc * F)
        dPr = (kr.T @ dy).reshape(dc, F * d)
    assert relerr(dP.cpu().numpy(), dPr) < 2e-5
    assert relerr(dPb.cpu().numpy(), cb.T @ dy) < 2e-5
    assert relerr(dcb.cpu().numpy(), dy @ Pb.T) < 2e-5


def test_cpg_fc_fb15k_shape_linearity(L):
    """FB15k-237 shape (dc=32, F=4608, d=200, B=512): y is linear in c and in f (size-independent property)."""
    B, dc, F, d = 512, 32, 4608, 200
    g = torch.Generator(device="cuda").manual_seed(0)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g)
    c1, c2, f, P = r(B, dc), r(B, dc), r(B, F).clamp_(min=0), r(dc, F * d) * 0.01
    cb, Pb = torch.zeros(B, dc, device="cuda"), torch.zeros(dc, d, device="cuda")
    lib = L.load()
    ws = ws_buf(lib.coper_cpg_fc_fwd_workspace_bytes(B, dc, F, d, 0))

    def run(c, ff):
        y = torch.zeros(B, d, device="cuda")
        L.call("coper_cpg_fc_fwd", L.ptr(c), L.ptr(ff), L.ptr(P), None, L.ptr(cb), L.ptr(Pb), B, dc, F, d, dc, 1.0, None, 0,
               L.ptr(y), L.ptr(ws), ws.numel(), 0)
        return y
    y1, y2, y12 = run(c1, f), run(c2, f), run((c1 + 2 * c2).contiguous(), f)
    assert relerr(y12.cpu().numpy(), (y1 + 2 * y2).cpu().numpy()) < 2e-5
    # spot-check 8 rows against fp64
    rows = [0, 1, 77, 128, 255, 300, 510, 511]
    yr = _cpg_ref(c1[rows].double().cpu().numpy(), f[rows].double().cpu().numpy(), P.double().cpu().numpy(),
                  cb[rows].double().cpu().numpy(), Pb.double().cpu().numpy())
    assert relerr(y1[rows].cpu().numpy(), yr) < 1e-5


# ------------------------------------------------------------------------------------------ scorer + BCE
@pytest.mark.parametrize("B,N,d", [(512, 40943, 200), (7, 97, 40), (130, 1003, 200), (33, 5000, 256)])
def test_score1n_fwd_and_bce(L, B, N, d):
    rng = np.random.default_rng(4)
    q = np.maximum(rng.normal(size=(B, d)), 0)
    E = rng.uniform(-0.05, 0.05, size=(N, d))
    bias = rng.normal(size=N) * 0.1
    ld = -(-N // 32) * 32
    tq, tE, tb = dev(q, torch.float32), dev(E, torch.float32), dev(bias, torch.float32)
    S = torch.zeros(B, ld, device="cuda")
    L.call("coper_score1n_fwd", L.ptr(tq), L.ptr(tE), L.ptr(tb), B, N, d, L.ptr(S), ld, None, 0, 0)
    Sr = q.astype(np.float32).astype(np.float64) @ E.astype(np.float32).astype(np.float64).T + bias.astype(np.float32)
    assert relerr(S[:, :N].cpu().numpy(), Sr) < 1e-5
    # BCE + gradient
    cfg = O.OracleConfig(num_ent=N, num_rel=2, ent_emb_size=d, rel_emb_size=2, conv_in_height=d // 4 if d % 10 else 10)
    _, _, _, rowptr, col = O.synthetic_batch(cfg, B, seed=9, mean_pos=4.0)
    words = -(-N // 32)
    bits = torch.zeros(B, words, dtype=torch.int32, device="cuda")
    L.call("coper_csr_to_bits", L.ptr(dev(rowptr, torch.int32)), L.ptr(dev(col, torch.int32)), B, 0, N, L.ptr(bits))
    z = O.csr_to_dense(rowptr, col, N, np.float64)
    pos = np.float32(np.float32(0.9) + np.float32(1.0 / N))
    neg = np.float32(1.0 / N)
    zs = np.where(z > 0, np.float64(pos), np.float64(neg))
    lib = L.load()
    ws = ws_buf(lib.coper_score1n_bce_workspace_bytes(B, N, d, 0))
    G = torch.zeros(B, ld, device="cuda")
    loss = torch.zeros(1, dtype=torch.float64, device="cuda")
    dq, dE, db = torch.zeros(B, d, device="cuda"), torch.zeros(N, d, device="cuda"), torch.zeros(N, device="cuda")
    inv = 1.0 / (B * N)
    L.call("coper_score1n_bce_fwd_bwd", L.ptr(tq), L.ptr(tE), None, L.ptr(tb), L.ptr(bits), B, N, d, float(pos), float(neg),
           inv, L.ptr(loss), L.ptr(G), ld, L.ptr(dq), L.ptr(dE), L.ptr(db), L.ptr(ws), ws.numel(), 0)
    el = np.maximum(Sr, 0) - Sr * zs + np.log1p(np.exp(-np.abs(Sr)))
    Gr = (O.sigmoid(Sr) - zs) * inv
    assert abs(loss.item() - el.sum()) < 1e-6 * el.sum()
    assert relerr(G[:, :N].cpu().numpy(), Gr) < 1e-5
    q32, E32 = q.astype(np.float32).astype(np.float64), E.astype(np.float32).astype(np.float64)
    assert relerr(dq.cpu().numpy(), Gr @ E32) < 1e-4
    assert relerr(dE.cpu().numpy(), Gr.T @ q32) < 1e-4
    assert relerr(db.cpu().numpy(), Gr.sum(0)) < 1e-4
    # dense multi-hot schema builds the same bit rows
    bits2 = torch.zeros_like(bits)
    L.call("coper_dense_to_bits", L.ptr(dev(z, torch.float32)), B, N, L.ptr(bits2))
    assert torch.equal(bits, bits2)


# ------------------------------------------------------------------------------------------ filtered rank
@pytest.mark.parametrize("B,N", [(512, 40943), (3, 5), (64, 1000003), (17, 4096), (1, 33)])
def test_filtered_rank_bit_exact(L, B, N):
    rng = np.random.default_rng(5)
    ld = -(-N // 32) * 32
    S = rng.normal(size=(B, ld)).astype(np.float32)
    if N >= 4096:
        S[:, ::7] = S[:, [0]]                                    # plenty of exact ties
    e2 = rng.integers(0, N, B)
    filt = rng.random((B, N)) < 0.03
    filt[np.arange(B), e2] = True                                # the gold is always a known true tail
    words = -(-N // 32)
    packed = np.zeros((B, words * 32), bool)
    packed[:, :N] = filt
    bits = np.packbits(packed.reshape(B, words, 32), axis=2, bitorder="little").view(np.uint32).reshape(B, words)
    tS, te2, tb = dev(S), dev(e2, torch.int64), dev(bits.view(np.int32))
    gold = torch.zeros(B, device="cuda")
    L.call("coper_gold_scores", L.ptr(tS), ld, B, N, L.ptr(te2), 0, L.ptr(gold))
    assert np.array_equal(gold.cpu().numpy(), S[np.arange(B), e2])
    ng = torch.zeros(B, dtype=torch.int32, device="cuda")
    ne = torch.zeros(B, dtype=torch.int32, device="cuda")
    L.call("coper_filtered_rank", L.ptr(tS), ld, B, N, L.ptr(te2), 0, L.ptr(gold), L.ptr(tb), L.ptr(ng), L.ptr(ne))
    rc, eq = O.rank_count(S[:, :N], e2, filt.astype(np.float32))
    assert np.array_equal(ng.cpu().numpy() + 1, rc)
    assert np.array_equal(ne.cpu().numpy(), eq)
    # sharding property: integer partial counts over any split of the entity range add up exactly
    cut = (N // 3) // 32 * 32
    if cut > 0:
        ng2 = torch.zeros(B, dtype=torch.int32, device="cuda")
        ne2 = torch.zeros(B, dtype=torch.int32, device="cuda")
        for lo, hi in ((0, cut), (cut, N)):
            Ss = dev(np.ascontiguousarray(S[:, lo:hi]))
            fb = np.zeros((B, -(-(hi - lo) // 32) * 32), bool)
            fb[:, :hi - lo] = filt[:, lo:hi]
            bs = np.packbits(fb.reshape(B, -1, 32), axis=2, bitorder="little").view(np.uint32).reshape(B, -1)
            L.call("coper_filtered_rank", L.ptr(Ss), hi - lo, B, hi - lo, L.ptr(te2), lo, L.ptr(gold),
                   L.ptr(dev(bs.view(np.int32))), L.ptr(ng2), L.ptr(ne2))
        assert torch.equal(ng, ng2) and torch.equal(ne, ne2)


# ------------------------------------------------------------------------------------------ BN / optimizer pieces
def test_bn_train_and_eval_paths(L):
    rng = np.random.default_rng(6)
    R, C = 73728 // 8, 32
    x = rng.normal(1.0, 2.0, size=(R, C))
    bn = {"gamma": rng.normal(1, 0.1, C), "beta": rng.normal(0, 0.1, C), "moving_mean": rng.normal(0, 0.1, C),
          "moving_var": rng.uniform(0.5, 1.5, C)}
    lib = L.load()
    nch = lib.coper_colstats_chunks(R)
    tx = dev(x, torch.float32)
    part = torch.zeros(nch * C * 2, device="cuda")
    t = {k: dev(v, torch.float32) for k, v in bn.items()}
    a, b, mean, inv = (torch.zeros(C, device="cuda") for _ in range(4))
    out = torch.zeros(R, C, device="cuda")
    for use_batch in (1, 0):
        L.call("coper_colstats", L.ptr(tx), R, C, L.ptr(part))
        L.call("coper_bn_finalize", L.ptr(part), nch, R, C, L.ptr(t["gamma"]), L.ptr(t["beta"]),
               L.ptr(t["moving_mean"]), L.ptr(t["moving_var"]), 0.9, 1e-3, use_batch, 0, 1, L.ptr(a), L.ptr(b),
               L.ptr(mean), L.ptr(inv))
        L.call("coper_bn_act_fwd", L.ptr(tx), R, C, L.ptr(a), L.ptr(b), 1, 1.0, None, 0, L.ptr(out))
        ref, cache, mm, mv = O._bn_forward(x, bn, bool(use_batch), True, 0.9)
        assert relerr(out.cpu().numpy(), np.maximum(ref, 0)) < 1e-5


def test_amsgrad_and_clip(L):
    rng = np.random.default_rng(7)
    n = 100003
    th, g = rng.normal(size=n).astype(np.float32), (rng.normal(size=n) * 3).astype(np.float32)
    tth, tg = dev(th), dev(g)
    vhat = torch.zeros(n, device="cuda")
    part = torch.zeros(256, dtype=torch.float64, device="cuda")
    clip = torch.zeros(2, device="cuda")
    state = torch.tensor([0.0, 0.9, 0.999, 0.0], device="cuda")
    seed = torch.zeros(1, dtype=torch.int64, device="cuda")
    L.call("coper_step_state_advance", L.ptr(state), L.ptr(seed), 1e-3, 0.9, 0.999)
    L.call("coper_sumsq", L.ptr(tg), n, 0, L.ptr(part))
    L.call("coper_clip_scale", L.ptr(part), 1, 5.0, L.ptr(clip))
    norm = np.sqrt((g.astype(np.float64) ** 2).sum())
    assert abs(clip[1].item() - norm) < 1e-6 * norm
    assert abs(clip[0].item() - 5.0 / norm) < 1e-6
    L.call("coper_amsgrad_step", L.ptr(tth), L.ptr(tg), None, None, L.ptr(vhat), n, L.ptr(state), 0.9, 0.999, 1e-8,
           L.ptr(clip), 1)
    opt = O.AMSGradOracle(1e-3)
    th64 = th.astype(np.float64)
    opt.apply({"x": (th64, g.astype(np.float64) * (5.0 / norm))})
    assert relerr(tth.cpu().numpy(), th64) < 1e-6
    assert seed.item() == 1 and abs(state[1].item() - 0.81) < 1e-6


def test_sgemm_all_layouts(L):
    rng = np.random.default_rng(8)
    M, N, K = 130, 77, 301
    A, Bm = rng.normal(size=(M, K)), rng.normal(size=(K, N))
    ref = A @ Bm
    for ta in (0, 1):
        for tb in (0, 1):
            a = dev(A.T if ta else A, torch.float32).contiguous()
            b = dev(Bm.T if tb else Bm, torch.float32).contiguous()
            c = torch.zeros(M, N, device="cuda")
            L.call("coper_sgemm", ta, tb, M, N, K, L.ptr(a), a.shape[1], L.ptr(b), b.shape[1], L.ptr(c), N, 0)
            assert relerr(c.cpu().numpy(), ref) < 1e-5


# ------------------------------------------------------------------------------------------ multi-tensor clip + AMSGrad
@pytest.mark.parametrize("bug_compat", [1, 0])
def test_multi_tensor_optimizer_matches_per_tensor(L, bug_compat):
    """coper_mt_sumsq / coper_clip_scale_n / coper_mt_amsgrad == the per-variable kernels, bit for bit, and the
    operand copies they emit == coper_prepare_operand of the updated variable."""
    lib = L.load()
    g = torch.Generator(device="cuda").manual_seed(1)
    shapes = [(40943, 200), (1,), (16384,), (16385,), (8, 4608 * 40), (3, 3, 1, 32), (200,), (22, 8)]
    SPARSE = 7                                   # the last tensor plays rel_emb: IndexedSlices rule
    th = [torch.randn(*s, device="cuda", generator=g) for s in shapes]
    gr = [torch.randn(*s, device="cuda", generator=g) * 3 for s in shapes]
    vh = [torch.rand(*s, device="cuda", generator=g) for s in shapes]
    m = [torch.randn(*s, device="cuda", generator=g) for s in shapes]
    v = [torch.rand(*s, device="cuda", generator=g) for s in shapes]
    th2, vh2, m2, v2 = ([t.clone() for t in x] for x in (th, vh, m, v))
    prep = {0: (1, torch.zeros(lib.coper_prepared_bytes(40943, 200, 1), dtype=torch.uint8, device="cuda")),
            4: (2, torch.zeros(lib.coper_prepared_bytes(8 * 4608, 40, 2), dtype=torch.uint8, device="cuda"))}
    desc = np.zeros(len(shapes), dtype=L.PARAM_DESC)
    chunks, offs = [], [0]
    for i in range(len(shapes)):
        desc[i]["theta"], desc[i]["grad"], desc[i]["vhat"] = th[i].data_ptr(), gr[i].data_ptr(), vh[i].data_ptr()
        desc[i]["m"], desc[i]["v"], desc[i]["n"] = m[i].data_ptr(), v[i].data_ptr(), th[i].numel()
        if i in prep:
            desc[i]["prepared"], desc[i]["prepared_prec"] = prep[i][1].data_ptr(), prep[i][0]
        if i == SPARSE:
            gsq = torch.rand(*shapes[i], device="cuda", generator=g) * 9
            desc[i]["grad_sq"], desc[i]["mode"] = gsq.data_ptr(), 1
        chunks += [(i, c) for c in range(max(1, -(-th[i].numel() // L.MT_CHUNK)))]
        offs.append(len(chunks))
    d_desc = torch.from_numpy(desc.view(np.uint8).copy()).cuda()
    d_chunks, d_offs = torch.tensor(chunks, dtype=torch.int32).cuda(), torch.tensor(offs, dtype=torch.int32).cuda()
    part = torch.zeros(len(chunks), dtype=torch.float64, device="cuda")
    sums = torch.zeros(len(shapes), dtype=torch.float64, device="cuda")
    state = torch.tensor([0.0, 0.9, 0.999, 0.0], device="cuda")
    L.call("coper_step_state_advance", L.ptr(state), None, 1e-2, 0.9, 0.999)
    clip = torch.zeros(2, device="cuda")
    L.call("coper_mt_sumsq", L.ptr(d_desc), len(shapes), L.ptr(d_chunks), len(chunks), L.ptr(d_offs), L.ptr(part), L.ptr(sums))
    ref = np.array([float((x.double() ** 2).sum().item()) for x in gr])
    ref[SPARSE] = float(gsq.double().sum().item())            # slice-wise norm of an IndexedSlices gradient
    assert np.allclose(sums.cpu().numpy(), ref, rtol=1e-6)
    L.call("coper_clip_scale_n", L.ptr(sums), len(shapes), 5.0, L.ptr(clip))
    norm = np.sqrt(ref.sum())
    assert abs(clip[1].item() - norm) < 1e-5 * norm and abs(clip[0].item() - 5.0 / max(norm, 5.0)) < 1e-6
    L.call("coper_mt_amsgrad", L.ptr(d_desc), L.ptr(d_chunks), len(chunks), L.ptr(state), 0.9, 0.999, 1e-8, L.ptr(clip),
           bug_compat)
    # IndexedSlices rule (utils/amsgrad.py:161-189) against a torch restatement
    cs, lr_t = clip[0].item(), state[0].item()
    m_ref = m2[SPARSE] * 0.9 + gr[SPARSE] * cs * 0.1
    v_ref = v2[SPARSE] * 0.999 + gsq * cs * cs * 0.001
    vh_ref = torch.maximum(vh2[SPARSE], v_ref)
    th_ref = th2[SPARSE] - lr_t * m_ref / (vh_ref.sqrt() + 1e-8)
    assert torch.allclose(m[SPARSE], m_ref, rtol=1e-6, atol=1e-7) and torch.allclose(v[SPARSE], v_ref, rtol=1e-6, atol=1e-7)
    assert torch.allclose(vh[SPARSE], vh_ref, rtol=1e-6, atol=1e-7) and torch.allclose(th[SPARSE], th_ref, rtol=1e-6, atol=1e-6)
    for i in range(len(shapes) - 1):
        L.call("coper_amsgrad_step", L.ptr(th2[i]), L.ptr(gr[i]), L.ptr(m2[i]), L.ptr(v2[i]), L.ptr(vh2[i]),
               th2[i].numel(), L.ptr(state), 0.9, 0.999, 1e-8, L.ptr(clip), bug_compat)
        assert torch.equal(th[i], th2[i]) and torch.equal(vh[i], vh2[i]), i
        if not bug_compat:
            assert torch.equal(m[i], m2[i]) and torch.equal(v[i], v2[i]), i
    for i, (rows, cols) in ((0, (40943, 200)), (4, (8 * 4608, 40))):
        pr, buf = prep[i]
        chk = torch.zeros_like(buf)
        L.call("coper_prepare_operand", L.ptr(th[i]), rows, cols, cols, pr, L.ptr(chk))
        n_bytes = rows * cols * (2 if pr == 1 else 8)
        assert torch.equal(buf[:n_bytes], chk[:n_bytes]), i


def test_reduce_partials_fixed_order(L):
    rng = np.random.default_rng(0)
    # (4, 1 << 20) / (8, 65536): the few-slabs float4 path (dbias of a sharded table); (4, 65538): n % 4 != 0 -> general path
    for S, n in ((37, 102400), (512, 288), (1, 5), (16, 40943), (144, 4096), (4, 1 << 20), (8, 65536), (4, 65538)):
        x = rng.normal(size=(S, n)).astype(np.float32)
        out = torch.full((n,), 7.0, device="cuda")
        L.call("coper_reduce_partials", L.ptr(dev(x)), S, n, 0.5, 1, L.ptr(out))
        ref = 7.0 + 0.5 * x.astype(np.float64).sum(0)
        assert np.abs(out.cpu().numpy() - ref).max() < 1e-5 * max(1.0, np.abs(ref).max())


@pytest.mark.parametrize("N,L,needed", [(5000, 100, 9), (14, 10, 3), (200, 200, 18), (70001, 1000, 90)])
def test_sample_labels_bit_exact_and_well_formed(N, L, needed):
    """coper_sample_labels (data.py:228-277 on the device) vs the NumPy restatement, plus the properties the reference's
    sampler guarantees: positives first (all of them, or the computed share), sampled entities distinct, labels ==
    membership in the row's true tails."""
    from coper_b200 import _lib as L_
    from oracle import dropout_hash as DH
    lib = L_.load()
    rng = np.random.default_rng(N + L)
    B = 96
    k = np.minimum(rng.geometric(0.2, B), N)
    k[:6] = [0, 1, min(needed, N), min(needed + 1, N), min(60, N), min(1500, N)]     # empty row ... > 1024 positives
    rowptr = np.zeros(B + 1, np.int32)
    rowptr[1:] = np.cumsum(k)
    col = np.concatenate([rng.choice(N, int(kk), replace=False) for kk in k]).astype(np.int32)
    trp, tcol = torch.as_tensor(rowptr).cuda(), torch.as_tensor(col).cuda()
    for seed in (1, 987654321012345):
        sd = torch.tensor([seed], dtype=torch.int64, device="cuda")
        lookup = torch.full((B, L), -1, dtype=torch.int32, device="cuda")
        labels = torch.full((B, L), -1.0, device="cuda")
        L_.call("coper_sample_labels", L_.ptr(trp), L_.ptr(tcol), B, N, L, needed, L_.ptr(sd), DH.SALT_SAMPLE,
                L_.ptr(lookup), L_.ptr(labels))
        lk, lab = lookup.cpu().numpy(), labels.cpu().numpy()
        ref_lk, ref_lab = DH.sample_labels(rowptr, col, N, L, needed, seed)
        assert np.array_equal(lk, ref_lk) and np.array_equal(lab, ref_lab)
        for b in range(B):
            pos = col[rowptr[b]:rowptr[b + 1]]
            P = len(pos)
            n_pos = P if P <= needed else L - min(L - needed, N)
            n_pos = min(n_pos, P, L)
            assert set(lk[b, :n_pos].tolist()) <= set(pos.tolist()) and len(set(lk[b, :n_pos].tolist())) == n_pos
            neg = lk[b, n_pos:]
            assert len(set(neg.tolist())) == L - n_pos and neg.min(initial=0) >= 0 and neg.max(initial=0) < N
            assert np.array_equal(lab[b], np.isin(lk[b], pos).astype(np.float32) if P else np.zeros(L, np.float32))
    # the sampled entities are uniform over [0, N): chi-square of their histogram over all rows and 20 seeds
    if N == 5000:
        cnt = np.zeros(N)
        for seed in range(20):
            sd = torch.tensor([seed * 104729 + 7], dtype=torch.int64, device="cuda")
            L_.call("coper_sample_labels", L_.ptr(trp), L_.ptr(tcol), B, N, L, needed, L_.ptr(sd), DH.SALT_SAMPLE,
                    L_.ptr(lookup), L_.ptr(labels))
            lk = lookup.cpu().numpy()
            for b in range(B):
                P = int(k[b])
                n_pos = min(P if P <= needed else L - min(L - needed, N), P, L)
                np.add.at(cnt, lk[b, n_pos:], 1)
        e = cnt.sum() / N
        chi2 = ((cnt - e) ** 2 / e).sum()
        assert abs(chi2 - (N - 1)) < 6 * np.sqrt(2 * (N - 1)), chi2


@pytest.mark.parametrize("B,dc,F,d,prec", [(64, 8, 128, 64, "auto"), (33, 5, 50, 300, "auto"), (130, 6, 96, 200, "bf16"),
                                           (16, 3, 64, 800 // 4, "fp32")])
def test_generate_and_apply_autograd_matches_torch_einsum(B, dc, F, d, prec):
    """coper_b200.generate_apply (the ConvE path's fused kernels as a torch op) vs the materialising formulation of
    CoPER_MINERVA/src/rl/graph_search/pn.py:125 — einsum('ij,ijk->ik', X, reshape(Q @ P, [B, F, d])) + Q @ Pb — and
    its autograd gradients, in fp64 torch."""
    from coper_b200.generate_apply import generate_and_apply
    g = torch.Generator().manual_seed(B + F)
    Q = torch.randn(B, dc, generator=g)
    X = torch.relu(torch.randn(B, F, generator=g))
    P = (torch.rand(dc, F * d, generator=g) - 0.5) * 0.2
    Pb = (torch.rand(dc, d, generator=g) - 0.5) * 0.2
    dY = torch.randn(B, d, generator=g)
    ref_in = [t.double().requires_grad_(True) for t in (Q, X, P, Pb)]
    q64, x64, p64, pb64 = ref_in
    y_ref = torch.einsum("ij,ijk->ik", x64, (q64 @ p64).reshape(B, F, d)) + q64 @ pb64
    y_ref.backward(dY.double())
    dev_in = [t.cuda().requires_grad_(True) for t in (Q, X, P, Pb)]
    qd, xd, pd, pbd = dev_in
    y = generate_and_apply(qd, xd, pd, pbd, prec=prec)
    y.backward(dY.cuda())
    tol = 5e-2 if prec == "bf16" else 2e-5
    assert relerr(y.detach().cpu().numpy(), y_ref.detach().numpy()) < tol
    for got, ref in zip(dev_in, ref_in):
        assert relerr(got.grad.cpu().numpy(), ref.grad.numpy()) < (5e-2 if prec == "bf16" else 1e-4)
    # no bias term
    y0 = generate_and_apply(qd.detach(), xd.detach(), pd.detach(), prec=prec)
    y0_ref = torch.einsum("ij,ijk->ik", x64.detach(), (q64.detach() @ p64.detach()).reshape(B, F, d))
    assert relerr(y0.cpu().numpy(), y0_ref.numpy()) < tol
