"""The single-launch forms of the small steps around the tensor-pipe kernels (round 2: the WN18RR-sized step is a
chain of ~45 dependent launches, so every launch removed from the chain is step time).  Each merged entry point must
give the SAME BITS as the sequence of calls it replaces - the summation orders are part of the contract - and the
sequence itself is checked against numpy / the oracle in test_gpu_kernels.py.  (Exception: the single-launch batch-norm
statistics add the same chunk partials in a different fixed order - fp64, rounded once - and are compared at 2e-6.)
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

_ALIVE = []


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


@pytest.fixture(scope="module")
def L():
    from coper_b200 import _lib
    _lib.load()
    return _lib


def same_bits(a, b):
    return np.array_equal(a.detach().cpu().numpy().view(np.uint32 if a.dtype == torch.float32 else np.uint64),
                          b.detach().cpu().numpy().view(np.uint32 if b.dtype == torch.float32 else np.uint64))


# ------------------------------------------------------------------------------------------ lookups + step state
@pytest.mark.parametrize("with_rel,advance", [(True, True), (True, False), (False, True), (False, False)])
def test_gather_rows2_equals_separate_calls(L, with_rel, advance):
    rng = np.random.default_rng(1)
    N, d, R, dr, B = 5000, 200, 22, 96, 513
    E = dev(rng.normal(size=(N, d)).astype(np.float32))
    Rt = dev(rng.normal(size=(R, dr)).astype(np.float32))
    e1 = dev(rng.integers(0, N, B), torch.int64)
    rel = dev(rng.integers(0, R, B), torch.int64)
    lo, hi = 1000, 4000                                 # sharded head lookup: rows outside are zero-filled
    x_ref, r_ref = torch.empty(B, d, device="cuda"), torch.empty(B, dr, device="cuda")
    L.call("coper_gather_rows", L.ptr(E[lo:]), lo, hi, d, L.ptr(e1), B, L.ptr(x_ref))
    L.call("coper_gather_rows", L.ptr(Rt), 0, R, dr, L.ptr(rel), B, L.ptr(r_ref))
    st_ref = dev(np.array([0.0, 0.9, 0.999, 0.0], np.float32))
    seed_ref = dev(np.array([77], np.uint64).view(np.int64), torch.int64)
    st, seed = st_ref.clone(), seed_ref.clone()
    L.call("coper_step_state_advance", L.ptr(st_ref), L.ptr(seed_ref), 0.003, 0.9, 0.999)
    x, r = torch.full((B, d), 7.0, device="cuda"), torch.full((B, dr), 7.0, device="cuda")
    L.call("coper_gather_rows2", L.ptr(E[lo:]), lo, hi, d, L.ptr(e1), B, L.ptr(x),
           L.ptr(Rt) if with_rel else None, 0, R if with_rel else 0, dr if with_rel else 0,
           L.ptr(rel) if with_rel else None, B if with_rel else 0, L.ptr(r) if with_rel else None,
           L.ptr(st) if advance else None, L.ptr(seed) if advance else None, 0.003, 0.9, 0.999)
    assert same_bits(x, x_ref)
    if with_rel:
        assert same_bits(r, r_ref)
    else:
        assert float(r.min()) == 7.0
    if advance:
        assert same_bits(st, st_ref) and int(seed.item()) == int(seed_ref.item()) == 78
    else:
        assert float(st[0].item()) == 0.0 and int(seed.item()) == 77


# ------------------------------------------------------------------------------------------ batch-norm statistics
@pytest.mark.parametrize("R,C,bessel", [(512, 200, 0), (512 * 18 * 8, 32, 1), (100, 7, 0), (128, 96, 0), (33000, 33, 1)])
def test_bn_stats_finalize_equals_two_calls(L, R, C, bessel):
    rng = np.random.default_rng(2)
    x = dev((rng.normal(size=(R, C)) * 3 + 1).astype(np.float32))
    gamma, beta = dev(rng.normal(size=C).astype(np.float32)), dev(rng.normal(size=C).astype(np.float32))
    mm0, mv0 = rng.normal(size=C).astype(np.float32), rng.uniform(0.5, 2, size=C).astype(np.float32)
    nch = L.load().coper_colstats_chunks(R)
    outs = []
    for merged in (False, True):
        part = torch.zeros(nch * C * 2, device="cuda")
        mm, mv = dev(mm0), dev(mv0)
        a, b, mean, inv = (torch.zeros(C, device="cuda") for _ in range(4))
        sync = torch.zeros(1, dtype=torch.int32, device="cuda")
        if merged:
            for _ in range(2):          # twice: the arrival counter must come back to zero
                mm.copy_(dev(mm0)); mv.copy_(dev(mv0))
                L.call("coper_bn_stats_finalize", L.ptr(x), R, C, L.ptr(part), L.ptr(sync), L.ptr(gamma), L.ptr(beta),
                       L.ptr(mm), L.ptr(mv), 0.1, 1e-3, 1, bessel, L.ptr(a), L.ptr(b), L.ptr(mean), L.ptr(inv))
                assert int(sync.item()) == 0
        else:
            L.call("coper_colstats", L.ptr(x), R, C, L.ptr(part))
            L.call("coper_bn_finalize", L.ptr(part), nch, R, C, L.ptr(gamma), L.ptr(beta), L.ptr(mm), L.ptr(mv), 0.1, 1e-3,
                   1, 1, bessel, L.ptr(a), L.ptr(b), L.ptr(mean), L.ptr(inv))
        outs.append((part, mm, mv, a, b, mean, inv))
    assert same_bits(outs[0][0], outs[1][0])                    # the chunk partials
    # the last block adds the (same) partials in its own fixed order: fp64 sums of fp32 partials, rounded once
    for u, v in zip(outs[0][1:], outs[1][1:]):
        assert np.allclose(u.cpu().numpy(), v.cpu().numpy(), rtol=2e-6, atol=1e-7)
    xn = x.cpu().numpy().astype(np.float64)
    assert np.allclose(outs[1][5].cpu().numpy(), xn.mean(0), rtol=1e-5, atol=1e-5)
    assert np.allclose(outs[1][6].cpu().numpy(), 1.0 / np.sqrt(xn.var(0) + 1e-3), rtol=1e-5)
    # run to run: same bits
    part2 = torch.zeros_like(outs[1][0])
    mm, mv = dev(mm0), dev(mv0)
    a2, b2, mean2, inv2 = (torch.zeros(C, device="cuda") for _ in range(4))
    sync = torch.zeros(1, dtype=torch.int32, device="cuda")
    L.call("coper_bn_stats_finalize", L.ptr(x), R, C, L.ptr(part2), L.ptr(sync), L.ptr(gamma), L.ptr(beta),
           L.ptr(mm), L.ptr(mv), 0.1, 1e-3, 1, bessel, L.ptr(a2), L.ptr(b2), L.ptr(mean2), L.ptr(inv2))
    for u, v in zip(outs[1][1:], (mm, mv, a2, b2, mean2, inv2)):
        assert same_bits(u, v)


@pytest.mark.parametrize("R,C,use_batch", [(512, 200, 1), (512 * 18 * 8, 32, 1), (100, 7, 0), (4000, 64, 1)])
def test_bn_bwd_stats_finalize_equals_two_calls(L, R, C, use_batch):
    rng = np.random.default_rng(3)
    x = dev(rng.normal(size=(R, C)).astype(np.float32))
    dout = dev(rng.normal(size=(R, C)).astype(np.float32))
    a, b = dev(rng.normal(size=C).astype(np.float32)), dev(rng.normal(size=C).astype(np.float32))
    mean, inv = dev(rng.normal(size=C).astype(np.float32) * 0.1), dev(rng.uniform(0.5, 2, size=C).astype(np.float32))
    seed = dev(np.array([5], np.int64), torch.int64)
    nch = L.load().coper_colstats_chunks(R)
    outs = []
    for merged in (False, True):
        part = torch.zeros(nch * C * 2, device="cuda")
        dg, db, c1, c2 = (torch.zeros(C, device="cuda") for _ in range(4))
        sync = torch.zeros(1, dtype=torch.int32, device="cuda")
        if merged:
            for _ in range(2):
                L.call("coper_bn_act_bwd_stats_finalize", L.ptr(dout), L.ptr(x), R, C, L.ptr(a), L.ptr(b), L.ptr(mean),
                       L.ptr(inv), 1, 0.8, L.ptr(seed), 99, L.ptr(part), L.ptr(sync), use_batch, L.ptr(dg), L.ptr(db),
                       L.ptr(c1), L.ptr(c2))
                assert int(sync.item()) == 0
        else:
            L.call("coper_bn_act_bwd_stats", L.ptr(dout), L.ptr(x), R, C, L.ptr(a), L.ptr(b), L.ptr(mean), L.ptr(inv), 1,
                   0.8, L.ptr(seed), 99, L.ptr(part))
            L.call("coper_bn_act_bwd_finalize", L.ptr(part), nch, R, C, use_batch, L.ptr(dg), L.ptr(db), L.ptr(c1),
                   L.ptr(c2))
        outs.append((part, dg, db, c1, c2))
    assert same_bits(outs[0][0], outs[1][0])
    for u, v in zip(outs[0][1:], outs[1][1:]):
        assert np.allclose(u.cpu().numpy(), v.cpu().numpy(), rtol=2e-6, atol=1e-6)
    assert float(outs[1][1].abs().max()) > 0


# ------------------------------------------------------------------------------------------ reductions
def test_reduce_partials2_equals_two_calls(L):
    rng = np.random.default_rng(4)
    S, na, nb = 128, 288, 32
    A = dev(rng.normal(size=(S, na)).astype(np.float32))
    Bm = dev(rng.normal(size=(S, nb)).astype(np.float32))
    for acc in (0, 1):
        oa0, ob0 = rng.normal(size=na).astype(np.float32), rng.normal(size=nb).astype(np.float32)
        ra, rb, ma, mb = dev(oa0), dev(ob0), dev(oa0), dev(ob0)
        L.call("coper_reduce_partials", L.ptr(A), S, na, 0.5, acc, L.ptr(ra))
        L.call("coper_reduce_partials", L.ptr(Bm), S, nb, 0.5, acc, L.ptr(rb))
        L.call("coper_reduce_partials2", L.ptr(A), na, L.ptr(ma), L.ptr(Bm), nb, L.ptr(mb), S, 0.5, acc)
        assert same_bits(ra, ma) and same_bits(rb, mb)
        ref = 0.5 * A.cpu().numpy().astype(np.float64).sum(0) + (oa0 if acc else 0)
        assert np.allclose(ma.cpu().numpy(), ref, rtol=1e-5, atol=1e-5)


def _descs(L, tensors, ext=None):
    """coper_param_desc array + chunk lists for a list of gradient tensors (dense mode)."""
    import ctypes as C
    d = np.zeros(len(tensors), L.PARAM_DESC)
    chunks, offsets = [], [0]
    for t, g in enumerate(tensors):
        d[t]["grad"] = g.data_ptr()
        d[t]["theta"] = g.data_ptr()
        d[t]["vhat"] = g.data_ptr()
        d[t]["n"] = g.numel()
        d[t]["mode"] = 2 if t == ext else 0
        if t != ext:
            chunks += [(t, c) for c in range((g.numel() + L.MT_CHUNK - 1) // L.MT_CHUNK)]
        offsets.append(len(chunks))
    return (dev(d.view(np.uint8)), dev(np.array(chunks, np.int32).reshape(-1, 2)), len(chunks),
            dev(np.array(offsets, np.int32)))


@pytest.mark.parametrize("ext", [None, 0])
@pytest.mark.parametrize("clip", [True, False])
def test_mt_sumsq_clip_equals_separate_calls(L, ext, clip):
    rng = np.random.default_rng(5)
    sizes = [40000 * 8, 40943, 3 * 3 * 32, 32, 200 * 1000, 22 * 200, 17, 65536 * 3 + 5, 1, 200, 200]
    grads = [dev((rng.normal(size=n) * 0.3).astype(np.float32)) for n in sizes]
    descs, chunks, nch, offs = _descs(L, grads, ext)
    nt = len(grads)
    parts = dev(rng.uniform(0, 5, size=7))
    deltas = dev(rng.normal(size=512))
    p_ref, s_ref, c_ref = torch.zeros(nch, dtype=torch.float64, device="cuda"), torch.zeros(nt, dtype=torch.float64, device="cuda"), torch.zeros(2, device="cuda")
    L.call("coper_mt_sumsq", L.ptr(descs), nt, L.ptr(chunks), nch, L.ptr(offs), L.ptr(p_ref), L.ptr(s_ref))
    if ext is not None:
        L.call("coper_sumsq_combine", L.ptr(parts), 7, L.ptr(deltas), 512, L.ptr(s_ref))
    L.call("coper_clip_scale_n", L.ptr(s_ref), nt, 5.0, L.ptr(c_ref))
    p, s, c = torch.zeros_like(p_ref), torch.full_like(s_ref, -1.0), torch.zeros_like(c_ref)
    L.call("coper_mt_sumsq_clip", L.ptr(descs), nt, L.ptr(chunks), nch, L.ptr(offs), L.ptr(p), L.ptr(s),
           0 if ext is not None else -1, L.ptr(parts) if ext is not None else None, 7 if ext is not None else 0,
           L.ptr(deltas) if ext is not None else None, 512 if ext is not None else 0, 5.0, L.ptr(c) if clip else None)
    assert same_bits(s, s_ref)
    if clip:
        assert same_bits(c, c_ref)
        tot = sum(float((g.double() ** 2).sum()) for t, g in enumerate(grads) if t != ext)
        if ext is not None:
            tot += max(float(parts.sum() + deltas.sum()), 0.0)
        assert abs(float(c[1]) - np.sqrt(tot)) <= 1e-5 * np.sqrt(tot)
    else:
        assert float(c.abs().max()) == 0.0


# ------------------------------------------------------------------------------------------ scatters
@pytest.mark.parametrize("R", [22, 474, 3000])        # <= 2048 table rows: one block per row; above: warp per position
@pytest.mark.parametrize("with_norm,with_sq", [(True, False), (False, True), (False, False)])
def test_segscatter_pair_equals_two_calls(L, with_norm, with_sq, R):
    rng = np.random.default_rng(6)
    N, d, dr, B = 3000, 200, 200, 512
    e1 = dev(rng.integers(0, 600, B), torch.int64)           # many duplicate heads
    rel = dev(rng.integers(0, R, B), torch.int64)
    dx0 = dev(rng.normal(size=(B, d)).astype(np.float32))
    drr = dev(rng.normal(size=(B, dr)).astype(np.float32))
    dE0 = rng.normal(size=(N, d)).astype(np.float32)
    lo, hi = 100, 500
    res = []
    for merged in (False, True):
        dE = dev(dE0[lo:hi])
        dEsq = torch.zeros(hi - lo, d, device="cuda") if with_sq else None
        dR, dRsq = torch.zeros(R, dr, device="cuda"), torch.zeros(R, dr, device="cuda")
        nd = torch.full((B,), 3.0, dtype=torch.float64, device="cuda") if with_norm else None
        if merged:
            L.call("coper_segscatter_add_pair", L.ptr(e1), B, L.ptr(dx0), d, L.ptr(dE), L.ptr(dEsq), lo, hi, L.ptr(nd),
                   L.ptr(rel), B, L.ptr(drr), dr, L.ptr(dR), L.ptr(dRsq), 0, R)
        else:
            if with_norm:
                L.call("coper_segscatter_add_pair", L.ptr(e1), B, L.ptr(dx0), d, L.ptr(dE), L.ptr(dEsq), lo, hi, L.ptr(nd),
                       None, 0, None, 0, None, None, 0, 0)
            else:
                L.call("coper_segscatter_add_sq", L.ptr(e1), B, L.ptr(dx0), d, L.ptr(dE), L.ptr(dEsq), lo, hi)
            L.call("coper_segscatter_add_sq", L.ptr(rel), B, L.ptr(drr), dr, L.ptr(dR), L.ptr(dRsq), 0, R)
        res.append([t for t in (dE, dEsq, dR, dRsq, nd) if t is not None])
    for u, v in zip(*res):
        assert same_bits(u, v)
    ref = np.zeros((R, dr))
    np.add.at(ref, rel.cpu().numpy(), drr.cpu().numpy().astype(np.float64))
    assert np.allclose(res[1][2 if with_sq else 1].cpu().numpy(), ref, atol=1e-4)      # dR


# ------------------------------------------------------------------------------------------ generator backward halves
@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "fp16x3", "bf16"])
def test_cpg_bwd_halves_equal_full_call(L, prec):
    rng = np.random.default_rng(7)
    B, dc, F, d, dcb = 96, 8, 64, 40, 8
    p = L.PREC[prec]
    c, f = dev(rng.normal(size=(B, dc)).astype(np.float32)), dev(rng.normal(size=(B, F)).astype(np.float32))
    P, Pb = dev(rng.normal(size=(dc, F * d)).astype(np.float32)), dev(rng.normal(size=(dcb, d)).astype(np.float32))
    cb, dy = dev(rng.normal(size=(B, dcb)).astype(np.float32)), dev(rng.normal(size=(B, d)).astype(np.float32))
    lib = L.load()
    nbytes = max(lib.coper_cpg_fc_fwd_workspace_bytes(B, dc, F, d, p), lib.coper_cpg_fc_bwd_workspace_bytes(B, dc, F, d, p))
    outs = []
    for split in (False, True):
        ws = torch.zeros(max(nbytes, 256), dtype=torch.uint8, device="cuda")
        dP, dPb = torch.full((dc, F * d), 9.0, device="cuda"), torch.full((dcb, d), 9.0, device="cuda")
        df, dcw, dcbo = (torch.full(s, 9.0, device="cuda") for s in ((B, F), (B, dc), (B, dcb)))
        args = (L.ptr(c), L.ptr(f), L.ptr(P), None, L.ptr(cb), L.ptr(Pb), L.ptr(dy), B, dc, F, d, dcb, L.ptr(dP),
                L.ptr(dPb), L.ptr(df), L.ptr(dcw), L.ptr(dcbo), L.ptr(ws), ws.numel(), p)
        if split:
            L.call("coper_cpg_fc_bwd", *args, L.CPG_BWD_INPUT_GRADS_ONLY)
            torch.cuda.synchronize()
            assert float(dP.min()) == 9.0 and float(dPb.min()) == 9.0          # untouched by the first half
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                L.call("coper_cpg_fc_bwd", *args, L.CPG_BWD_WEIGHT_GRADS_ONLY)
            torch.cuda.current_stream().wait_stream(side)
        else:
            L.call("coper_cpg_fc_bwd", *args, 0)
        outs.append((dP, dPb, df, dcw, dcbo))
    for u, v in zip(*outs):
        assert same_bits(u, v)
    ref = np.einsum("bi,bk,bj->kij", f.cpu().numpy().astype(np.float64), c.cpu().numpy().astype(np.float64),
                    dy.cpu().numpy().astype(np.float64)).reshape(dc, F * d)
    tol = 2e-2 if prec == "bf16" else 1e-5
    assert np.abs(outs[1][0].cpu().numpy() - ref).max() <= tol * np.abs(ref).max()


# ------------------------------------------------------------------------------------------ inference batch norm
@pytest.mark.parametrize("R,C,relu", [(512, 200, 1), (512 * 18 * 8, 32, 1), (100, 7, 0), (64, 30, 1)])
def test_bn_act_fwd_moving_equals_two_calls(L, R, C, relu):
    rng = np.random.default_rng(8)
    x = dev(rng.normal(size=(R, C)).astype(np.float32))
    gamma, beta = dev(rng.normal(size=C).astype(np.float32)), dev(rng.normal(size=C).astype(np.float32))
    mm, mv = dev(rng.normal(size=C).astype(np.float32)), dev(rng.uniform(0.5, 2, size=C).astype(np.float32))
    a, b, mean, inv = (torch.zeros(C, device="cuda") for _ in range(4))
    ref, out = torch.zeros(R, C, device="cuda"), torch.zeros(R, C, device="cuda")
    L.call("coper_bn_finalize", None, 0, R, C, L.ptr(gamma), L.ptr(beta), L.ptr(mm), L.ptr(mv), 0.1, 1e-3, 0, 0, 0,
           L.ptr(a), L.ptr(b), L.ptr(mean), L.ptr(inv))
    L.call("coper_bn_act_fwd", L.ptr(x), R, C, L.ptr(a), L.ptr(b), relu, 1.0, None, 0, L.ptr(ref))
    L.call("coper_bn_act_fwd_moving", L.ptr(x), R, C, L.ptr(gamma), L.ptr(beta), L.ptr(mm), L.ptr(mv), 1e-3, relu,
           L.ptr(out))
    assert same_bits(out, ref)
    xn, g, be = x.cpu().numpy().astype(np.float64), gamma.cpu().numpy(), beta.cpu().numpy()
    want = (xn - mm.cpu().numpy()) / np.sqrt(mv.cpu().numpy() + 1e-3) * g + be
    if relu:
        want = np.maximum(want, 0)
    assert np.allclose(out.cpu().numpy(), want, rtol=1e-5, atol=1e-5)


# ------------------------------------------------------------------------------------------ conv backward with Conv1BN folded in
@pytest.mark.parametrize("B,H,W,KH,C,keep", [(37, 20, 10, 3, 32, 0.7), (8, 16, 16, 3, 32, 1.0), (5, 10, 10, 3, 8, 0.8),
                                             (4, 12, 8, 2, 32, 0.9)])
def test_conv_bwd_bn_equals_apply_then_conv_bwd(L, B, H, W, KH, C, keep):
    rng = np.random.default_rng(11)
    KW = KH
    OH, OW = H - KH + 1, W - KW + 1
    n = OH * OW * C
    x0 = dev(rng.normal(size=(B, H * W)).astype(np.float32))
    wc = dev(rng.normal(size=(KH * KW * C)).astype(np.float32))
    z = dev(rng.normal(size=(B, n)).astype(np.float32))
    dout = dev(rng.normal(size=(B, n)).astype(np.float32))
    a, b = dev(rng.normal(size=C).astype(np.float32)), dev(rng.normal(size=C).astype(np.float32))
    mean, inv = dev(rng.normal(size=C).astype(np.float32) * 0.1), dev(rng.uniform(0.5, 2, size=C).astype(np.float32))
    c1, c2 = dev(rng.normal(size=C).astype(np.float32) * 0.01), dev(rng.normal(size=C).astype(np.float32) * 0.01)
    seed = dev(np.array([21], np.int64), torch.int64)
    slabs = L.load().coper_conv_bwd_slabs(B, H, W, KH, KW, C, 0)
    outs = []
    for fused in (False, True):
        dz = torch.zeros(B, n, device="cuda")
        dx0 = torch.zeros(B, H * W, device="cuda")
        dw, db = torch.zeros(slabs, KH * KW * C, device="cuda"), torch.zeros(slabs, C, device="cuda")
        if fused:
            L.call("coper_conv_bwd_bn", L.ptr(dout), L.ptr(z), L.ptr(x0), B, H, W, L.ptr(wc), KH, KW, C, 0, L.ptr(a), L.ptr(b),
                   L.ptr(mean), L.ptr(inv), L.ptr(c1), L.ptr(c2), 1, keep, L.ptr(seed), 123, L.ptr(dx0), L.ptr(dw), L.ptr(db),
                   L.ptr(dz))
        else:
            L.call("coper_bn_act_bwd_apply", L.ptr(dout), L.ptr(z), B * OH * OW, C, L.ptr(a), L.ptr(b), L.ptr(mean),
                   L.ptr(inv), L.ptr(c1), L.ptr(c2), 1, keep, L.ptr(seed), 123, 1.0, 0, L.ptr(dz))
            L.call("coper_conv_bwd", L.ptr(dz), L.ptr(x0), B, H, W, L.ptr(wc), KH, KW, C, 0, L.ptr(dx0), L.ptr(dw), L.ptr(db))
        outs.append((dx0, dw, db))
    for u, v in zip(*outs):
        assert same_bits(u, v)
    assert float(outs[1][0].abs().max()) > 0 and float(outs[1][1].abs().max()) > 0
