"""The generator backward's T-kernel with the context-invariant dy tile resident in shared memory for all dc context
groups (bf16 / fp16x3), with the forward and the rest of the backward alongside.  Against fp64 at the tolerances of
``test_gpu_kernels.py::test_cpg_fc_fwd_bwd``, at the shapes that exercise the resident region's bookkeeping: CTAs that
get more than one tile and refill the region (B = 2048) or keep it (two tiles of the same m-block in a row), K extents
of 2 to 4 k-blocks (d = 72, 200, 256; the last one partial), dc = 1 (plain), dc = 32, a one-hot context (param_lookup),
B not a multiple of 128, and F = 4640 (73 forward k-blocks: a last split shorter than the others)."""
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


def dev(a):
    t = torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float32).cuda()
    _ALIVE.append(t)
    return t


def relerr(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return np.abs(a - b).max() / (np.abs(b).max() + 1e-30)


def _bf16r(x):
    return torch.as_tensor(np.asarray(x), dtype=torch.float32).to(torch.bfloat16).to(torch.float64).numpy()


@pytest.fixture(scope="module")
def L():
    from coper_b200 import _lib
    _lib.load()
    return _lib


CASES = {
    "refill_B2048": (2048, 8, 4640, 200, "dense"),
    "dc32_ragged_batch": (300, 32, 4640, 200, "dense"),
    "plain_dc1": (512, 1, 4608, 200, "ones"),
    "param_lookup_onehot": (512, 22, 4608, 200, "onehot"),
    "d256_same_mblock_twice": (512, 4, 6272, 256, "dense"),     # backward: 4 x 49 tiles on 148 SMs
    "d72": (640, 8, 1536, 72, "dense"),
}


@pytest.mark.parametrize("prec", ["fp16x3", "bf16"])
@pytest.mark.parametrize("case", list(CASES))
def test_cpg_resident_operand(L, case, prec):
    B, dc, F, d, ctx = CASES[case]
    p = L.PREC[prec]
    rng = np.random.default_rng(11)
    if ctx == "ones":
        c = np.ones((B, dc))
    elif ctx == "onehot":
        c = np.eye(dc)[rng.integers(0, dc, B)]
    else:
        c = rng.normal(size=(B, dc))
    f = np.maximum(rng.normal(size=(B, F)), 0)
    P = rng.normal(size=(dc, F * d)) * 0.01
    cb = rng.normal(size=(B, dc))
    Pb = rng.normal(size=(dc, d))
    dy = rng.normal(size=(B, d))
    c, f, P, cb, Pb, dy = (a.astype(np.float32).astype(np.float64) for a in (c, f, P, cb, Pb, dy))
    lib = L.load()
    nbytes = max(lib.coper_cpg_fc_fwd_workspace_bytes(B, dc, F, d, p), lib.coper_cpg_fc_bwd_workspace_bytes(B, dc, F, d, p))
    ws = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device="cuda")
    tc, tf, tP, tcb, tPb = (dev(a) for a in (c, f, P, cb, Pb))
    y = torch.full((B, d), float("nan"), device="cuda")
    L.call("coper_cpg_fc_fwd", L.ptr(tc), L.ptr(tf), L.ptr(tP), None, L.ptr(tcb), L.ptr(tPb), B, dc, F, d, dc, 1.0, None, 0,
           L.ptr(y), L.ptr(ws), ws.numel(), p)
    dP = torch.zeros(dc, F * d, device="cuda")
    dPb = torch.zeros(dc, d, device="cuda")
    df = torch.zeros(B, F, device="cuda")
    dcw = torch.zeros(B, dc, device="cuda")
    dcb = torch.zeros(B, dc, device="cuda")
    L.call("coper_cpg_fc_bwd", L.ptr(tc), L.ptr(tf), L.ptr(tP), None, L.ptr(tcb), L.ptr(tPb), L.ptr(dev(dy)),
           B, dc, F, d, dc, L.ptr(dP), L.ptr(dPb), L.ptr(df), L.ptr(dcw), L.ptr(dcb), L.ptr(ws), ws.numel(), p, 1)

    # fp64 references on the operands the engine consumes (bf16: f, P, dy and c * dy rounded; c scales in fp32),
    # one context group at a time
    fr, dyr = (_bf16r(f), _bf16r(dy)) if prec == "bf16" else (f, dy)
    P3 = P.reshape(dc, F, d)
    yr = cb @ Pb
    dfr = np.zeros((B, F))
    dcr = np.zeros((B, dc))
    dPr = np.zeros((dc, F, d))
    for k in range(dc):
        Pk = _bf16r(P3[k]) if prec == "bf16" else P3[k]
        yr += c[:, k:k + 1] * (fr @ Pk)
        T = dyr @ Pk.T
        dfr += c[:, k:k + 1] * T
        dcr[:, k] = (f * T).sum(1)
        dyc = c[:, k:k + 1] * dy
        dPr[k] = fr.T @ (_bf16r(dyc.astype(np.float32)) if prec == "bf16" else dyc)
    assert relerr(y.cpu().numpy(), yr) < 1e-5
    assert relerr(df.cpu().numpy(), dfr) < 2e-5
    assert relerr(dcw.cpu().numpy(), dcr) < 2e-5
    assert relerr(dP.cpu().numpy(), dPr.reshape(dc, F * d)) < 2e-5
    assert relerr(dPb.cpu().numpy(), cb.T @ dy) < 2e-5
    assert relerr(dcb.cpu().numpy(), dy @ Pb.T) < 2e-5
