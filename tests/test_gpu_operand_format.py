"""coper_prepare_operand, byte for byte, against a NumPy restatement of the prepared operand format.

  * bf16: round to nearest even, [rows, ldp] with ldp = cols rounded up to 8;
  * tf32x3: hi = cvt.rna (add half an ulp of tf32 to the magnitude, clear the low 13 bits), lo = x - hi; two fp32
    planes [rows, ldp], ldp = cols rounded up to 4;
  * fp16x3: e from frexp of max |x| (largest magnitude lands in [2^10, 2^11), clamped to [-100, 100], 0 for an all-zero
    operand), hi = fp16(x * 2^e), lo = fp16(x * 2^e - hi); two fp16 planes [rows, ldp], ldp = cols rounded up to 8, then
    the trailer at align_up(rows * ldp * 4, 256): word 0 = e, words 1 and 2 = max |x| as float bits.
Padding columns are zero in every plane.  The layouts cover the dense, strided, column-tail (cols % 8 != 0) and
misaligned-source (scalar load) paths, and both fp16x3 preparations (<= 4 Mi elements: one launch; above: two).
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
PREC = {"bf16": 1, "tf32x3": 2, "fp16x3": 3}

# name: (rows, cols, ld_src, source offset in floats, all zero)
LAYOUTS = {
    "dense": (512, 200, 200, 0, False),
    "large": (40943, 200, 200, 0, False),             # 8.2 M elements: fp16x3 takes the two-launch path
    "strided": (300, 200, 213, 0, False),
    "strided_large": (21000, 203, 208, 0, False),     # 4.26 M elements > 4 Mi, strided, cols % 8 != 0
    "cols37": (129, 37, 37, 0, False),
    "misaligned": (257, 64, 64, 1, False),
    "misaligned_large": (40943, 200, 200, 1, False),
    "zeros": (64, 40, 40, 0, True),
}


def ref_bf16(x):
    b = x.view(np.uint32).astype(np.uint64)
    return ((b + 0x7FFF + ((b >> 16) & 1)) >> 16).astype(np.uint16)


def ref_tf32(x):
    b = x.view(np.uint32)
    hi = ((b & 0x7FFFFFFF) + 0x1000) & ~np.uint32(0x1FFF) | (b & 0x80000000)
    hi = hi.astype(np.uint32).view(np.float32)
    return hi, (x - hi).astype(np.float32)


def ref_fp16x3_exponent(m):
    if not (m > 0) or not (m < 3.0e38):
        return 0
    _, ex = np.frexp(np.float32(m))
    return int(min(max(10 - (int(ex) - 1), -100), 100))


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("prec", list(PREC))
def test_prepare_operand_matches_restatement(prec, layout):
    from coper_b200 import _lib as L
    lib = L.load()
    rows, cols, ld, off, zero = LAYOUTS[layout]
    rng = np.random.default_rng(rows + cols + ld + off)
    if zero:
        src = np.zeros(rows * ld + off, np.float32)
    else:
        # magnitudes over six decades: the fp16x3 lo plane and its subnormal range are exercised
        src = (rng.standard_normal(rows * ld + off) * 10.0 ** rng.uniform(-3, 3, rows * ld + off)).astype(np.float32)
    x = src[off:].reshape(rows, ld)[:, :cols]
    p = PREC[prec]
    ldp = -(-cols // 4) * 4 if prec == "tf32x3" else -(-cols // 8) * 8
    t_src = torch.from_numpy(src).cuda()
    nbytes = lib.coper_prepared_bytes(rows, cols, p)
    out = torch.full((nbytes,), 0xA5, dtype=torch.uint8, device="cuda")
    L.call("coper_prepare_operand", L.ptr(t_src[off:]), rows, cols, ld, p, L.ptr(out))
    got = out.cpu().numpy()

    xp = np.zeros((rows, ldp), np.float32)
    xp[:, :cols] = x
    if prec == "bf16":
        assert np.array_equal(got[:rows * ldp * 2].view(np.uint16).reshape(rows, ldp), ref_bf16(xp))
    elif prec == "tf32x3":
        hi, lo = ref_tf32(xp)
        planes = got[:rows * ldp * 8].view(np.uint32).reshape(2, rows, ldp)
        assert np.array_equal(planes[0], hi.view(np.uint32))
        assert np.array_equal(planes[1], lo.view(np.uint32))
    else:
        m = np.float32(np.abs(x).max())
        e = ref_fp16x3_exponent(m)
        xs = (xp * np.float32(2.0 ** e)).astype(np.float32)
        hi = xs.astype(np.float16)
        lo = (xs - hi.astype(np.float32)).astype(np.float16)
        planes = got[:rows * ldp * 4].view(np.uint16).reshape(2, rows, ldp)
        assert np.array_equal(planes[0], hi.view(np.uint16))
        assert np.array_equal(planes[1], lo.view(np.uint16))
        tr = -(-(rows * ldp * 4) // 256) * 256
        words = got[tr:tr + 12].view(np.uint32)
        assert int(words[0].view(np.int32)) == e
        assert words[1] == m.view(np.uint32) and words[2] == m.view(np.uint32)
        if zero:
            assert e == 0 and words[1] == 0
