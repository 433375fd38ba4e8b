"""The fused-norm and split forms of the training scorer without a GPU: the argument checks of
coper_score1n_bce_fwd_bwd_norm / coper_score1n_bce_dE / coper_score1n_bce_fwd_bwd that run before anything is
launched."""
import pytest

from coper_b200 import _lib, build

ERR_INVALID_ARG, ERR_UNSUPPORTED = -1, -3
FAKE = 256           # never dereferenced: every case below is rejected before a launch
FP32, TF32X3 = 0, 2


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def _bce(lib, name, prec, dE=FAKE, dE_sumsq=FAKE, B=130, N=1003, d=200):
    head = (FAKE, FAKE, None, FAKE, FAKE, B, N, d, 0.9, 1.0 / N, 1.0 / (B * N), FAKE, FAKE, 1024, FAKE, dE, FAKE)
    if name == "coper_score1n_bce_fwd_bwd_norm":
        return lib.coper_score1n_bce_fwd_bwd_norm(*head, dE_sumsq, FAKE, 1 << 30, prec, None)
    return lib.coper_score1n_bce_fwd_bwd(*head, FAKE, 1 << 30, prec, None)


def test_norm_form_needs_a_tensor_pipe_engine(lib):
    # the CUDA-core engine does not fuse the squared norm of dE
    assert _bce(lib, "coper_score1n_bce_fwd_bwd_norm", FP32) == ERR_UNSUPPORTED
    assert lib.coper_score1n_bce_dE(FAKE, 130, 1003, 200, 1e-5, FAKE, FAKE, FAKE, FAKE, 1 << 30, FP32,
                                    None) == ERR_UNSUPPORTED


def test_norm_form_needs_its_sum_output(lib):
    assert _bce(lib, "coper_score1n_bce_fwd_bwd_norm", TF32X3, dE_sumsq=None) == ERR_INVALID_ARG


def test_split_call_needs_the_norm_form(lib):
    # dE == NULL (the split form, dE by a later coper_score1n_bce_dE) only through the _norm entry point, and only on
    # a tensor-pipe engine
    assert _bce(lib, "coper_score1n_bce_fwd_bwd", TF32X3, dE=None) == ERR_INVALID_ARG
    assert _bce(lib, "coper_score1n_bce_fwd_bwd_norm", FP32, dE=None) == ERR_INVALID_ARG


def test_dE_call_rejects_missing_outputs(lib):
    for dE, dbias in ((None, FAKE), (FAKE, None)):
        assert lib.coper_score1n_bce_dE(FAKE, 130, 1003, 200, 1e-5, dE, FAKE, dbias, FAKE, 1 << 30, TF32X3,
                                        None) == ERR_INVALID_ARG
