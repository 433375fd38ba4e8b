"""coper_score_sampled_bce_fwd_bwd_sharded without a GPU: its workspace query and the argument checks that run before
anything is launched."""
import pytest

from coper_b200 import _lib, build

ERR_INVALID_ARG, ERR_UNSUPPORTED, ERR_WORKSPACE = -1, -3, -4


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def test_sharded_workspace_holds_the_sort_keys(lib):
    for B, L in ((130, 12), (512, 1000)):
        plain = lib.coper_score_sampled_workspace_bytes(B, L)
        assert lib.coper_score_sampled_sharded_workspace_bytes(B, L) >= plain + 4 * B * L
    assert lib.coper_score_sampled_sharded_workspace_bytes(0, 12) == 256


def _call(lib, N=1003, d=200, lo=0, hi=512, ws_bytes=1 << 30, B=130, L=12):
    fake = 256           # never dereferenced: every case below is rejected before a launch
    return lib.coper_score_sampled_bce_fwd_bwd_sharded(fake, fake, fake, fake, fake, B, L, N, d, 0.9, 1.0 / N,
                                                       1.0 / (B * L), fake, fake, fake, fake, fake, fake, fake, fake,
                                                       lo, hi, fake, ws_bytes, None)


@pytest.mark.parametrize("lo, hi", [(-1, 512), (512, 512), (600, 512), (512, 1004)])
def test_sharded_scorer_rejects_bad_row_ranges(lib, lo, hi):
    assert _call(lib, lo=lo, hi=hi) == ERR_INVALID_ARG


def test_sharded_scorer_rejects_unsupported_shapes(lib):
    assert _call(lib, N=1 << 31, hi=512) == ERR_INVALID_ARG
    assert _call(lib, d=257) == ERR_UNSUPPORTED
    assert _call(lib, ws_bytes=16) == ERR_WORKSPACE
