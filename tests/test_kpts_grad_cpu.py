"""CPU-only checks of the keypoint-gradient entry dcd_gmw_kpts_bwd: argument validation happens before any CUDA call."""
import pytest

from dcd_b200 import _lib

OK_N, OK_n, OK_DEPTH = 4, 73, 12


@pytest.fixture(scope="module")
def lib():
    from dcd_b200.build import build_library
    return _lib.load_library(build_library())


def test_kpts_bwd_argument_validation_without_a_gpu(lib):
    need = lib.dcd_gmw_bwd_scratch_bytes(OK_N, OK_n, OK_DEPTH)
    assert need > 0

    def call(p4=16, p6=16, N=OK_N, n=OK_n, depth=OK_DEPTH, scratch=256, nbytes=need, g2=8, g3=8):
        return lib.dcd_gmw_kpts_bwd(p4, p6, N, n, depth, scratch, nbytes, g2, g3, 0)

    assert call(p4=0) == -1 and call(p6=0) == -1 and call(scratch=0) == -1      # null pointers
    assert call(g2=0, g3=0) == -1                                                 # no output
    assert call(N=-1) == -1 and call(N=0) == -1                                   # N < 1, as dcd_gmw_weights_bwd
    assert call(n=1) == -1 and call(n=257) == -1 and call(depth=0) == -1
    assert call(nbytes=need - 4) == -2                                            # scratch too small
    assert call(scratch=256 + 64) == -2                                           # scratch misaligned
