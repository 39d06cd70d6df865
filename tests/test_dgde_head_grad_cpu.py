"""CPU-only checks of the detector-head backward entries (dcd_poi_gather_bwd, dcd_dgde_locate_bwd,
dcd_dgde_depth_ensemble_bwd): argument validation happens before any CUDA call, so every rejected call returns without a GPU."""
import pytest

from dcd_b200 import _lib

INVALID, UNSUPPORTED = -1, -4
MAX_K = 1024          # DCD_POI_BWD_MAX_K


@pytest.fixture(scope="module")
def lib():
    from dcd_b200.build import build_library
    return _lib.load_library(build_library())


def test_poi_gather_bwd_argument_validation_without_a_gpu(lib):
    def call(g=16, idx=16, B=2, K=50, C=440, HW=96 * 320, out=16):
        return lib.dcd_poi_gather_bwd(g, idx, B, K, C, HW, out, 0)

    assert call(out=0) == INVALID                                                   # no output
    assert call(g=0) == INVALID and call(idx=0) == INVALID                          # null inputs with K > 0
    assert call(B=-1) == INVALID and call(K=-1) == INVALID                          # negative sizes
    assert call(C=0) == INVALID and call(HW=0) == INVALID
    assert call(K=MAX_K + 1) == UNSUPPORTED and call(K=1 << 40) == UNSUPPORTED      # the duplicate scan's bound
    assert call(B=0) == 0 and call(B=0, g=0, idx=0, out=0) == 0                     # no image: no-op


def test_dgde_locate_bwd_argument_validation_without_a_gpu(lib):
    def call(K=16, pts=16, ofs=16, pad=16, dep=16, g=16, N=7, go=16, gp=16, gd=16):
        return lib.dcd_dgde_locate_bwd(K, pts, ofs, pad, dep, g, N, 4.0, go, gp, gd, 0)

    for kw in ("K", "pts", "ofs", "pad", "dep", "g"):
        assert call(**{kw: 0}) == INVALID, kw                                        # null inputs
    assert call(go=0, gp=0, gd=0) == INVALID                                        # no output
    assert call(N=-1) == INVALID
    assert call(N=0) == 0 and call(N=0, K=0, go=0, gp=0, gd=0) == 0                  # N = 0: no-op


def test_dgde_depth_ensemble_bwd_argument_validation_without_a_gpu(lib):
    def call(kp=16, dims=16, K=16, direct=16, lud=16, luk=16, sc=16, N=5, gkd=16, gd=16, ge=16, gs=16,
             o_kp=16, o_dims=16, o_dir=16, o_lud=16, o_luk=16, o_sc=16):
        return lib.dcd_dgde_depth_ensemble_bwd(kp, dims, K, direct, lud, luk, sc, N, 4.0, 1e-3, 0.1, 100.0, gkd, gd, ge, gs,
                                               o_kp, o_dims, o_dir, o_lud, o_luk, o_sc, 0)

    for kw in ("kp", "dims", "K"):
        assert call(**{kw: 0}) == INVALID, kw                                        # null inputs
    assert call(gkd=0, gd=0, ge=0, gs=0) == INVALID                                 # no upstream gradient
    assert call(o_kp=0, o_dims=0, o_dir=0, o_lud=0, o_luk=0, o_sc=0) == INVALID     # no output
    assert call(luk=0) == INVALID                                                   # ensemble gradient without its channels
    assert call(lud=0) == INVALID                                                   # direct depth without its uncertainty
    assert call(sc=0) == INVALID                                                    # score gradient without the scores
    assert call(direct=0, lud=0, o_lud=0) == INVALID and call(direct=0, lud=0, o_dir=0) == INVALID
    assert call(N=-1) == INVALID
    assert call(N=0) == 0 and call(N=0, kp=0, gkd=0, gd=0, ge=0, gs=0) == 0          # N = 0: no-op
