"""CPU-only checks of the plan-free correspondence backward dcd_gmw_transport_terms_bwd: argument validation happens before
any CUDA call."""
import pytest

from dcd_b200 import _lib

OK_N, OK_n = 4, 73


@pytest.fixture(scope="module")
def lib():
    from dcd_b200.build import build_library
    return _lib.load_library(build_library())


def test_transport_terms_bwd_argument_validation_without_a_gpu(lib):
    fwd_need = lib.dcd_gmw_transport_workspace_bytes(OK_N, OK_n)
    need = lib.dcd_gmw_transport_bwd_workspace_bytes(OK_N, OK_n)
    assert fwd_need > 0 and need > 0

    def call(f4=16, f6=16, fws=256, fbytes=fwd_need, u=16, v=16, gt=16, N=OK_N, n=OK_n, lam=10.0, iters=32, tol=1e-7,
             g4=16, g6=16, info=0, ws=512, nbytes=need):
        return lib.dcd_gmw_transport_terms_bwd(f4, f6, fws, fbytes, u, v, gt, N, n, lam, iters, tol, g4, g6, info, ws, nbytes, 0)

    for name in ("f4", "f6", "fws", "u", "v", "gt", "g4", "g6", "ws"):                       # null pointers
        assert call(**{name: 0}) == -1, name
    assert call(N=0) == -1 and call(N=-1) == -1                                              # N < 1
    assert call(n=1) == -1 and call(n=257) == -1                                             # n out of range
    assert call(lam=0.0) == -1 and call(iters=0) == -1 and call(tol=-1.0) == -1              # as dcd_gmw_transport_bwd
    assert call(fbytes=fwd_need - 4) == -2                                                   # forward workspace (K) too small
    assert call(fws=256 + 64) == -2                                                          # ... or misaligned
    assert call(nbytes=need - 4) == -2                                                       # backward workspace too small
    assert call(ws=512 + 64) == -2                                                           # ... or misaligned
    big = 65536
    assert call(N=big, fbytes=lib.dcd_gmw_transport_workspace_bytes(big, OK_n),
                nbytes=lib.dcd_gmw_transport_bwd_workspace_bytes(big, OK_n)) == -4            # objects map to gridDim.y / .z
