"""CPU-only checks of the frame-epilogue backward (dcd_dgde_frame_bwd, dcd_dgde_locate_solve_bwd, dcd_gmw_ray_rescale_bwd): the
companion header include/dcd_b200_grad.h declares them and the library exports them, every entry point validates its arguments before any CUDA call, and the Python
wrappers reject gradients into the constants before any launch.  refine_detections stays inference-only."""
import os
import re

import pytest
import torch

import dcd_b200
from dcd_b200 import _lib, ops

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INVALID = -1
F = 256                      # a fake, aligned "device" address: every rejected call below must fail before touching it


@pytest.fixture(scope="module")
def lib():
    from dcd_b200.build import build_library
    return _lib.load_library(build_library())


def header_functions(name):
    src = open(os.path.join(ROOT, "include", name)).read()
    return src, set(re.findall(r"\b(dcd_[a-z0-9_]+)\s*\(", re.sub(r"/\*.*?\*/", "", src, flags=re.S)))


def test_grad_header_declares_the_backward_exports_and_the_library_exports_them(lib):
    src, names = header_functions("dcd_b200_grad.h")
    assert names == {"dcd_dgde_frame_bwd", "dcd_dgde_locate_solve_bwd", "dcd_gmw_ray_rescale_bwd"}
    assert " %d exported functions." % len(names) in src
    assert '#include "dcd_b200.h"' in src                           # one ABI: the same status codes, flags and version
    _, base = header_functions("dcd_b200.h")
    assert not names & base and names == set(_lib.GRAD_SIGNATURES)
    for n in names:
        assert hasattr(lib, n), n
    assert lib.dcd_version() == 2


def test_frame_bwd_validates_before_any_cuda_call(lib):
    n, C = 73, 415

    def call(N=4, n=n, B=1, bi=0, C=C, H=96, W=320, ch2=50, ch3=196, cho=4, fm=F, dims=F, up=(F, F, F, F), gm=F, gd=F):
        return lib.dcd_dgde_frame_bwd(fm, F, bi, B, C, H, W, ch2, ch3, cho, F, F, F, dims, N, n, 2.0, 80.0, 3, 4.0, *up, gm, gd, 0)

    assert call(up=(0, 0, 0, 0)) == INVALID                          # no upstream gradient at all
    assert call(N=-1) == INVALID
    assert call(n=1) == INVALID and call(n=257) == INVALID
    assert call(ch2=C - 2 * n + 1) == INVALID                        # channel groups outside the map
    assert call(ch3=C - 3 * n + 1) == INVALID and call(cho=C - 1) == INVALID and call(cho=-1) == INVALID
    assert call(ch3=50 + 2 * n - 1) == INVALID                       # overlapping groups (one channel, two gradients)
    assert call(C=0) == INVALID and call(H=0) == INVALID and call(B=0) == INVALID
    assert call(B=2) == INVALID                                      # several images need batch_idx
    assert call(fm=0) == INVALID and call(gm=0) == INVALID
    assert call(dims=0) == INVALID                                   # grad_dims without dims
    for k in range(4):                                               # any single upstream gradient is enough to get past
        up = [0, 0, 0, 0]
        up[k] = F
        assert call(up=tuple(up), fm=0) == INVALID
    assert call(N=0) == 0 and call(N=0, fm=0, gm=0, up=(0, F, 0, 0)) == 0     # N = 0: no-op


def test_locate_solve_bwd_validates_before_any_cuda_call(lib):
    def call(N=7, n=73, kp=F, dims=F, gd=F, gl=F, outs=(F, F, F, F, F)):
        return lib.dcd_dgde_locate_solve_bwd(kp, F, F, F, F, F, F, dims, N, n, 2.0, 80.0, 3, 4.0, gd, gl, *outs, 0)

    assert call(gd=0, gl=0) == INVALID                               # no upstream gradient
    assert call(outs=(0, 0, 0, 0, 0)) == INVALID                     # no output
    assert call(N=-1) == INVALID
    assert call(n=1) == INVALID and call(n=257) == INVALID
    assert call(kp=0) == INVALID
    assert call(dims=0) == INVALID                                   # grad_dims without dims
    assert call(N=0) == 0 and call(N=0, kp=0) == 0


def test_ray_rescale_bwd_validates_before_any_cuda_call(lib):
    def call(N=5, raw=F, g=F, outs=(F, F, F)):
        return lib.dcd_gmw_ray_rescale_bwd(raw, F, F, g, N, *outs, 0)

    assert call(g=0) == INVALID                                      # no upstream gradient
    assert call(outs=(0, 0, 0)) == INVALID                           # no output
    assert call(raw=0) == INVALID
    assert call(N=-1) == INVALID
    assert call(N=0) == 0 and call(N=0, raw=0, g=0) == 0


@pytest.fixture
def no_library_call(monkeypatch):
    def forbidden():
        raise AssertionError("the library was reached")
    monkeypatch.setattr(ops._lib, "lib", forbidden)


def test_wrappers_raise_when_a_constant_requires_grad(no_library_call):
    N, n = 3, 8
    fm = torch.zeros(1, 415, 8, 8, requires_grad=True)
    base = dict(indexs=torch.arange(N), pred_rots=torch.zeros(N), P=torch.eye(3, 4), pad_size=torch.zeros(2))
    for name in ("pred_rots", "P", "pad_size"):
        kw = dict(base)
        kw[name] = kw[name].clone().requires_grad_(True)
        with pytest.raises(RuntimeError, match="`%s` receives no gradient" % name):
            dcd_b200.frame_depths_from_map(fm, dims=torch.ones(N, 3), n=n, **kw)
        with pytest.raises(RuntimeError, match="`%s` receives no gradient" % name):
            dcd_b200.compute_pairs_kpts_depth(torch.zeros(N, n, 2, requires_grad=True), torch.zeros(N, 2), torch.zeros(N, 2),
                                              kw["pad_size"], torch.zeros(N, n, 3), kw["pred_rots"], kw["P"])
    # differentiable inputs get as far as the device check (CPU tensors here), and so do constants under no_grad
    with pytest.raises(RuntimeError, match="CUDA tensors"):
        dcd_b200.frame_depths_from_map(fm, dims=torch.ones(N, 3, requires_grad=True), n=n, **base)
    with pytest.raises(RuntimeError, match="CUDA tensors"):
        dcd_b200.ray_rescale(torch.ones(N, 3, requires_grad=True), torch.ones(N, requires_grad=True), torch.ones(N, 3))
    with torch.no_grad():
        with pytest.raises(RuntimeError, match="CUDA tensors"):
            dcd_b200.frame_depths_from_map(fm, dims=torch.ones(N, 3), n=n, **dict(base, P=torch.eye(3, 4).requires_grad_()))


def test_refine_detections_stays_inference_only(no_library_call):
    N = 3
    gmw = dcd_b200.GMW()
    for name in ("pred_regression", "pred_rots", "dims"):
        t = {"pred_regression": torch.zeros(1, 415, 8, 8), "indexs": torch.arange(N), "pred_rots": torch.zeros(N),
             "P": torch.eye(3, 4), "pad_size": torch.zeros(2), "dims": torch.ones(N, 3)}
        t[name] = t[name].clone().requires_grad_(True)
        with pytest.raises(RuntimeError, match="inference-only"):
            dcd_b200.refine_detections(gmw=gmw, **t)
