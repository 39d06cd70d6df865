"""CPU-only checks of the DGDE -> GMW refine chain (dcd_dgde_gmw_refine_fwd / dcd_b200.refine_detections): the header
declares both entry points, the C entry point validates its arguments before any CUDA call, and the Python wrapper rejects
bad input before it reaches the library."""
import os
import re

import pytest
import torch

import dcd_b200
from dcd_b200 import _lib, ops

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DCD_E_INVALID, DCD_E_WORKSPACE = -1, -2


@pytest.fixture(scope="module")
def lib():
    from dcd_b200.build import build_library
    return _lib.load_library(build_library())


def _header():
    return open(os.path.join(ROOT, "include", "dcd_b200.h")).read()


def test_header_declares_the_refine_exports_and_the_export_count():
    src = _header()
    code = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = set(re.findall(r"\b(dcd_[a-z0-9_]+)\s*\(", code))
    assert {"dcd_dgde_gmw_refine_workspace_bytes", "dcd_dgde_gmw_refine_fwd"} <= names
    assert " %d exported functions." % len(names) in src and len(names) == 31
    assert re.search(r"#define DCD_GMW_KPTS\s+73\b", src)
    assert set(names) == set(_lib.SIGNATURES)


def test_refine_entry_point_validates_before_any_cuda_call(lib):
    L = lib
    F = 256                      # a fake, aligned "device" address: every call below must fail before touching it
    n, depth, C = 73, 12, 415

    def call(N=4, n=n, k=1500, chunk=1024, B=1, bi=0, dims=F, ws=F, wsb=1 << 40, p4=F, out=F, C=C, ch2=50):
        return L.dcd_dgde_gmw_refine_fwd(F, F, bi, B, C, 96, 320, ch2, 196, 4, F, F, F, dims, p4, F, N, n, depth, k, chunk,
                                         out, F, F, F, 0, 0, 0, ws, wsb, 0)

    assert call(N=0) == 0                                            # nothing to do: no launch
    assert call(n=72) == DCD_E_INVALID                               # GMW reads keypoints 0..72
    assert call(n=257) == DCD_E_INVALID
    assert call(dims=0) == DCD_E_INVALID                             # the rescale needs h
    assert call(k=0) == DCD_E_INVALID and call(k=2629) == DCD_E_INVALID
    assert call(chunk=0) == DCD_E_INVALID
    assert call(B=2) == DCD_E_INVALID                                # several images need batch_idx
    assert call(ch2=C - 2 * n + 1) == DCD_E_INVALID                  # channel group past the map
    assert call(p4=F + 4) == DCD_E_INVALID                           # parameter blobs 16-byte aligned
    assert call(out=0) == DCD_E_INVALID
    assert call(ws=0) == DCD_E_INVALID
    assert call(wsb=16) == DCD_E_WORKSPACE
    assert call(ws=F + 64) == DCD_E_WORKSPACE
    assert L.dcd_dgde_gmw_refine_workspace_bytes(4, 72, depth, 1024) == 0
    assert L.dcd_dgde_gmw_refine_workspace_bytes(0, 73, depth, 1024) == 0
    # the workspace holds GMW's 73-keypoint inputs for all N objects, then dcd_gmw_depth_fwd's workspace for 73 keypoints
    for N, chunk, nk in ((4, 1024, 73), (301, 7, 73), (5, 1, 100)):
        kin = -(-N * 73 * 2 * 4 // 256) * 256 + -(-N * 73 * 3 * 4 // 256) * 256
        assert L.dcd_dgde_gmw_refine_workspace_bytes(N, nk, depth, chunk) == kin + L.dcd_gmw_depth_workspace_bytes(N, 73, depth, chunk)


@pytest.fixture
def no_library_call(monkeypatch):
    def forbidden():
        raise AssertionError("the library was reached")
    monkeypatch.setattr(ops._lib, "lib", forbidden)


def _inputs(N=3, requires_grad=None):
    t = {"pred_regression": torch.zeros(1, 415, 8, 8), "indexs": torch.arange(N), "pred_rots": torch.zeros(N),
         "P": torch.eye(3, 4), "pad_size": torch.zeros(2), "dims": torch.ones(N, 3)}
    if requires_grad:
        t[requires_grad] = t[requires_grad].clone().requires_grad_(True)
    return t


def test_refine_wrapper_rejects_bad_input_before_any_launch(no_library_call):
    gmw = dcd_b200.GMW()
    with pytest.raises(RuntimeError, match="CUDA tensors"):
        dcd_b200.refine_detections(gmw=gmw, **_inputs())
    t = _inputs()
    t["dims"] = None
    with pytest.raises(ValueError, match="dims"):
        dcd_b200.refine_detections(gmw=gmw, **t)
    with pytest.raises(ValueError, match="n >= 73"):
        dcd_b200.refine_detections(gmw=gmw, n=72, **_inputs())
    for name in ("pred_regression", "pred_rots", "dims"):
        with pytest.raises(RuntimeError, match="inference-only"):
            dcd_b200.refine_detections(gmw=gmw, **_inputs(requires_grad=name))
    with torch.no_grad():                                        # under no_grad the same inputs get as far as the device check
        with pytest.raises(RuntimeError, match="CUDA tensors"):
            dcd_b200.refine_detections(gmw=gmw, **_inputs(requires_grad="dims"))
