"""GPU tests of the plan-free correspondence branch: GMW.transport_terms, dcd_b200.correspondence_loss and
dcd_gmw_transport_terms_bwd.

The terms backward runs the dense backward's passes on the plan rebuilt from the forward's K, u and v (the forward's own two
roundings) and on dL/dP = alpha 11^T + beta I formed in registers.  With the same plan and the same dL/dP values its results
are therefore bit-identical to dcd_gmw_transport_bwd with a dense dL/dP, and the main bar here is torch.equal against that
path: through the C ABI, and end to end against GMW.forward with with_edge_P = True and the reference's correspondence loss
(there dL/dP = g (1 - 2 I), and alpha + beta = g - 2 g = -g exactly).  One test anchors the result to autograd through the
oracle's unrolled FP64 Sinkhorn independently of the dense path.
"""
import pytest
import torch

import dcd_b200
from dcd_b200 import _lib, ops, synth
from dcd_b200._lib import check, ptr, stream_ptr
from oracle import dcd_oracle as O
from oracle.make_golden import transport_inputs
from test_gpu_gmw import cu, make_model
from test_gpu_gmw_kpts_grad import _leaves
from test_gpu_transport import anchored_ok, n_of_edges

pytestmark = pytest.mark.gpu
DEV = "cuda"
LAMBDA, TOL, ITERS = 10.0, 1e-9, 100
CG_ITERS, CG_TOL = ops.SINKHORN_CG_ITERATIONS, ops.SINKHORN_CG_TOLERANCE


def nan_buffer(nbytes):
    return torch.full(((nbytes + 255) // 256 * 64,), float("nan"), device=DEV)


def abi_forward(a, c, with_P):
    """dcd_gmw_transport_fwd on channel-major features [N,128,E] -> (P or None, u, v, sums, forward workspace)."""
    L = _lib.lib()
    N, _, E = a.shape
    n = n_of_edges(E)
    P = torch.empty((N, E, E), device=DEV) if with_P else None
    u, v, sums = torch.empty((N, E), device=DEV), torch.empty((N, E), device=DEV), torch.empty((N, 2), device=DEV)
    tws = nan_buffer(L.dcd_gmw_transport_workspace_bytes(N, n))
    check(L.dcd_gmw_transport_fwd(ptr(a), ptr(c), N, n, LAMBDA, TOL, ITERS, ptr(P), ptr(u), ptr(v), ptr(sums), ptr(tws),
                                  tws.numel() * 4, stream_ptr()), "dcd_gmw_transport_fwd")
    return P, u, v, sums, tws


def abi_dense_bwd(a, c, P, u, v, V):
    L = _lib.lib()
    N, _, E = a.shape
    ga, gc, info = torch.empty_like(a), torch.empty_like(c), torch.empty((N, 8), device=DEV)
    ws = nan_buffer(L.dcd_gmw_transport_bwd_workspace_bytes(N, n_of_edges(E)))
    check(L.dcd_gmw_transport_bwd(ptr(a), ptr(c), ptr(P), ptr(u), ptr(v), ptr(V), N, n_of_edges(E), LAMBDA, CG_ITERS, CG_TOL,
                                  ptr(ga), ptr(gc), ptr(info), ptr(ws), ws.numel() * 4, stream_ptr()), "dcd_gmw_transport_bwd")
    return ga, gc, info


def abi_terms_bwd(a, c, tws, u, v, grad_terms):
    L = _lib.lib()
    N, _, E = a.shape
    ga, gc, info = torch.empty_like(a), torch.empty_like(c), torch.empty((N, 8), device=DEV)
    ws = nan_buffer(L.dcd_gmw_transport_bwd_workspace_bytes(N, n_of_edges(E)))
    check(L.dcd_gmw_transport_terms_bwd(ptr(a), ptr(c), ptr(tws), tws.numel() * 4, ptr(u), ptr(v), ptr(grad_terms), N,
                                        n_of_edges(E), LAMBDA, CG_ITERS, CG_TOL, ptr(ga), ptr(gc), ptr(info), ptr(ws),
                                        ws.numel() * 4, stream_ptr()), "dcd_gmw_transport_terms_bwd")
    return ga, gc, info


def features(E, N, seed, sharp=0.0):
    f4, f6, _ = transport_inputs(E, N, seed, sharp)
    return f4.transpose(1, 2).contiguous().to(DEV), f6.transpose(1, 2).contiguous().to(DEV)


@pytest.mark.parametrize("n,N,sharp", [(20, 3, 0.0), (40, 2, 0.0), (73, 2, 0.0), (73, 1, 0.03)])
def test_terms_backward_bit_identical_to_dense_backward(n, N, sharp):
    """E = 190 (E % 4 != 0: the scalar loops), 780 and 2628 (the float4 loops); sharp = 0.03: a nearly diagonal plan."""
    E = n * (n - 1) // 2
    a, c = features(E, N, 2100 + n, sharp)
    g = torch.Generator().manual_seed(n)
    alpha, beta = torch.randn(N, generator=g).to(DEV), torch.randn(N, generator=g).to(DEV)
    eye = torch.eye(E, device=DEV)
    V = alpha[:, None, None] * torch.ones(E, E, device=DEV) + beta[:, None, None] * eye
    P, u, v, sums, tws = abi_forward(a, c, with_P=True)
    dense = abi_dense_bwd(a, c, P, u, v, V)
    terms = abi_terms_bwd(a, c, tws, u, v, torch.stack((alpha, beta), 1).contiguous())
    torch.cuda.synchronize()
    info = terms[2].cpu()
    print("n=%d N=%d sharp=%g: cg iterations %s, converged %s" % (n, N, sharp, info[:, 3].tolist(), info[:, 2].tolist()))
    assert all(bool(torch.isfinite(t).all()) for t in terms[:2]) and float(terms[0].abs().max()) > 0
    assert torch.equal(dense[0], terms[0]) and torch.equal(dense[1], terms[1])
    assert torch.equal(dense[2][:, :4], terms[2][:, :4])                 # cg_info: |r|^2, |r0|^2, converged, iterations


def dense_forward_sums(model, k2, k3):
    """(sum P, trace P) of dcd_gmw_transport_fwd on the features of the saving (training) forward."""
    L = _lib.lib()
    N, n = k2.shape[0], k2.shape[1]
    E = n * (n - 1) // 2
    f4, f6 = torch.empty((N, 128, E), device=DEV), torch.empty((N, 128, E), device=DEV)
    w = torch.empty((N, E), device=DEV)
    ws = nan_buffer(L.dcd_gmw_workspace_bytes(N, n, model.depth, 1))
    with torch.no_grad():
        check(L.dcd_gmw_weights_fwd(ptr(k2), ptr(k3), ptr(model.params4), ptr(model.params6), N, n, model.depth, 1, ptr(w),
                                    ptr(f4), ptr(f6), ptr(ws), ws.numel() * 4, stream_ptr()), "dcd_gmw_weights_fwd")
    return abi_forward(f4, f6, with_P=False)[3]


def train_step(model, k2, k3, Z, idx, gt, w_cls, w_reg, plan_free, need_params=True, need_kpts=True):
    """loss = w_cls * correspondence loss + w_reg * reg loss, backward -> dict of gradients and forward outputs."""
    model.zero_grad(set_to_none=True)
    for p in model.parameters():
        p.requires_grad_(need_params)
    a, b = (_leaves(k2, k3) if need_kpts else (k2, k3))
    if plan_free:
        w, terms = model.transport_terms(a, b)
        cls = dcd_b200.correspondence_loss(terms)
        out = terms
    else:
        model.with_edge_P = True
        try:
            w, P = model(a, b)
        finally:
            model.with_edge_P = False
        cls = O.correspondence_loss(P, torch.eye(P.shape[1], device=DEV).expand_as(P))
        out = P
    loss = w_cls * cls
    if w_reg:
        loss = loss + w_reg * dcd_b200.compute_reg_loss(Z, w, gt, idx)[0]
    loss.backward()
    res = {"params4": model.params4.grad, "params6": model.params6.grad, "kpts_2d": a.grad if need_kpts else None,
           "kpts_3d": b.grad if need_kpts else None, "reg_weights": w.detach(), "out": out.detach(), "loss": loss.detach()}
    for p in model.parameters():
        p.requires_grad_(True)
    return res


def setup(n, depth, N, seed):
    ob = synth.make_objects(N=N, n=n, seed=seed)
    model = make_model(O.random_state_dict(seed % 1000, depth=depth), depth)
    k2, k3, rot, gt = cu(ob.kps_norm, ob.kps_3d, ob.rot_y, ob.gt_depth)
    with torch.no_grad():
        Z, idx = dcd_b200.compute_z(k2, k3, rot, num_k=min(1500, n * (n - 1) // 4))
    return model, k2, k3, Z, idx, gt


GRADS = ("params4", "params6", "kpts_2d", "kpts_3d")


@pytest.mark.parametrize("n,depth", [(20, 2), (73, 12)])
@pytest.mark.parametrize("w_cls,w_reg", [(1.0, 0.0), (0.1, 1.0)])
def test_transport_terms_end_to_end_bit_identical_to_edge_P(n, depth, w_cls, w_reg):
    model, k2, k3, Z, idx, gt = setup(n, depth, 2, 2200 + n)
    dense = train_step(model, k2, k3, Z, idx, gt, w_cls, w_reg, plan_free=False)
    terms = train_step(model, k2, k3, Z, idx, gt, w_cls, w_reg, plan_free=True)
    for key in GRADS:
        assert terms[key] is not None and float(terms[key].abs().max()) > 0, key
        assert torch.equal(terms[key], dense[key]), key
    assert torch.equal(terms["reg_weights"], dense["reg_weights"])
    assert torch.equal(terms["out"], dense_forward_sums(model, k2, k3))
    P = dense["out"].double()
    ref = torch.stack((P.sum((-2, -1)), P.diagonal(dim1=-2, dim2=-1).sum(-1)), 1)
    rel = float(((terms["out"].double() - ref).abs() / ref.abs()).max())
    print("n=%d depth %d cls %g reg %g: terms vs the plan's sums (FP64) %.3g, loss %.7g vs %.7g"
          % (n, depth, w_cls, w_reg, rel, float(terms["loss"]), float(dense["loss"])))
    assert rel < 1e-6
    assert abs(float(terms["loss"]) - float(dense["loss"])) <= 1e-5 * abs(float(dense["loss"]))


def test_transport_terms_keypoint_gradients_vs_fp64_unrolled_sinkhorn():
    """n = 73: loss = correspondence_loss(terms) + 0.1 reg through transport_terms against autograd through the oracle's
    UNROLLED Sinkhorn (O.gmw_edge_transport) in FP64, with the bar of
    test_gpu_gmw_kpts_grad.test_kpts_gradients_through_the_correspondence_branch."""
    n, N, depth, tol = 73, 2, 2, 5e-3
    ob = synth.make_objects(N=N, n=n, seed=1400 + n)
    sd = O.random_state_dict(70 + n, depth=depth)
    k2, k3, rot, gt = cu(ob.kps_norm, ob.kps_3d, ob.rot_y, ob.gt_depth)
    with torch.no_grad():
        Z, idx = dcd_b200.compute_z(k2, k3, rot, num_k=min(1500, n * (n - 1) // 4))
    model = make_model(sd, depth)
    a, b = _leaves(k2, k3)
    w, terms = model.transport_terms(a, b)
    (dcd_b200.correspondence_loss(terms) + 0.1 * dcd_b200.compute_reg_loss(Z, w, gt, idx)[0]).backward()
    mine = {"kpts_2d": a.grad, "kpts_3d": b.grad}
    E = n * (n - 1) // 2
    eye = torch.eye(E, device=DEV).expand(N, E, E)

    def oracle(dtype):
        ao, bo = _leaves(k2, k3, dtype)
        Po, wo = O.gmw_edge_transport(ao, bo, {k: v.to(device=DEV, dtype=dtype) for k, v in sd.items()}, depth)
        (O.correspondence_loss(Po, eye.to(dtype)) + 0.1 * O.compute_reg_loss(Z.to(dtype), wo, gt.to(dtype), idx)[0]).backward()
        return {"kpts_2d": ao.grad, "kpts_3d": bo.grad}

    ref64, ref32 = oracle(torch.float64), oracle(torch.float32)
    for key in ("kpts_2d", "kpts_3d"):
        ok, e_o, e_r = anchored_ok(mine[key], ref64[key], ref32[key], tol)
        print("transport_terms, cls + 0.1 reg, n=%d %s: ours vs f64 %.3g, FP32 oracle vs f64 %.3g" % (n, key, e_o, e_r))
        assert ok, (key, e_o, e_r)


def _partial_step(model, k2, k3, which, path, R):
    """path: "terms" (GMW.transport_terms), "plan" (GMW.forward with with_edge_P) or "weights" (GMW.forward without it)."""
    model.zero_grad(set_to_none=True)
    a, b = _leaves(k2, k3)
    if path == "terms":
        w, terms = model.transport_terms(a, b)
        loss = {"trace": lambda: terms[:, 1].sum(), "sum": lambda: terms[:, 0].sum(), "reg": lambda: (w * R).sum()}[which]()
    else:
        model.with_edge_P = path == "plan"
        try:
            w, P = model(a, b)
        finally:
            model.with_edge_P = False
        loss = {"trace": lambda: P.diagonal(dim1=-2, dim2=-1).sum(), "sum": lambda: P.sum(), "reg": lambda: (w * R).sum()}[which]()
    loss.backward()
    return {"params4": model.params4.grad.clone(), "params6": model.params6.grad.clone(), "kpts_2d": a.grad, "kpts_3d": b.grad}


@pytest.mark.parametrize("which", ["trace", "sum", "reg"])
def test_partial_cotangents(which, monkeypatch):
    """A loss on trace P only (dL/dP = g I), on sum P only (g 11^T), or on reg_weights only: bit-identical to the dense path
    (GMW.forward with with_edge_P).  The reg-only loss runs no transport backward on either path, and equals GMW.forward
    without with_edge_P bit for bit."""
    n, depth, N = 40, 2, 2
    model, k2, k3, _, _, _ = setup(n, depth, N, 2300)
    R = torch.randn(N, n * (n - 1) // 2, generator=torch.Generator().manual_seed(23)).to(DEV)
    L = _lib.lib()
    calls = {"dcd_gmw_transport_bwd": 0, "dcd_gmw_transport_terms_bwd": 0}
    for name in calls:
        def counted(*args, _name=name, _real=getattr(L, name)):
            calls[_name] += 1
            return _real(*args)

        monkeypatch.setattr(L, name, counted)
    expected = 0 if which == "reg" else 1
    dense = _partial_step(model, k2, k3, which, "plan", R)
    assert calls["dcd_gmw_transport_bwd"] == expected
    terms = _partial_step(model, k2, k3, which, "terms", R)
    assert calls["dcd_gmw_transport_terms_bwd"] == expected
    others = [dense] + ([_partial_step(model, k2, k3, which, "weights", R)] if which == "reg" else [])
    for key in GRADS:
        assert float(terms[key].abs().max()) > 0, key
        for other in others:
            assert torch.equal(terms[key], other[key]), key


def test_frozen_parameters_and_frozen_keypoints():
    """Frozen parameters with keypoints that require grad: no parameter .grad, keypoint gradients of the trainable run bit
    for bit.  And the reverse: keypoints without grad, parameter gradients of the full run bit for bit."""
    model, k2, k3, Z, idx, gt = setup(73, 12, 2, 2400)
    full = train_step(model, k2, k3, Z, idx, gt, 0.1, 1.0, plan_free=True)
    frozen = train_step(model, k2, k3, Z, idx, gt, 0.1, 1.0, plan_free=True, need_params=False)
    assert frozen["params4"] is None and frozen["params6"] is None
    assert torch.equal(frozen["kpts_2d"], full["kpts_2d"]) and torch.equal(frozen["kpts_3d"], full["kpts_3d"])
    fixed = train_step(model, k2, k3, Z, idx, gt, 0.1, 1.0, plan_free=True, need_kpts=False)
    assert torch.equal(fixed["params4"], full["params4"]) and torch.equal(fixed["params6"], full["params6"])


def test_no_grad_empty_poisoned_and_rerun(monkeypatch):
    n, depth, N = 73, 12, 3
    model, k2, k3, Z, idx, gt = setup(n, depth, N, 2500)
    E = n * (n - 1) // 2
    # torch.no_grad(): edge_transport(materialise=False) bit for bit, nothing kept beyond the two outputs
    with torch.no_grad():
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated()
        w, terms = model.transport_terms(k2, k3)
        torch.cuda.synchronize()
        kept = torch.cuda.memory_allocated() - before
        w0, P0, sums0 = model.edge_transport(k2, k3, materialise=False)
    assert P0 is None and not w.requires_grad and not terms.requires_grad
    assert torch.equal(w, w0) and torch.equal(terms, sums0)
    assert kept <= (N * E * 4 + 511) // 512 * 512 + 512, kept
    # N = 0: empty outputs, with and without autograd
    k2e, k3e = k2[:0], k3[:0]
    with torch.no_grad():
        we, te = model.transport_terms(k2e, k3e)
    assert we.shape == (0, E) and te.shape == (0, 2)
    model.zero_grad(set_to_none=True)
    we, te = model.transport_terms(k2e, k3e)
    assert we.shape == (0, E) and te.shape == (0, 2)
    (we.sum() + te.sum()).backward()
    assert float(model.params4.grad.abs().max()) == 0
    # NaN-poisoned workspaces change nothing; reruns are bit-identical
    first = train_step(model, k2, k3, Z, idx, gt, 0.1, 1.0, plan_free=True)
    again = train_step(model, k2, k3, Z, idx, gt, 0.1, 1.0, plan_free=True)
    monkeypatch.setattr(ops, "POISON_WORKSPACES", True)
    poisoned = train_step(model, k2, k3, Z, idx, gt, 0.1, 1.0, plan_free=True)
    for key in GRADS + ("reg_weights", "out"):
        assert torch.equal(again[key], first[key]), key
        assert torch.equal(poisoned[key], first[key]), key


@pytest.mark.parametrize("w_cls,w_reg", [(1.0, 0.0), (0.1, 1.0)])
def test_graphed_step_correspondence_loss(w_cls, w_reg):
    """GraphedGmwStep with a correspondence loss: replayed gradients equal the eager terms step's and the eager dense step's
    (edge_P + correspondenceLoss, GMW/main.py:456-457) bit for bit; the loss matches both to rel 1e-5."""
    n, depth, b = 73, 12, 8
    ob = synth.make_objects(N=b, n=n, seed=2600)
    model = make_model(O.random_state_dict(26, depth=depth), depth)
    k2, k3, rot, gt = cu(ob.kps_norm, ob.kps_3d, ob.rot_y, ob.gt_depth)

    def eager_step(plan_free):                                # returns nothing that keeps its autograd graph alive
        model.zero_grad(set_to_none=True)
        Z, idx = dcd_b200.compute_z(k2, k3, rot)
        if plan_free:
            w, terms = model.transport_terms(k2, k3)
            cls = dcd_b200.correspondence_loss(terms)
        else:
            model.with_edge_P = True
            try:
                w, P = model(k2, k3)
            finally:
                model.with_edge_P = False
            cls = O.correspondence_loss(P, torch.eye(P.shape[1], device=DEV).expand_as(P))
        reg, _ = dcd_b200.compute_reg_loss(Z, w, gt, idx)
        loss = w_reg * reg + w_cls * cls
        loss.backward()
        return float(loss.detach()), (model.params4.grad.clone(), model.params6.grad.clone())

    loss_terms, terms = eager_step(True)
    loss_dense, dense = eager_step(False)
    model.zero_grad(set_to_none=True)
    step = dcd_b200.GraphedGmwStep(model, batch=b, n=n, cls_weight=w_cls, reg_weight=w_reg)
    step(k2, k3, rot, gt)
    loss_graph = float(step(k2, k3, rot, gt))                 # a second replay: nothing accumulates
    torch.cuda.synchronize()
    graph = (model.params4.grad.clone(), model.params6.grad.clone())
    print("graphed step, cls %g reg %g: loss graphed %.7g, eager terms %.7g, eager dense %.7g"
          % (w_cls, w_reg, loss_graph, loss_terms, loss_dense))
    for x, y, z in zip(graph, terms, dense):
        assert float(x.abs().max()) > 0
        assert torch.equal(x, y) and torch.equal(x, z)
    assert abs(loss_graph - loss_dense) <= 1e-5 * abs(loss_dense)
    assert abs(loss_graph - loss_terms) <= 1e-5 * abs(loss_terms)


def _peak_bytes(fn):
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def test_memory_of_one_cls_step():
    """One cls-only training step at n = 73, b = 8: the terms path's peak is at least one [b,E,E] FP32 tensor below the dense
    path's (expected: about four)."""
    n, depth, b = 73, 12, 8
    E = n * (n - 1) // 2
    model, k2, k3, Z, idx, gt = setup(n, depth, b, 2700)
    peaks = {}
    for plan_free in (False, True):
        peaks[plan_free] = _peak_bytes(lambda: train_step(model, k2, k3, Z, idx, gt, 1.0, 0.0, plan_free=plan_free))
    print("cls step n=73 b=8: peak above the inputs, dense %.1f MB, terms %.1f MB, one [b,E,E] tensor %.1f MB"
          % (peaks[False] / 1e6, peaks[True] / 1e6, b * 4 * E * E / 1e6))
    assert peaks[False] - peaks[True] >= b * 4 * E * E


def test_n256_single_object():
    """n = 256 (E = 32 640), N = 1 through the C ABI: the terms backward runs and its feature gradients equal the dense
    backward's bit for bit.  The dense side holds K, P and a dense V, 4.26 GB each."""
    n, N = 256, 1
    E = n * (n - 1) // 2
    need = 4 * (4 * E * E) + (1 << 30)
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip("needs %.1f GB free, %.1f GB available" % (need / 1e9, free / 1e9))
    g = torch.Generator().manual_seed(2800)          # features as oracle.make_golden.transport_inputs draws them, without its E x E V
    f4 = torch.randn(N, E, 128, generator=g) * (0.5 + torch.rand(N, E, 1, generator=g))
    f6 = torch.randn(N, E, 128, generator=g) * 1.3
    a, c = f4.transpose(1, 2).contiguous().to(DEV), f6.transpose(1, 2).contiguous().to(DEV)
    alpha, beta = torch.tensor([0.37], device=DEV), torch.tensor([-0.74], device=DEV)
    P, u, v, sums, tws = abi_forward(a, c, with_P=True)
    V = torch.full((N, E, E), float(alpha), device=DEV)
    V.diagonal(dim1=1, dim2=2).fill_(float(alpha + beta))     # alpha 11^T + beta I with the FP32 sum on the diagonal
    dense = abi_dense_bwd(a, c, P, u, v, V)
    del V, P
    terms = abi_terms_bwd(a, c, tws, u, v, torch.stack((alpha, beta), 1).contiguous())
    torch.cuda.synchronize()
    print("n=256: cg iterations %s" % terms[2][:, 3].tolist())
    assert bool(torch.isfinite(terms[0]).all()) and float(terms[0].abs().max()) > 0
    assert torch.equal(dense[0], terms[0]) and torch.equal(dense[1], terms[1])
    assert torch.equal(dense[2][:, :4], terms[2][:, :4])
