"""GPU parity of the keypoint gradients of GMW.forward and compute_z (dcd_gmw_kpts_bwd, dcd_edge_solve_bwd with K = NULL).

Oracle: autograd through oracle/dcd_oracle.py w.r.t. kpts_2d / kpts_3d, in FP64 and in FP32 on CUDA (TF32 off: the
reference's arithmetic).  Bar: the per-tensor FP64 anchor of test_gpu_gmw._anchored,
    |ours - f64|_max <= max(4 |FP32 oracle - f64|_max, 1e-4 max|f64|),
and on small nets whose ReLU inputs keep a margin from zero a direct 1e-4 max|f64| (DESIGN.md section 2, "Gradients": a
ReLU input within FP32 noise of 0 flips and moves the gradient by far more than rounding, in the reference's own FP32 run
as much as here).
"""
import pytest
import torch

import dcd_b200
from dcd_b200 import patch, synth
from oracle import dcd_oracle as O
from test_gpu_gmw import _anchored, _relu_margin, cu, make_model
from test_gpu_patch import reference_shaped_gmw
from test_gpu_transport import anchored_ok

pytestmark = pytest.mark.gpu
DEV = "cuda"
KEYS = ("kpts_2d", "kpts_3d")


def _cotangent(N, E, seed):
    return torch.randn(N, E, generator=torch.Generator().manual_seed(seed)).to(DEV)


def _leaves(k2, k3, dtype=torch.float32):
    return k2.detach().to(dtype).clone().requires_grad_(True), k3.detach().to(dtype).clone().requires_grad_(True)


def ours_grads(model, k2, k3, R, dtype=torch.float32):
    """d/dkeypoints of sum(reg_weights * R) through dcd_b200.GMW."""
    a, b = _leaves(k2, k3, dtype)
    w, _ = model(a, b)
    (w * R).sum().backward()
    return {"kpts_2d": a.grad, "kpts_3d": b.grad}


def oracle_grads(k2, k3, sd, depth, R, dtype):
    """The same by autograd through the oracle, on CUDA, in `dtype`."""
    a, b = _leaves(k2.to(DEV), k3.to(DEV), dtype)
    w = O.gmw_reg_weights(a, b, {k: v.to(device=DEV, dtype=dtype) for k, v in sd.items()}, depth)
    (w * R.to(dtype)).sum().backward()
    return {"kpts_2d": a.grad, "kpts_3d": b.grad}


def assert_anchored(mine, ref32, ref64, what):
    worst_o, worst_r, bad = _anchored(mine, ref32, ref64)
    print("%s: keypoint gradients, worst tensor ours vs f64 %.3g, FP32 oracle vs f64 %.3g" % (what, worst_o, worst_r))
    assert not bad, bad


@pytest.mark.parametrize("n,depth,N", [(12, 2, 3), (20, 1, 2), (16, 3, 2)])
def test_kpts_gradients_small_well_posed(n, depth, N):
    # the first seed whose ReLU inputs keep a margin, as test_gpu_gmw.test_weight_gradients_small_well_posed picks it
    for seed in range(200, 260):
        ob = synth.make_objects(N=N, n=n, seed=seed)
        sd = O.random_state_dict(seed, depth=depth)
        if _relu_margin(ob.kps_norm, ob.kps_3d, sd, depth) > 2e-5:
            break
    else:
        pytest.skip("no seed with a ReLU margin found")
    k2, k3 = cu(ob.kps_norm, ob.kps_3d)
    R = _cotangent(N, n * (n - 1) // 2, seed)
    mine = ours_grads(make_model(sd, depth), k2, k3, R)
    ref64 = oracle_grads(k2, k3, sd, depth, R, torch.float64)
    ref32 = oracle_grads(k2, k3, sd, depth, R, torch.float32)
    for key in KEYS:
        amax = float(ref64[key].abs().max())
        e64 = float((mine[key].double() - ref64[key]).abs().max())
        e32 = float((mine[key] - ref32[key]).abs().max())
        print("n=%d depth %d seed %d %s: ours vs f64 %.3g, vs FP32 oracle %.3g (of max|f64|)" % (n, depth, seed, key, e64 / amax,
                                                                                                 e32 / amax))
        assert e64 <= 1e-4 * amax, key
        assert e32 <= 2e-4 * amax, key


@pytest.mark.parametrize("n,depth,N", [(73, 12, 4), (256, 12, 2), (40, 2, 2), (56, 2, 2), (74, 2, 2), (100, 2, 2)])
def test_kpts_gradients_fp64_anchored(n, depth, N):
    """The reference's size (n = 73, depth 12), the stress shape (n = 256, E = 32 640) and other n at depth 2 (the edge-axis
    padding of the last tile differs for each: E % 128 = 20, 0, 12, 92, 99, 86)."""
    ob = synth.make_objects(N=N, n=n, seed=1300 + n)
    sd = O.random_state_dict(60 + n, depth=depth)
    k2, k3 = cu(ob.kps_norm, ob.kps_3d)
    R = _cotangent(N, n * (n - 1) // 2, n)
    mine = ours_grads(make_model(sd, depth), k2, k3, R)
    assert all(bool(torch.isfinite(v).all()) for v in mine.values())
    assert_anchored(mine, oracle_grads(k2, k3, sd, depth, R, torch.float32), oracle_grads(k2, k3, sd, depth, R, torch.float64),
                    "n=%d depth %d N=%d" % (n, depth, N))


@pytest.mark.parametrize("n,N,tol", [(20, 2, 1e-3), (73, 2, 5e-3)])
def test_kpts_gradients_through_the_correspondence_branch(n, N, tol):
    """with_edge_P: loss = correspondenceLoss(edge_P, eye) + 0.1 reg (GMW/main.py:453-461), keypoint gradients through the
    implicit Sinkhorn backward and the MLP, against autograd through the oracle's UNROLLED Sinkhorn in FP64; bar in the
    style of test_gpu_transport.anchored_ok (|ours - f64| <= max(2 |FP32 oracle - f64|, tol max|f64|))."""
    depth = 2
    ob = synth.make_objects(N=N, n=n, seed=1400 + n)
    sd = O.random_state_dict(70 + n, depth=depth)
    k2, k3, rot, gt = cu(ob.kps_norm, ob.kps_3d, ob.rot_y, ob.gt_depth)
    num_k = min(1500, n * (n - 1) // 4)
    with torch.no_grad():
        Z, idx = dcd_b200.compute_z(k2, k3, rot, num_k=num_k)
    model = make_model(sd, depth)
    model.with_edge_P = True
    a, b = _leaves(k2, k3)
    w, P = model(a, b)
    eye = torch.eye(P.shape[1], device=DEV).expand_as(P)
    (O.correspondence_loss(P, eye) + 0.1 * dcd_b200.compute_reg_loss(Z, w, gt, idx)[0]).backward()
    mine = {"kpts_2d": a.grad, "kpts_3d": b.grad}

    def oracle(dtype):
        ao, bo = _leaves(k2, k3, dtype)
        Po, wo = O.gmw_edge_transport(ao, bo, {k: v.to(device=DEV, dtype=dtype) for k, v in sd.items()}, depth)
        (O.correspondence_loss(Po, eye.to(dtype)) + 0.1 * O.compute_reg_loss(Z.to(dtype), wo, gt.to(dtype), idx)[0]).backward()
        return {"kpts_2d": ao.grad, "kpts_3d": bo.grad}

    ref64, ref32 = oracle(torch.float64), oracle(torch.float32)
    for key in KEYS:
        ok, e_o, e_r = anchored_ok(mine[key], ref64[key], ref32[key], tol)
        print("cls + 0.1 reg, n=%d %s: ours vs f64 %.3g, FP32 oracle vs f64 %.3g" % (n, key, e_o, e_r))
        assert ok, (key, e_o, e_r)


def test_kpts_gradients_end_to_end_through_compute_z_and_gmw():
    """compute_z -> GMW -> compute_reg_loss (GMW/main.py:453-461): the gradient reaches kpts_2d / kpts_3d through both the
    edge depths and the edge weights, against the same composition of oracle functions (differentiable O.compute_z)."""
    n, depth, N = 73, 12, 2
    ob = synth.make_objects(N=N, n=n, seed=1500)
    sd = O.random_state_dict(81, depth=depth)
    k2, k3, rot, gt = cu(ob.kps_norm, ob.kps_3d, ob.rot_y, ob.gt_depth)
    a, b = _leaves(k2, k3)
    Z, idx = dcd_b200.compute_z(a, b, rot)
    assert Z.requires_grad
    w, _ = make_model(sd, depth)(a, b, rot, None)
    dcd_b200.compute_reg_loss(Z, w, gt, idx)[0].backward()
    mine = {"kpts_2d": a.grad, "kpts_3d": b.grad}
    assert torch.equal(idx, O.compute_z(k2, k3, rot)[1])

    def oracle(dtype):
        ao, bo = _leaves(k2, k3, dtype)
        Zo, _ = O.compute_z(ao, bo, rot.to(dtype))
        wo = O.gmw_reg_weights(ao, bo, {k: v.to(device=DEV, dtype=dtype) for k, v in sd.items()}, depth)
        O.compute_reg_loss(Zo, wo, gt.to(dtype), idx)[0].backward()
        return {"kpts_2d": ao.grad, "kpts_3d": bo.grad}

    assert_anchored(mine, oracle(torch.float32), oracle(torch.float64), "compute_z -> GMW -> reg loss, n=73 depth 12")


def test_compute_z_gradient():
    """compute_z alone: Z_v_raw is differentiable like the reference's (GMW/main.py:373-411); the values of Z and idx do
    not change with autograd on; the u column's gradient is exactly 0; pred_rot receives none."""
    n, N = 73, 6
    ob = synth.make_objects(N=N, n=n, seed=1600)
    k2, k3, rot = cu(ob.kps_norm, ob.kps_3d, ob.rot_y)
    with torch.no_grad():
        Z0, idx0 = dcd_b200.compute_z(k2, k3, rot)
    a, b = _leaves(k2, k3)
    r = rot.clone().requires_grad_(True)
    Z, idx = dcd_b200.compute_z(a, b, r)
    assert torch.equal(Z.detach(), Z0) and torch.equal(idx, idx0)
    R = _cotangent(N, Z.shape[1], 16)
    (Z * R).sum().backward()
    ao, bo = _leaves(k2, k3)
    (O.compute_z(ao, bo, rot)[0] * R).sum().backward()
    for mine, ref in ((a.grad, ao.grad), (b.grad, bo.grad)):
        assert float((mine - ref).abs().max()) <= 1e-4 * float(ref.abs().max())
    assert bool((a.grad[:, :, 0] == 0).all()) and float(a.grad[:, :, 1].abs().max()) > 0
    assert r.grad is None


def test_frozen_parameters_and_no_side_effects():
    """A trained GMW as a differentiable refiner: frozen parameters, keypoints that require grad.  The backward runs (the
    saving forward is taken), the keypoint gradients are those of the run with trainable parameters bit for bit, the
    parameters get no .grad; requesting keypoint gradients leaves the parameter gradients bit-identical; one keypoint
    tensor alone gets the same gradient as with both; repeated runs are bit-identical."""
    n, depth, N = 73, 12, 4
    ob = synth.make_objects(N=N, n=n, seed=1700)
    model = make_model(O.random_state_dict(82, depth=depth), depth)
    k2, k3 = cu(ob.kps_norm, ob.kps_3d)
    R = _cotangent(N, n * (n - 1) // 2, 17)

    def run(need2=True, need3=True):
        model.zero_grad(set_to_none=True)
        a, b = k2.clone().requires_grad_(need2), k3.clone().requires_grad_(need3)
        w, _ = model(a, b)
        (w * R).sum().backward()
        g4 = None if model.params4.grad is None else model.params4.grad.clone()
        g6 = None if model.params6.grad is None else model.params6.grad.clone()
        return a.grad, b.grad, g4, g6

    full = run()
    again = run()
    params_only = run(False, False)
    only3 = run(False, True)
    only2 = run(True, False)
    assert all(torch.equal(x, y) for x, y in zip(full, again))
    assert torch.equal(params_only[2], full[2]) and torch.equal(params_only[3], full[3])
    assert only3[0] is None and torch.equal(only3[1], full[1]) and only2[1] is None and torch.equal(only2[0], full[0])
    for p in model.parameters():
        p.requires_grad_(False)
    frozen = run()
    assert frozen[2] is None and frozen[3] is None
    assert torch.equal(frozen[0], full[0]) and torch.equal(frozen[1], full[1])
    frozen3 = run(False, True)
    assert torch.equal(frozen3[1], full[1])


def test_inference_with_grad_requiring_keypoints_is_untouched():
    """Under torch.no_grad() keypoints that require grad do not switch to the saving forward: bit-identical weights."""
    n, N = 73, 25
    ob = synth.make_objects(N=N, n=n, seed=1800)
    model = make_model(O.random_state_dict(83))
    k2, k3 = cu(ob.kps_norm, ob.kps_3d)
    a, b = _leaves(k2, k3)
    with torch.no_grad():
        plain, _ = model(k2, k3)
        w, _ = model(a, b)
    assert not w.requires_grad and torch.equal(w, plain)


@pytest.mark.parametrize("with_edge_P", [False, True])
def test_kpts_gradients_through_the_patch(with_edge_P):
    """patch.install(gmw_model=...) on a module with the reference GMW's parameter tree: its forward goes through
    GMW.forward_blobs, so keypoint gradients arrive exactly as through dcd_b200.GMW with the same weights."""
    n, depth, N = 20, 2, 2
    sd = O.random_state_dict(84, depth=depth)
    ob = synth.make_objects(N=N, n=n, seed=1900)
    k2, k3, rot = cu(ob.kps_norm, ob.kps_3d, ob.rot_y)
    R = _cotangent(N, n * (n - 1) // 2, 19)

    def grads(module):
        a, b = _leaves(k2, k3)
        w, P = module(a, b, rot, None)
        loss = (w * R).sum()
        if with_edge_P:
            loss = loss + O.correspondence_loss(P, torch.eye(P.shape[1], device=DEV).expand_as(P))
        loss.backward()
        return a.grad, b.grad

    ref_module = reference_shaped_gmw(sd, depth).to(DEV)
    patch.install(gmw_model=ref_module, with_edge_P=with_edge_P)
    try:
        via_patch = grads(ref_module)
    finally:
        patch.uninstall()
    model = make_model(sd, depth)
    model.with_edge_P = with_edge_P
    direct = grads(model)
    assert all(bool(torch.isfinite(g).all()) for g in via_patch)
    assert torch.equal(via_patch[0], direct[0]) and torch.equal(via_patch[1], direct[1])


def test_float64_keypoints_get_float64_gradients():
    """The FP32 cast stays in the graph: float64 keypoints receive float64 gradients, equal to the FP32 run's."""
    n, depth, N = 40, 2, 3
    ob = synth.make_objects(N=N, n=n, seed=2000)
    model = make_model(O.random_state_dict(85, depth=depth), depth)
    k2, k3 = cu(ob.kps_norm, ob.kps_3d)
    R = _cotangent(N, n * (n - 1) // 2, 20)
    g32 = ours_grads(model, k2, k3, R)
    g64 = ours_grads(model, k2, k3, R, torch.float64)
    for key in KEYS:
        assert g64[key].dtype == torch.float64 and torch.equal(g64[key], g32[key].double())
