"""FP64 parity of the GMW MLP backward (gmw_mlp_bwd_tc.cu) at the tile and CTA layouts that training runs.

mlp_bwd_tc_kernel cuts the N T tiles of 128 edges (T = ceil(E / 128)) into contiguous ranges, one per CTA, with
min(N T, SMs / 2) CTAs per net.  Three paths depend on where those ranges fall: the weight gradient accumulates in tensor
memory across a CTA's tiles, a range that crosses an object boundary reloads that object's context-norm statistics, and
the padded columns of a partial last tile are masked out of the weight gradient, the data gradient and the running maximum.
BWD_GEOMETRY lists keypoint counts whose tail E % 128 differs; `regime_N` picks N per n so that each of the four range
layouts occurs (fewer tiles than CTAs, exactly one tile per CTA, ranges crossing objects, many tiles per CTA with ranges
ending inside objects).

Random keypoints put some ReLU input within FP32 rounding noise of zero at these sizes, which makes the FP32 oracle itself
1-3 % off FP64 (DESIGN.md section 2) and leaves only a loose bar.  Quantised objects (`quantised_objects`: each object's n
keypoints drawn from `pool` distinct values) have at most pool^2 distinct edge features, so a seeded search finds weights and
keypoints whose FP64 ReLU margin is well above rounding noise (`pinned_case`); E, the tile layout, the statistics over all E
edges and a random per-edge cotangent are unchanged, so a dropped, duplicated or misplaced edge still changes the result.
A batch is made of copies of 1-3 such base objects in turn, each copy with its own cotangent: a copy's forward is its
base's, so the FP64 parameter gradient is sum_b J_b^T (sum over the copies of b of R) -- one oracle run per base, whatever N.

Bar, per tensor: |ours - f64|_max <= max(2 |FP32 oracle - f64|_max, floor max|f64|), dead block biases against the global max
(test_gpu_gmw._anchored with c = 2).  floor = 1e-4, and 2e-4 for parameter gradients that sum over more than 2^16 edges (N E):
there the FP16x3 split's dropped lo x lo products add up to ~1.1e-4 of the first preconv weight's max (measured on B200 at
n = 73 N = 64 and n = 256 N = 3, depth 2-3) while the FP32 oracle's blocked sums stay at 2-5e-5.
"""
import functools

import pytest
import torch

from dcd_b200 import synth
from oracle import dcd_oracle as O
from test_gpu_gmw import _anchored, _relu_margin, cu, make_model
from test_gpu_gmw_kpts_grad import _cotangent, ours_grads, oracle_grads

pytestmark = pytest.mark.gpu
DEV = "cuda"
TE = 128                                   # edges per tile of the layer-wise kernels
KEYS = ("kpts_2d", "kpts_3d")
B200_SMS = 148

# n, E = n (n - 1) / 2, T = ceil(E / 128), E % 128 (the valid columns of the last tile; 0 = full)
BWD_GEOMETRY = (
    (16, 120, 1, 120),        # one partial tile per object
    (17, 136, 2, 8),
    (23, 253, 2, 125),
    (33, 528, 5, 16),
    (46, 1035, 9, 11),
    (73, 2628, 21, 68),       # the reference's keypoint count
    (74, 2701, 22, 13),
    (100, 4950, 39, 86),
    (129, 8256, 65, 64),
    (256, 32640, 255, 0),     # the stress shape: every tile full, T > SMs / 2
)
assert all(E == n * (n - 1) // 2 and T == -(-E // TE) and tail == E % TE for n, E, T, tail in BWD_GEOMETRY)
GEOMETRY_T = {n: T for n, _, T, _ in BWD_GEOMETRY}
REGIMES = ("under", "exact", "cross", "many")

# FP64 ReLU margin a pinned case must exceed: two orders above the FP32 rounding noise of a normalised activation (~1e-7).
# The same 2e-5 serves at depth 12 (24 norms per net): with pool 4 the first seeds reach 3-4e-5 at n = 73 and n = 256.
MARGIN = 2e-5
POOL = {1: 6, 2: 6, 3: 6, 12: 4}


def bwd_ctas(N, T, sms):
    """CTAs per net of mlp_bwd_tc_kernel (bwd_tc_ctas, capped at 128 like launch_gmw_weights_bwd)."""
    return min(N * T, max(1, sms // 2), 128)


def cta_ranges(N, T, sms):
    """[t_begin, t_end) tile range of every CTA, as mlp_bwd_tc_kernel splits the N T tiles."""
    nt, c = N * T, bwd_ctas(N, T, sms)
    return [(nt * b // c, nt * (b + 1) // c) for b in range(c)]


def crosses_objects(N, T, sms):
    """Some CTA range holds tiles of two objects (the statistics reload inside a range)."""
    return any(lo // T != (hi - 1) // T for lo, hi in cta_ranges(N, T, sms))


def ends_inside_objects(N, T, sms):
    """Some CTA range starts in the middle of an object (the accumulator restarts mid-object)."""
    return any(lo % T for lo, _ in cta_ranges(N, T, sms))


def regime_N(T, regime, sms):
    """N for one range layout of the backward's N T tiles over C = min(SMs / 2, 128) CTAs, or None where n cannot have it:
    under: N T < C (one tile per CTA, some CTAs idle); exact: N T = C; cross: C < N T < 2 C with a range crossing an object
    boundary; many: N T >= 4 C (several tiles per CTA; for T > 1 with ranges that begin inside an object)."""
    C = min(max(1, sms // 2), 128)
    if regime == "under":
        return (C - 1) // T if T < C else None
    if regime == "exact":
        return C // T if C % T == 0 else None
    if regime == "cross":
        return next((N for N in range(C // T + 1, -(-2 * C // T)) if N * T < 2 * C and crosses_objects(N, T, sms)), None)
    if regime == "many":
        N = -(-4 * C // T)
        while T > 1 and not (ends_inside_objects(N, T, sms) and crosses_objects(N, T, sms)):
            N += 1
        return N
    raise ValueError(regime)


def quantised_objects(N, n, pool, seed):
    """(kpts_2d [N,n,2], kpts_3d [N,n,3]): each object's n keypoints are drawn from `pool` keypoints of a synth object
    (projection-consistent 2D and 3D), every pool value used at least once, with the same index pattern in 2D and 3D."""
    assert 1 < pool <= n
    ob = synth.make_objects(N=N, n=pool, seed=seed)
    g = torch.Generator().manual_seed(seed)
    idx = torch.stack([torch.cat((torch.arange(pool), torch.randint(pool, (n - pool,), generator=g)))[torch.randperm(n, generator=g)]
                       for _ in range(N)])
    k2 = ob.kps_norm.gather(1, idx[..., None].expand(N, n, 2))
    k3 = ob.kps_3d.gather(1, idx[..., None].expand(N, n, 3))
    return k2.contiguous(), k3.contiguous()


@functools.lru_cache(maxsize=None)
def pinned_case(n, depth, bases, pool=None, margin=None, seeds=64):
    """The first seed (0, 1, ...) whose `bases` quantised objects and random weights keep every FP64 ReLU input at least
    `margin` away from zero -> (kpts_2d, kpts_3d, state_dict, seed, margin found); CPU tensors."""
    pool, margin = pool or POOL[depth], margin or MARGIN
    for seed in range(seeds):
        k2, k3 = quantised_objects(bases, n, pool, 7000 + seed)
        sd = O.random_state_dict(seed, depth=depth)
        m = _relu_margin(k2, k3, sd, depth)
        if m > margin:
            print("pinned n=%d depth %d bases %d pool %d: seed %d, FP64 ReLU margin %.3g" % (n, depth, bases, pool, seed, m))
            return k2, k3, sd, seed, m
    raise AssertionError("no seed with a ReLU margin > %g (n=%d depth %d)" % (margin, n, depth))


def bases_for(n, N, depth):
    """Base objects of a batch: 3 in turn (neighbours always differ), fewer for N < 3.  At depth 12 two (n = 73), or one
    (n = 256: the FP64 oracle keeps ~13 GB of activations per object)."""
    return min(N, 3 if depth <= 3 else (2 if n < 256 else 1))


def boundary_objects(N, T, sms, limit=10):
    """Objects 0 and N - 1 and up to `limit` objects at CTA range boundaries: those a range begins inside (their tiles are
    split over two CTAs) and those that follow another object within one range."""
    at = set()
    for lo, hi in cta_ranges(N, T, sms):
        if lo % T:
            at.add(lo // T)
        if lo // T != (hi - 1) // T:
            at.add((hi - 1) // T)
    at = sorted(at - {0, N - 1})
    if len(at) > limit:
        at = [at[i * len(at) // limit] for i in range(limit)]
    return sorted({0, N - 1, *at})


def sm_count():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def oracle_param_grads(k2, k3, sd, depth, R, dtype):
    """Parameter gradients of sum(reg_weights * R) by autograd through the oracle, on CUDA, in `dtype`."""
    sdg = {k: v.to(device=DEV, dtype=dtype).clone().requires_grad_(True) for k, v in sd.items()}
    w = O.gmw_reg_weights(k2.to(device=DEV, dtype=dtype), k3.to(device=DEV, dtype=dtype), sdg, depth)
    (w * R.to(device=DEV, dtype=dtype)).sum().backward()
    return {k: v.grad for k, v in sdg.items()}


def run_copies(n, depth, N, R=None, bases=None):
    """Copies of `bases` pinned objects in turn, one forward + backward of sum(reg_weights * R) through dcd_b200.GMW
    -> (case, pick [N] base of each copy, R, parameter gradients, keypoint gradients)."""
    bases = bases or bases_for(n, N, depth)
    case = pinned_case(n, depth, bases)
    k2b, k3b, sd, seed, _ = case
    pick = torch.arange(N) % bases
    k2, k3 = cu(k2b[pick].contiguous(), k3b[pick].contiguous())
    if R is None:
        R = _cotangent(N, n * (n - 1) // 2, 100 + seed)
    model = make_model(sd, depth)
    kg = ours_grads(model, k2, k3, R)
    return case, pick, R, model.reference_grads(), kg


def check_params(case, pick, R, depth, mine, what):
    """Parameter gradients against sum_b J_b^T (sum over the copies of b of R): the oracle on the bases alone."""
    k2b, k3b, sd, _, _ = case
    Rb = torch.zeros(k2b.shape[0], R.shape[1], dtype=torch.float64, device=DEV).index_add_(0, pick.to(DEV), R.double())
    ref64 = oracle_param_grads(k2b, k3b, sd, depth, Rb, torch.float64)
    ref32 = oracle_param_grads(k2b, k3b, sd, depth, Rb, torch.float32)
    floor = 2e-4 if R.shape[0] * R.shape[1] > 1 << 16 else 1e-4
    worst_o, worst_r, bad = _anchored(mine, ref32, ref64, c=2.0, floor=floor)
    print("%s: parameter gradients (%d tensors), worst ours vs f64 %.3g, FP32 oracle vs f64 %.3g"
          % (what, len(ref64), worst_o, worst_r))
    assert not bad, bad[:5]
    return worst_o, worst_r


def check_kpts(case, pick, R, depth, mine, sel, what):
    """Keypoint gradients of the copies `sel` against the oracle on their bases with their own cotangents."""
    k2b, k3b, sd, _, _ = case
    b = pick[sel]
    k2, k3, Rs = k2b[b].contiguous(), k3b[b].contiguous(), R[sel]
    ref64 = oracle_grads(k2, k3, sd, depth, Rs, torch.float64)
    ref32 = oracle_grads(k2, k3, sd, depth, Rs, torch.float32)
    worst_o, worst_r, bad = _anchored({k: v[sel] for k, v in mine.items()}, ref32, ref64, c=2.0)
    print("%s: keypoint gradients of %d copies, worst ours vs f64 %.3g, FP32 oracle vs f64 %.3g" % (what, len(sel), worst_o, worst_r))
    assert not bad, bad
    return ref64


def _geometry_cases():
    """Every range layout each table n has on a B200, at depths 1, 2, 3 in turn (n with fewer than three layouts repeat
    them), and depth 12 at n = 73 (ranges crossing objects) and n = 256 (many tiles per CTA)."""
    cases = []
    for n, _, T, _ in BWD_GEOMETRY:
        regs = [r for r in REGIMES if regime_N(T, r, B200_SMS) is not None]
        for i in range(max(3, len(regs))):
            cases.append((n, regs[i % len(regs)], 1 + i % 3))
    return cases + [(73, "cross", 12), (256, "many", 12)]


GEOMETRY_CASES = _geometry_cases()


@pytest.mark.parametrize("n,regime,depth", [pytest.param(*c, id="n%d-%s-depth%d" % c) for c in GEOMETRY_CASES])
def test_backward_fp64_parity_at_every_tile_and_cta_layout(n, regime, depth):
    """Parameter gradients (every tensor: 4 + 6 * depth per net) and keypoint gradients of sum(reg_weights * R) at every
    tail E % 128 of BWD_GEOMETRY and every CTA range layout of the device, against FP64 at the bar of the module docstring.
    Keypoint gradients are checked on the first and last object and on the objects at CTA range boundaries."""
    sms = sm_count()
    T = GEOMETRY_T[n]
    N = regime_N(T, regime, sms)
    if N is None:
        pytest.skip("n = %d has no '%s' layout on %d SMs" % (n, regime, sms))
    what = "n=%d %s N=%d depth %d (%d tiles, %d CTAs)" % (n, regime, N, depth, N * T, bwd_ctas(N, T, sms))
    case, pick, R, mine, kg = run_copies(n, depth, N)
    check_params(case, pick, R, depth, mine, what)
    check_kpts(case, pick, R, depth, kg, boundary_objects(N, T, sms), what)


@pytest.mark.parametrize("n,N,depth", [(16, 300, 3), (73, 64, 2), (256, 3, 2)])
def test_backward_fp64_parity_for_large_batches_of_copies(n, N, depth):
    """Many objects per CTA (n = 16: 300 one-tile objects over 74 CTAs), 1344 tiles at n = 73 and three n = 256 objects (765
    tiles, every range begins inside an object), each copy with its own cotangent: one FP64 oracle run per base object."""
    sms = sm_count()
    T = GEOMETRY_T[n]
    what = "n=%d N=%d depth %d (%d tiles, %d CTAs)" % (n, N, depth, N * T, bwd_ctas(N, T, sms))
    case, pick, R, mine, kg = run_copies(n, depth, N)
    check_params(case, pick, R, depth, mine, what)
    check_kpts(case, pick, R, depth, kg, boundary_objects(N, T, sms), what)


@pytest.mark.parametrize("n", [17, 73])
@pytest.mark.parametrize("edge", ["0", "127", "128", "E-1"])
def test_single_edge_cotangent(n, edge):
    """R one-hot on one edge of the last object: the first edge, the last of tile 0, the first of tile 1 and E - 1, the last
    valid column of a partial tile (E % 128 = 8 and 68).  The gradients are nonzero and match FP64; every other object's
    keypoint gradients are exactly 0."""
    depth, T, E = 2, GEOMETRY_T[n], n * (n - 1) // 2
    N = regime_N(T, "cross", sm_count())
    e = E - 1 if edge == "E-1" else int(edge)
    R = torch.zeros(N, E, device=DEV)
    R[N - 1, e] = 1.0
    case, pick, R, mine, kg = run_copies(n, depth, N, R=R)
    what = "n=%d N=%d one-hot edge %d of object %d" % (n, N, e, N - 1)
    assert max(float(v.abs().max()) for v in mine.values()) > 0
    check_params(case, pick, R, depth, mine, what)
    for k in KEYS:
        assert bool((kg[k][:N - 1] == 0).all()), k
        assert float(kg[k][N - 1].abs().max()) > 0, k
    check_kpts(case, pick, R, depth, kg, [N - 1], what)


def _model_grads(model, k2, k3, R):
    model.zero_grad(set_to_none=True)
    kg = ours_grads(model, k2, k3, R)
    return model.params4.grad.clone(), model.params6.grad.clone(), kg


BATCH_SPLIT_TOL = 1e-4      # measured on B200: 3.1e-5 of the tensor's max


def test_batch_invariance_of_forward_and_backward():
    """Plain random objects (no quantisation), n = 73, depth 3, N = 10 (210 tiles over the CTAs) against the sub-batches
    [0, 3) + [3, 10) (63 and 147 tiles) and every object alone (21 tiles): the CTA range boundaries fall elsewhere in each.
    The saving forward is bit-identical per object (its statistics are per object, its FP16 scales depend on the weights
    only).  The backward scales each object's gradient images by that object's own maximum, so each object's keypoint
    gradients are bit-identical to its solo run; the parameter gradient of the batch sums per-CTA partials whose split
    follows the CTA ranges, so it equals the sum over the sub-batches to rounding only."""
    n, depth, N = 73, 3, 10
    ob = synth.make_objects(N=N, n=n, seed=2100)
    model = make_model(O.random_state_dict(86, depth=depth), depth)
    k2, k3 = cu(ob.kps_norm, ob.kps_3d)
    R = _cotangent(N, n * (n - 1) // 2, 21)
    w_all = model(k2, k3)[0]
    assert w_all.requires_grad
    for lo, hi in ((0, 3), (3, 10), (0, 7), (7, 10)) + tuple((i, i + 1) for i in range(N)):
        assert torch.equal(model(k2[lo:hi].contiguous(), k3[lo:hi].contiguous())[0], w_all[lo:hi]), (lo, hi)
    g4, g6, kg = _model_grads(model, k2, k3, R)
    parts = [_model_grads(model, k2[lo:hi].contiguous(), k3[lo:hi].contiguous(), R[lo:hi]) for lo, hi in ((0, 3), (3, 10))]
    worst = 0.0
    for full, a, b in ((g4, parts[0][0], parts[1][0]), (g6, parts[0][1], parts[1][1])):
        worst = max(worst, float((full - (a + b)).abs().max()) / float(full.abs().max()))
    print("batch vs sum of sub-batches: parameter gradients differ by %.3g of max" % worst)
    assert worst <= BATCH_SPLIT_TOL
    for i in range(N):
        solo = _model_grads(model, k2[i:i + 1].contiguous(), k3[i:i + 1].contiguous(), R[i:i + 1])[2]
        for k in KEYS:
            assert torch.equal(kg[k][i:i + 1], solo[k]), (i, k)


@pytest.mark.parametrize("k", [40, -40])
def test_cotangent_power_of_two_scaling_is_exact(k):
    """The gradient images are scaled by a power of two taken from the running maximum (pow2_scale): scaling R by 2^k
    scales every parameter and keypoint gradient by exactly 2^k."""
    n, depth, N = 73, 2, 5
    ob = synth.make_objects(N=N, n=n, seed=2200)
    model = make_model(O.random_state_dict(87, depth=depth), depth)
    k2, k3 = cu(ob.kps_norm, ob.kps_3d)
    R = _cotangent(N, n * (n - 1) // 2, 22)
    s = 2.0 ** k
    base, scaled = _model_grads(model, k2, k3, R), _model_grads(model, k2, k3, R * s)
    assert torch.equal(scaled[0], base[0] * s) and torch.equal(scaled[1], base[1] * s)
    for key in KEYS:
        assert torch.equal(scaled[2][key], base[2][key] * s), key
    assert float(base[0].abs().max()) > 0


def test_zero_cotangent_gives_exact_zeros():
    n, depth, N = 73, 2, 5
    ob = synth.make_objects(N=N, n=n, seed=2300)
    model = make_model(O.random_state_dict(88, depth=depth), depth)
    k2, k3 = cu(ob.kps_norm, ob.kps_3d)
    g4, g6, kg = _model_grads(model, k2, k3, torch.zeros(N, n * (n - 1) // 2, device=DEV))
    for t in (g4, g6, kg["kpts_2d"], kg["kpts_3d"]):
        assert bool((t == 0).all())


SCALE_SHIFTS = (0, 4, 8, 12, 16, 20, 24)


def test_per_object_cotangent_range():
    """Object b's cotangent scaled by 2^-s_b, s_b = 0 ... 24 in one batch (n = 73, depth 2, 147 tiles, ranges crossing
    objects): each object's keypoint gradients against FP64 relative to that object's own max, at the module's bar for
    every s.  With one scale per net, block and stage for the whole batch, an object 2^-12 below the largest already missed
    it (1.4e-4 on B200): its FP16 lo parts were subnormal.  The gradient images now take one scale per object."""
    n, depth = 73, 2
    N = len(SCALE_SHIFTS)
    R = _cotangent(N, n * (n - 1) // 2, 300) * torch.tensor([2.0 ** -s for s in SCALE_SHIFTS], device=DEV)[:, None]
    (k2b, k3b, sd, _, _), pick, R, _, kg = run_copies(n, depth, N, R=R)
    k2, k3 = k2b[pick].contiguous(), k3b[pick].contiguous()
    ref64 = oracle_grads(k2, k3, sd, depth, R, torch.float64)
    ref32 = oracle_grads(k2, k3, sd, depth, R, torch.float32)
    bad = []
    for i, s in enumerate(SCALE_SHIFTS):
        e_o = e_r = 0.0
        for k in KEYS:
            amax = float(ref64[k][i].abs().max())
            e_o = max(e_o, float((kg[k][i].double() - ref64[k][i]).abs().max()) / amax)
            e_r = max(e_r, float((ref32[k][i].double() - ref64[k][i]).abs().max()) / amax)
        print("cotangent 2^-%d: keypoint gradients ours vs f64 %.3g, FP32 oracle vs f64 %.3g (of the object's max)" % (s, e_o, e_r))
        if not e_o <= max(2 * e_r, 1e-4):
            bad.append((s, e_o, e_r))
    assert not bad, bad
