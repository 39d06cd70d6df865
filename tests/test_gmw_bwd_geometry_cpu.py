"""CPU checks of the helpers of tests/test_gpu_gmw_bwd_geometry.py: the quantised objects are seeded and use every pool
value, the CTA range layouts are what their names say, and every pinned case finds a seed with an FP64 ReLU margin."""
import pytest
import torch

import test_gpu_gmw_bwd_geometry as G


def test_quantised_objects_are_seeded_and_use_every_pool_value():
    a, b = G.quantised_objects(4, 23, 6, 5), G.quantised_objects(4, 23, 6, 5)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert not torch.equal(a[0], G.quantised_objects(4, 23, 6, 6)[0])
    k2, k3 = a
    assert k2.shape == (4, 23, 2) and k3.shape == (4, 23, 3)
    for i in range(4):
        joint = torch.cat((k2[i].double(), k3[i].double()), dim=1)
        # six distinct keypoints in 2D, in 3D and jointly: the same index pattern in both
        assert len(torch.unique(k2[i], dim=0)) == len(torch.unique(k3[i], dim=0)) == len(torch.unique(joint, dim=0)) == 6


@pytest.mark.parametrize("sms", [148, 132, 80])
def test_cta_range_layouts(sms):
    C = min(sms // 2, 128)
    for n, E, T, tail in G.BWD_GEOMETRY:
        assert T == G.GEOMETRY_T[n] and (E - 1) // G.TE == T - 1 and E - (T - 1) * G.TE == (tail or G.TE)
        for regime in G.REGIMES:
            N = G.regime_N(T, regime, sms)
            if N is None:
                continue
            ranges = G.cta_ranges(N, T, sms)
            assert ranges[0][0] == 0 and ranges[-1][1] == N * T
            assert all(r[1] == q[0] and r[0] < r[1] for r, q in zip(ranges, ranges[1:]))
            if regime in ("under", "exact"):
                assert (N * T < C if regime == "under" else N * T == C) and all(hi - lo == 1 for lo, hi in ranges)
            elif regime == "cross":
                assert C < N * T < 2 * C and G.crosses_objects(N, T, sms)
            else:
                assert N * T >= 4 * C and G.crosses_objects(N, T, sms) and (T == 1 or G.ends_inside_objects(N, T, sms))
            sel = G.boundary_objects(N, T, sms)
            assert sel[0] == 0 and sel[-1] == N - 1 and len(sel) <= 12


def test_b200_layouts_and_cases():
    """On a B200 (74 CTAs per net) every table n has a layout with several tiles per CTA, and every depth 1 ... 3 runs at
    every n."""
    Ns = {n: {r: G.regime_N(T, r, G.B200_SMS) for r in G.REGIMES} for n, _, T, _ in G.BWD_GEOMETRY}
    assert Ns[16] == {"under": 73, "exact": 74, "cross": 75, "many": 296}
    assert Ns[73] == {"under": 3, "exact": None, "cross": 5, "many": 15}
    assert Ns[256] == {"under": None, "exact": None, "cross": None, "many": 3}
    for n, _, _, _ in G.BWD_GEOMETRY:
        assert {d for m, _, d in G.GEOMETRY_CASES if m == n} >= {1, 2, 3}
    assert (73, "cross", 12) in G.GEOMETRY_CASES and (256, "many", 12) in G.GEOMETRY_CASES


def test_margin_search_finds_a_seed_for_every_case():
    cases = {(n, depth, G.bases_for(n, G.regime_N(G.GEOMETRY_T[n], r, G.B200_SMS), depth)) for n, r, depth in G.GEOMETRY_CASES}
    for n, depth, bases in sorted(cases):
        k2, k3, sd, seed, margin = G.pinned_case(n, depth, bases)
        assert margin > G.MARGIN and k2.shape == (bases, n, 2)
    again = G.pinned_case.__wrapped__(73, 2, 3)              # the search is deterministic (pinned_case caches it)
    first = G.pinned_case(73, 2, 3)
    assert again[3] == first[3] and again[4] == first[4] and torch.equal(again[0], first[0]) and torch.equal(again[1], first[1])
