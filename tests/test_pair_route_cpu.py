"""Pins the float64 reference of the pair-routing tests (tests/pair_route_ref.py) to the oracle,
on the CPU: the reference is the oracle's `distr_routing` with the shift-and-add convolution in
place of the grouped conv1d, and its error bound is the formula stated there.  The GPU cases'
topologies are checked here to take the `seg_sum` branches they claim."""

import numpy as np
import pytest
import torch

import pair_route_ref as R
from oracle import hbv_oracle as O

PAR_NAMES = ('route_a', 'route_b', 'route_tau')


def _rel(a, b, floor=0.0):
    a, b = a.detach().double(), b.detach().double()
    den = max(b.abs().max().item(), floor)
    return (a - b).abs().max().item() / (den if den > 0 else 1.0)


# route_a / route_b do not enter a one-tap UH (w0 / w0 = 1): their gradient is rounding noise
# around zero in both evaluations, so gradients are compared relative to at least 1
GRAD_FLOOR = 1.0


def _both(topo, T, lenF, lag_uh, bounds, seed):
    """Reference and oracle in float64 on the same inputs: (out, g_qs, g_par) of each."""
    g = torch.Generator().manual_seed(seed)
    G, U = topo.shape
    rows, cols = R.topo_pairs(topo)
    qs = torch.rand(T, U, generator=g, dtype=torch.float64) * 5
    areas = torch.rand(U, generator=g, dtype=torch.float64) * 99 + 1
    par = torch.rand(rows.numel(), 3, generator=g, dtype=torch.float64)
    cot = torch.randn(T, G, generator=g, dtype=torch.float64)
    res = []
    for which in ('ref', 'oracle'):
        q = qs.clone().requires_grad_(True)
        p = par.clone().requires_grad_(True)
        if which == 'ref':
            out = R.route_ref(q, p, rows, cols, G, areas, R.topo_denom(topo, areas), lenF, lag_uh, bounds)
        else:
            distr = dict(zip(PAR_NAMES, R.descale(p, bounds, lag_uh)))
            out = O.distr_routing(q.unsqueeze(-1), distr, topo.double(), areas, lenF=lenF, lag_uh=lag_uh).squeeze(-1)
        gq, gp = torch.autograd.grad(out, (q, p), cot)
        res.append((out.detach(), gq, gp))
    return res


def test_reference_matches_oracle_nested_network():
    topo = R.nested_topology(seed=5)
    ref, orc = _both(topo, 150, 72, True, R.DEFAULT_BOUNDS, seed=1)
    for name, a, b in zip(('flow', 'g_qs', 'g_par'), ref, orc):
        assert _rel(a, b) < 1e-12, name


@pytest.mark.parametrize('lag_uh', [True, False])
@pytest.mark.parametrize('lenF,T', [(1, 5), (15, 5), (16, 17), (17, 16), (72, 129), (128, 127), (128, 300)])
def test_reference_matches_oracle_tap_edges(lenF, T, lag_uh):
    bounds = R.DEFAULT_BOUNDS[:2] + ((0.0, float(min(T, lenF))),)
    ref, orc = _both(R.small_topology(), T, lenF, lag_uh, bounds, seed=lenF + T)
    for name, a, b, fl in zip(('flow', 'g_qs', 'g_par'), ref, orc, (0.0, 0.0, GRAD_FLOOR)):
        assert _rel(a, b, fl) < 1e-12, f'{name} (lenF {lenF}, T {T}, lag {lag_uh})'


def test_reference_matches_oracle_lag_edges():
    """Physical lags with unit bounds, as the GPU case gives them: integers, a lag past the
    window (all-zero UH), one just inside it, and negative lags."""
    topo = R.many_gage_topology()
    g = torch.Generator().manual_seed(3)
    rows, cols = R.topo_pairs(topo)
    P = rows.numel()
    taus = torch.tensor([0.0, 1.0, 17.0, 47.999, 48.0, 0.5, 19.0, 19.5, 20.0, -0.5, -3.0], dtype=torch.float64)
    par = torch.stack([torch.rand(P, generator=g, dtype=torch.float64) * 5,
                       torch.rand(P, generator=g, dtype=torch.float64) * 12, taus[rows % len(taus)]], dim=1)
    qs = torch.rand(20, topo.shape[1], generator=g, dtype=torch.float64) * 5
    areas = torch.rand(topo.shape[1], generator=g, dtype=torch.float64) * 99 + 1
    out = R.route_ref(qs, par, rows, cols, topo.shape[0], areas, R.topo_denom(topo, areas), 72, True, R.UNIT_BOUNDS)
    distr = dict(zip(PAR_NAMES, R.descale(par, R.UNIT_BOUNDS)))
    ref = O.distr_routing(qs.unsqueeze(-1), distr, topo.double(), areas, lenF=72).squeeze(-1)
    assert _rel(out, ref) < 1e-12
    gone = taus[torch.arange(topo.shape[0]) % len(taus)] >= 20
    assert torch.equal(out[:, gone], torch.zeros_like(out[:, gone]))


@pytest.mark.parametrize('T', [300, 100])
def test_uh_conv_direct_matches_uh_conv_128_taps(T):
    """128 taps, over a series longer and shorter than the UH; values and both gradients."""
    g = torch.Generator().manual_seed(T)
    x = (torch.rand(9, 1, T, generator=g, dtype=torch.float64) * 5).requires_grad_(True)
    a = torch.rand(128, 9, 1, generator=g, dtype=torch.float64) * 5
    b = torch.rand(128, 9, 1, generator=g, dtype=torch.float64) * 12
    uh = O.uh_gamma(a, b, lenF=128).permute(1, 2, 0).contiguous().requires_grad_(True)
    assert uh.shape == (9, 1, 128)
    cot = torch.randn(9, 1, T, generator=g, dtype=torch.float64)
    y1 = O.uh_conv_direct(x, uh)
    y2 = O.uh_conv(x, uh)
    assert _rel(y1, y2) < 1e-13
    for d1, d2 in zip(torch.autograd.grad(y1, (x, uh), cot), torch.autograd.grad(y2, (x, uh), cot)):
        assert _rel(d1, d2) < 1e-13


def test_sum_bound_hand_example():
    """4 (M + n) 2^-24 S_abs + 1e-30, by hand: M = 2 taps; a gage of 1 pair with S_abs = 1 and
    one of 3 pairs with S_abs = 2 -> 12 / 2^24 and 40 / 2^24."""
    s_abs = torch.tensor([[1.0, 2.0], [0.0, 0.0]], dtype=torch.float64)
    bd = R.sum_bound(s_abs, 2, torch.tensor([1, 3]))
    assert bd[0, 0].item() == 12 / 2 ** 24 + 1e-30
    assert bd[0, 1].item() == 40 / 2 ** 24 + 1e-30
    assert bd[1, 0].item() == 1e-30 and bd[1, 1].item() == 1e-30
    ref = torch.tensor([[1.0, 2.0], [0.0, 0.0]], dtype=torch.float64)
    inside = ref + torch.tensor([[11.9, -39.9], [0.0, 0.0]], dtype=torch.float64) / 2 ** 24
    assert R.check_bound(inside, ref, s_abs, 2, [1, 3], 'inside') <= 1.0
    outside = ref + torch.tensor([[0.0, 40.1], [0.0, 0.0]], dtype=torch.float64) / 2 ** 24
    with pytest.raises(AssertionError, match='bound'):
        R.check_bound(outside, ref, s_abs, 2, [1, 3], 'outside')
    nonzero = ref.clone()
    nonzero[1, 0] = 1e-20                       # a zero sum must come out exactly zero
    with pytest.raises(AssertionError, match='bound'):
        R.check_bound(nonzero, ref, s_abs, 2, [1, 3], 'zero')
    nan = ref.clone()
    nan[0, 0] = float('nan')
    with pytest.raises(AssertionError, match='bound'):
        R.check_bound(nan, ref, s_abs, 2, [1, 3], 'nan')


def test_descale_rounds_like_the_kernel():
    """Physical values rounded to float32 as fmaf(p, hi - lo, lo) gives them (lo = 0: one
    rounding of p * hi), with the gradient hi - lo."""
    p = torch.rand(1000, 3, generator=torch.Generator().manual_seed(4), dtype=torch.float32)
    p64 = p.double().requires_grad_(True)
    vals = R.descale(p64, R.DEFAULT_BOUNDS)
    for i, v in enumerate(vals):
        hi = np.float32(R.DEFAULT_BOUNDS[i][1])
        assert torch.equal(v, (p[:, i] * float(hi)).double())
        (g,) = torch.autograd.grad(v.sum(), p64)
        assert torch.equal(g[:, i], torch.full_like(g[:, i], float(hi)))
        assert torch.equal(g[:, [k for k in range(3) if k != i]], torch.zeros_like(g[:, :2]))
    assert len(R.descale(p64, R.DEFAULT_BOUNDS, lag_uh=False)) == 2


def test_gpu_case_topologies():
    """The topologies of the GPU cases and the seg_sum branches (forward over gages, adjoint
    over units) they take: all four combinations."""
    def branches(topo):
        P = int((topo == 1).sum())
        return R.seg_sum_branch(P, topo.shape[0]), R.seg_sum_branch(P, topo.shape[1])

    c4 = R.config4_topology()
    assert c4.shape == (63, 2500) and (c4.sum(0) == 1).all() and int(c4[-1].sum()) == 20
    nested = R.nested_topology(seed=5)
    per_unit = (nested == 1).sum(0)
    assert nested.shape == (42, 300)
    assert int(per_unit.max()) == 40 and int((per_unit == 0).sum()) == 1
    assert int(((nested == 1).sum(1) == 0).sum()) == 1
    half = (nested == 0.5).nonzero()
    assert half.shape[0] == 1 and int(per_unit[half[0, 1]]) == 0
    seen = {branches(c4), branches(nested), branches(R.small_topology()), branches(R.many_gage_topology())}
    assert branches(c4) == ('wide', 'rows') and branches(nested) == ('wide', 'wide')
    assert branches(R.small_topology()) == ('rows', 'rows') and branches(R.many_gage_topology()) == ('rows', 'wide')
    assert len(seen) == 4
