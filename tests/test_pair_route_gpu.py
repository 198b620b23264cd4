"""The pair-routing kernels (K4', csrc/pair_route.cu) against a float64 reference, at the length
of BASELINE config 4 and on the topologies and shapes where their index arithmetic can go wrong.

K4' is the distributed (gage, unit) routing of `Hbv_2_hourly` (config 4 runs it on every
training step: 2,500 units x 17,520 hourly steps, 63 gages, 72 taps, fractional lag) and, with
an identity index, the 72-tap per-unit routing `unit_routing`.

Reference (tests/pair_route_ref.py): the oracle's `uh_gamma`, `frac_shift1d`, shift-and-add
`uh_conv_direct`, `scatter_add` and `denom` clamp, evaluated in float64 on the device; its
gradients come from autograd.  The oracle's own `distr_routing` in float32 is the arbiter
yardstick for the parameter gradients.

Checks, none of them tuned:
  * routed flow and g_qs, elementwise:  |new - fp64| <= 4 (M + n_terms) 2^-24 S_abs + 1e-30,
    S_abs the same sum of absolute terms (the flow itself; for g_qs the adjoint of |cotangent|),
    n_terms the pairs of the gage (forward) or of the unit (adjoint);
  * parameter gradients, per column: the arbiter gate err(new, fp64) <= 2 err(ref fp32, fp64)
    + 1e-6, and err(new, ref fp32) <= max(RTOL_GRAD, err(ref fp32, fp64)).  d/d(route_a, route_b)
    are differences of moments of the gamma UH, a cancellation, so a fixed 1e-4 alone means
    little for them.
Each case prints its worst error over its bound (pytest -s shows it).

`seg_sum` runs its 'wide' kernel (a warp per segment) when n_pairs >= 8 * n_segments and its
'rows' kernel otherwise; the forward sums over gages, the adjoint over units.  Every case states
the pair it takes, and together they take all four.
"""

import math

import pytest
import torch

import pair_route_ref as R
from conftest import RTOL_GRAD, arbiter_gate, assert_close

pytestmark = pytest.mark.gpu

PAR_NAMES = ('route_a', 'route_b', 'route_tau')


def _dev():
    return torch.device('cuda:0')


def _inputs(T, n_units, n_pairs, seed):
    """Qs in [0, 5] mm/h, areas in [1, 100], parameters in [0, 1], cotangent signed."""
    dev = _dev()
    g = torch.Generator(device=dev).manual_seed(seed)
    qs = torch.rand(T, n_units, generator=g, device=dev) * 5
    areas = torch.rand(n_units, generator=g, device=dev) * 99 + 1
    par = torch.rand(n_pairs, 3, generator=g, device=dev)
    return qs, areas, par, g


def _oracle32(qs, par, topo, areas, lenF, lag_uh, bounds):
    """The oracle's distr_routing in float32 (TF32 off for its grouped conv1d) -> [T, n_gages]."""
    from oracle import hbv_oracle as O
    distr = dict(zip(PAR_NAMES, R.descale(par, bounds, lag_uh)))
    with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
        return O.distr_routing(qs.unsqueeze(-1), distr, topo, areas, lenF=lenF, lag_uh=lag_uh).squeeze(-1)


def _run_kernels(topo, qs, areas, par, cot, lenF, lag_uh, bounds):
    from hydrodl2_b200 import routing
    q = qs.clone().requires_grad_(True)
    p = par.clone().requires_grad_(True)
    out = routing.distr_routing(q.unsqueeze(-1), p, topo, areas, lenF=lenF, lag_uh=lag_uh, bounds=bounds)
    out = out.squeeze(-1)
    (out * cot).sum().backward()
    torch.cuda.synchronize()
    return out.detach(), q.grad, p.grad


def _check_par_grad(what, new, r32, r64, M, lag_uh, g_uh0, theta, bounds):
    """Per-column gates of the [n_pairs, 3] parameter gradient; returns the worst err / allowed."""
    worst = {}
    for j, name in enumerate(PAR_NAMES):
        tag = f'{what}: d/d{name}'
        if j == 2 and not lag_uh:
            assert torch.equal(new[:, 2], torch.zeros_like(new[:, 2])), f'{tag}: nonzero without the lag'
            continue
        if j < 2 and M == 1:
            # one tap: the UH is w0 / w0 = 1 (times 1 - f), so route_a / route_b do not enter the
            # result and the fp64 gradient is rounding noise.  The kernel's is the rounding residue
            # of (g_u - s0) u (L - mL) with s0 = g_u u, mL = u L, u = 1 to 2 roundings, L = ln 0.5
            # (t - mT, t = 0.5, over theta^2 for route_b), comfortably inside
            # |g| <= 4 (M + 1) 2^-24 |dL/duh[0]| |c| (hi - lo), c = ln 2 or 0.5 / theta^2.
            span = bounds[j][1] - bounds[j][0]
            c = math.log(2.0) if j == 0 else 0.5 / theta.double() ** 2
            lim = 4 * (M + 1) * R.U32 * g_uh0.abs() * c * span + 1e-30
            r = float((new[:, j].double().abs() / lim).max())
            assert r <= 1.0, f'{tag}: one tap, |gradient| {r:.3g} x its rounding bound'
            worst[name] = r
            continue
        e_new, e_ref = arbiter_gate(new[:, j], r32[:, j], r64[:, j], f'{tag} arbiter')
        assert_close(new[:, j], r32[:, j], max(RTOL_GRAD, e_ref), f'{tag} vs ref fp32')
        worst[name] = e_new / (2 * e_ref + 1e-6)
    return worst


def _check_routing(what, topo, qs, areas, par, cot, lenF, lag_uh=True, bounds=R.DEFAULT_BOUNDS,
                   branches=None):
    """Kernels vs the float64 reference (flow, g_qs, parameter gradient).  Returns the kernels'
    (out, g_qs, g_par)."""
    dev = qs.device
    topo = topo.to(dev)
    T, U = qs.shape
    G = topo.shape[0]
    M = min(T, lenF)
    rows, cols = R.topo_pairs(topo)
    P = rows.numel()
    if branches is not None:
        assert (R.seg_sum_branch(P, G), R.seg_sum_branch(P, U)) == branches, what
    out, gq, gp = _run_kernels(topo, qs, areas, par, cot, lenF, lag_uh, bounds)

    q64 = qs.double().requires_grad_(True)
    p64 = par.double().requires_grad_(True)
    out64, uh64 = R.route_ref(q64, p64, rows, cols, G, areas, R.topo_denom(topo, areas), lenF, lag_uh, bounds,
                              keep_uh=True)
    c64 = cot.double()
    gq64, gp64, guh64 = torch.autograd.grad(out64, (q64, p64, uh64), c64, retain_graph=True)
    (gq_abs,) = torch.autograd.grad(out64, q64, c64.abs())
    out64 = out64.detach()

    p32 = par.clone().requires_grad_(True)
    (gp32,) = torch.autograd.grad(_oracle32(qs, p32, topo, areas, lenF, lag_uh, bounds), p32, cot)

    n_gage = torch.bincount(rows, minlength=G)
    n_unit = torch.bincount(cols, minlength=U)
    r_out = R.check_bound(out, out64, out64, M, n_gage, f'{what}: routed flow')
    r_gq = R.check_bound(gq, gq64, gq_abs, M, n_unit, f'{what}: g_qs')
    theta = torch.relu(R.descale(par, bounds, lag_uh)[1]) + 0.5
    r_par = _check_par_grad(what, gp, gp32, gp64, M, lag_uh, guh64[0, :, 0], theta, bounds)
    print(f'{what}: worst err / bound: flow {r_out:.3f}, g_qs {r_gq:.3f}; parameter gradients '
          + ', '.join(f'{k} {v:.3f}' for k, v in r_par.items()))
    return out, gq, gp


# --------------------------------------------------------------------------------------------
# config 4: 2,500 units x 17,520 steps, 63 gages
# --------------------------------------------------------------------------------------------
C4_T, C4_UNITS, C4_PER_GAGE = 17520, 2500, 40


def _config4_inputs():
    topo = R.config4_topology(C4_UNITS, C4_PER_GAGE).to(_dev())
    qs, areas, par, g = _inputs(C4_T, C4_UNITS, C4_UNITS, seed=40)
    cot = torch.randn(C4_T, topo.shape[0], generator=g, device=_dev())
    return topo, qs, areas, par, cot


def test_config4_length():
    """Forward 'wide' (2,500 pairs over 63 gages), adjoint 'rows' (2,500 units of one pair);
    9 time chunks in the d/dUH pass; 17,520 = 136 x 128 + 112, so the last tile is partial."""
    from hydrodl2_b200 import _cabi
    assert _cabi.load().hbv_b200_pair_chunks(C4_T) == 9
    assert C4_T % 128 != 0
    topo, qs, areas, par, cot = _config4_inputs()
    assert topo.shape[0] == 63 and int(topo[-1].sum()) == 20
    _check_routing('config 4 (T 17520, 2500 units, 63 gages)', topo, qs, areas, par, cot, 72,
                   branches=('wide', 'rows'))


def test_config4_deterministic():
    """Two runs of the config-4 case: bit-identical flow, g_qs and parameter gradient."""
    topo, qs, areas, par, cot = _config4_inputs()
    a = _run_kernels(topo, qs, areas, par, cot, 72, True, R.DEFAULT_BOUNDS)
    b = _run_kernels(topo, qs, areas, par, cot, 72, True, R.DEFAULT_BOUNDS)
    for name, x, y in zip(('flow', 'g_qs', 'g_par'), a, b):
        assert torch.equal(x, y), f'config 4: {name} differs between two identical runs'


# --------------------------------------------------------------------------------------------
# nested gauges
# --------------------------------------------------------------------------------------------
def test_nested_network():
    """Forward 'wide', adjoint 'wide' (5,759 pairs over 42 gages / 300 units).  T = 4,100: three
    d/dUH chunks, the last ending in a partial tile.  Units on 40 gages, a unit on none, a gage
    with none, and a 0.5 entry that counts in its gage's upstream area only."""
    from hydrodl2_b200 import _cabi
    T = 4100
    assert _cabi.load().hbv_b200_pair_chunks(T) == 3 and T % 128 != 0
    topo = R.nested_topology(seed=5).to(_dev())
    per_unit = (topo == 1).sum(0)
    assert int(per_unit.max()) == 40 and int((per_unit == 0).sum()) == 1
    assert int(((topo == 1).sum(1) == 0).sum()) == 1 and int((topo == 0.5).sum()) == 1
    P = int((topo == 1).sum())
    qs, areas, par, g = _inputs(T, topo.shape[1], P, seed=41)
    cot = torch.randn(T, topo.shape[0], generator=g, device=_dev())
    out, gq, _ = _check_routing('nested network (T 4100, 300 units, 42 gages)', topo, qs, areas, par, cot, 72,
                                branches=('wide', 'wide'))
    empty_gage = ((topo == 1).sum(1) == 0).nonzero()[0, 0]
    lone_unit = (per_unit == 0).nonzero()[0, 0]
    assert torch.equal(out[:, empty_gage], torch.zeros_like(out[:, empty_gage]))
    assert torch.equal(gq[:, lone_unit], torch.zeros_like(gq[:, lone_unit]))


# --------------------------------------------------------------------------------------------
# tap-count edges
# --------------------------------------------------------------------------------------------
@pytest.mark.parametrize('lag_uh', [True, False], ids=['lag', 'nolag'])
@pytest.mark.parametrize('T', [1, 5, 127, 129, 300])
@pytest.mark.parametrize('lenF', [1, 15, 16, 17, 72, 128])
def test_tap_edges(lenF, T, lag_uh):
    """Forward 'rows', adjoint 'rows' (24 pairs over 4 gages / 12 units).  M = min(T, lenF) taps,
    padded to 16 in the convolution and to 8 in d/dUH; the lag spans [0, M) so that it moves the
    UH inside the window."""
    topo = R.small_topology().to(_dev())
    P = int((topo == 1).sum())
    qs, areas, par, g = _inputs(T, topo.shape[1], P, seed=1000 + 7 * lenF + T)
    cot = torch.randn(T, topo.shape[0], generator=g, device=_dev())
    M = min(T, lenF)
    bounds = R.DEFAULT_BOUNDS[:2] + ((0.0, float(M)),)
    _check_routing(f'taps lenF {lenF}, T {T}, lag {lag_uh}', topo, qs, areas, par, cot, lenF, lag_uh, bounds,
                   branches=('rows', 'rows'))


# --------------------------------------------------------------------------------------------
# lag edges
# --------------------------------------------------------------------------------------------
LAGS = (0.0, 1.0, 17.0, 47.999, 48.0, 0.5, 19.0, 19.5, 20.0, -0.5, -3.0)


def test_lag_edges():
    """Forward 'rows', adjoint 'wide' (200 pairs over 40 gages / 6 units).  T = 20, so M = 20.
    The lag is given physically with unit bounds so that it is exact: every pair of gage g has
    tau = LAGS[g % 11].  An integer tau has no fractional part; tau >= M shifts the whole UH out
    of the window, and such gages must give exact zeros, with zero gradients for their pairs; a
    negative tau (only the physical form can give one) shifts the UH forward, as the reference's
    `frac_shift1d` does, and its adjoint must not read d/dUH before tap 0."""
    T, lenF = 20, 72
    topo = R.many_gage_topology().to(_dev())
    rows, _ = R.topo_pairs(topo)
    P = rows.numel()
    qs, areas, par, g = _inputs(T, topo.shape[1], P, seed=42)
    cot = torch.randn(T, topo.shape[0], generator=g, device=_dev())
    tau_g = torch.tensor(LAGS, dtype=torch.float32, device=_dev())[torch.arange(topo.shape[0], device=_dev()) % len(LAGS)]
    par = torch.stack([par[:, 0] * 5, par[:, 1] * 12, tau_g[rows]], dim=1)
    assert float(par[:, 2].max()) == 48.0 and float(par[:, 2].min()) == -3.0
    out, _, gp = _check_routing('lag edges (T 20)', topo, qs, areas, par, cot, lenF, True, R.UNIT_BOUNDS,
                                branches=('rows', 'wide'))
    gone = tau_g >= T
    assert torch.equal(out[:, gone], torch.zeros_like(out[:, gone]))
    assert bool((out[:, ~gone] > 0).any(dim=0).all())
    assert torch.equal(gp[gone[rows]], torch.zeros_like(gp[gone[rows]]))


# --------------------------------------------------------------------------------------------
# the two parameter conventions
# --------------------------------------------------------------------------------------------
def test_normalised_and_physical_conventions():
    """The same pairs through (a) normalised parameters with the default bounds and (b) the
    physical dict of `Hbv_2_hourly.distr_routing` (unit bounds).  (b) is checked against the
    reference; both descale to the same float32 values, so (a) and (b) must give the same flow
    bit for bit, and each dict entry's gradient times its span must be (a)'s gradient column."""
    import hydrodl2_b200 as hydrodl2
    T = 500
    topo = R.small_topology().to(_dev())
    P = int((topo == 1).sum())
    qs, areas, par, g = _inputs(T, topo.shape[1], P, seed=43)
    cot = torch.randn(T, topo.shape[0], generator=g, device=_dev())
    M = hydrodl2.load_model('hbv_2_hourly', ver_name='Hbv_2_hourly')
    m = M({'dynamic_params': {'Hbv_2_hourly': ['parBETA']}, 'nmul': 1, 'routing': False}, device=_dev())
    phys = m._descale_distr_parameters(par)
    ref_out, ref_gq, ref_gp = _check_routing('physical convention', topo, qs, areas,
                                             torch.stack([phys[k] for k in PAR_NAMES], dim=1), cot, 72,
                                             True, R.UNIT_BOUNDS)
    # (a) normalised
    out_n, gq_n, gp_n = _run_kernels(topo, qs, areas, par, cot, 72, True, R.DEFAULT_BOUNDS)
    # (b) the model's method, dict in
    leaves = {k: v.detach().clone().requires_grad_(True) for k, v in phys.items()}
    q = qs.clone().unsqueeze(-1).requires_grad_(True)
    out_p = m.distr_routing(q, leaves, topo, areas)['Qs_rout'].squeeze(-1)
    (out_p * cot).sum().backward()
    assert torch.equal(out_n, ref_out) and torch.equal(out_p.detach(), ref_out)
    assert torch.equal(gq_n, ref_gq) and torch.equal(q.grad.squeeze(-1), ref_gq)
    for j, k in enumerate(PAR_NAMES):
        span = R.DEFAULT_BOUNDS[j][1] - R.DEFAULT_BOUNDS[j][0]
        assert torch.equal(leaves[k].grad, ref_gp[:, j]), f'dict entry {k}: gradient'
        assert torch.equal(leaves[k].grad * span, gp_n[:, j]), f'{k}: normalised gradient != physical x {span}'


# --------------------------------------------------------------------------------------------
# unit_routing on more than 32,768 units
# --------------------------------------------------------------------------------------------
def test_unit_routing_over_32768_units():
    """`unit_routing` splits 33,000 units into calls of 32,768 and 232.  Per-unit gamma UH
    (72 taps, no lag), forward 'rows' and adjoint 'rows' (one pair per segment).  Every unit is
    checked; the worst errors on each side of unit 32,768 are printed."""
    from hydrodl2_b200 import routing
    from oracle import hbv_oracle as O
    T, B, lenF = 200, 33000, 72
    cut = routing._MAX_UNITS_PER_CALL
    assert cut < B
    bounds = R.DEFAULT_BOUNDS[:2] + ((0.0, 0.0),)
    qs, _, par, g = _inputs(T, B, B, seed=44)
    par[:, 2] = 0
    cot = torch.randn(T, B, generator=g, device=_dev())
    q = qs.clone().requires_grad_(True)
    ab = par[:, :2].clone().requires_grad_(True)
    out = routing.unit_routing(q, ab, lenF, bounds[:2])
    (out * cot).sum().backward()
    out = out.detach()

    ar = torch.arange(B, device=_dev())
    ones = torch.ones(B, dtype=torch.float64, device=_dev())
    q64 = qs.double().requires_grad_(True)
    p64 = par.double().requires_grad_(True)
    out64 = R.route_ref(q64, p64, ar, ar, B, ones, ones, lenF, False, bounds)
    c64 = cot.double()
    gq64, gp64 = torch.autograd.grad(out64, (q64, p64), c64, retain_graph=True)
    (gq_abs,) = torch.autograd.grad(out64, q64, c64.abs())
    out64 = out64.detach()

    # float32: the oracle's uh_gamma + uh_conv, as in the hourly model's `routing=True` branch
    ab32 = par[:, :2].clone().requires_grad_(True)
    a, b = R.descale(ab32, bounds, lag_uh=False)
    uh = O.uh_gamma(a.view(1, B, 1).expand(lenF, B, 1), b.view(1, B, 1).expand(lenF, B, 1), lenF=lenF)
    with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
        y32 = O.uh_conv(qs.T.contiguous().unsqueeze(1), uh.permute(1, 2, 0).contiguous()).squeeze(1).T
    (gp32,) = torch.autograd.grad(y32, ab32, cot)

    for lo, hi in ((0, cut), (cut, B)):
        side = f'unit_routing units {lo}..{hi - 1}'
        r_out = R.check_bound(out[:, lo:hi], out64[:, lo:hi], out64[:, lo:hi], lenF, 1, f'{side}: flow')
        r_gq = R.check_bound(q.grad[:, lo:hi], gq64[:, lo:hi], gq_abs[:, lo:hi], lenF, 1, f'{side}: g_q')
        print(f'{side}: worst err / bound: flow {r_out:.3f}, g_q {r_gq:.3f}')
    r_par = _check_par_grad('unit_routing 33000 units', torch.cat([ab.grad, torch.zeros_like(ab.grad[:, :1])], 1),
                            torch.cat([gp32, torch.zeros_like(gp32[:, :1])], 1), gp64, lenF, False, None, None,
                            bounds)
    print('unit_routing 33000 units: parameter gradients ' + ', '.join(f'{k} {v:.3f}' for k, v in r_par.items()))
    # the units next to the cut route with their own parameters
    assert bool((out[:, cut - 2:cut + 2] > 0).all())


# --------------------------------------------------------------------------------------------
# refusals
# --------------------------------------------------------------------------------------------
def test_refusals():
    """More than 128 taps is refused unless T is shorter (M = min(lenF, T) taps run, and the
    result is that of lenF = T); a parameter row count that is not the topology's pair count
    raises ValueError."""
    from hydrodl2_b200 import routing
    topo = R.small_topology().to(_dev())
    P = int((topo == 1).sum())
    qs, areas, par, _ = _inputs(200, topo.shape[1], P, seed=45)
    with pytest.raises(RuntimeError, match='lenF > 128'):
        routing.distr_routing(qs.unsqueeze(-1), par, topo, areas, lenF=129)
    short = qs[:100].contiguous().unsqueeze(-1)
    long_f = routing.distr_routing(short, par, topo, areas, lenF=1000)
    assert torch.equal(long_f, routing.distr_routing(short, par, topo, areas, lenF=100))
    with pytest.raises(ValueError, match='pairs'):
        routing.distr_routing(qs.unsqueeze(-1), par[:-1], topo, areas)
    with pytest.raises(ValueError, match='pairs'):
        routing.distr_routing(qs.unsqueeze(-1), torch.cat([par, par[:1]]), topo, areas)
